/* microsound_b200.h -- C ABI of the B200-native Microsound render kernels.
 *
 * The reference (maetyu-d/audio-suite, microsound_0.2.1/main_v2.py) is pure Python/numpy and has no
 * FFI of its own; its boundary for this path is the Python function
 *     render(params: dict, progress=None) -> (float64[out_n, 2], meta)        main_v2.py:588-792
 * which audio_suite_b200.render() reproduces.  This header is the layer *below* that function:
 * what the Python host binds with ctypes (audio_suite_b200/_abi.py), one entry point per stage of
 * render(), each citing the reference lines it replaces.
 *
 * Conventions: every function returns 0 on success and a negative value on error (message from
 * ms_last_error(), thread-local).  No function throws.  All data pointers are DEVICE pointers owned
 * by the caller (torch tensors: tensor.data_ptr()) unless the name says host.  `stream` is a
 * cudaStream_t passed as void*.  Offsets are in elements of the pointed-to type.  The library keeps
 * only internal plan caches (twiddle / chirp tables); it never returns memory it allocated.
 */
#ifndef MICROSOUND_B200_H
#define MICROSOUND_B200_H
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define MS_ABI_VERSION 1

int ms_version(void);
const char* ms_last_error(void);
/* 1 when the library was built from the CUDA sources for sm_100a (always, for the shipped .so). */
int ms_is_cuda_build(void);
/* kernels this library has launched since it was loaded (bench.py reports the delta per step). */
unsigned long long ms_launch_count(void);
/* bytes of job descriptors the library itself has copied host->device since it was loaded. */
unsigned long long ms_h2d_bytes(void);
/* observer called after every kernel launch with the kernel's type name and its stream (NULL: off).  bench.py
 * records a CUDA event there to time the individual kernels of a step; the product never sets it. */
void ms_set_launch_hook(void (*hook)(const char* kernel, void* stream));

/* ---- spectral stage: lowpass_fft (main_v2.py:39-59), fft_partial_stretch (:117-128),
 *      unfold_multiband / bandpass_fft (:492-500, :61-101), tilted_noise shaping (:224-233),
 *      spectral_diffusion_stereo's rotation (:432-435; odd lengths only, even lengths use ms_stereo_post).
 * One job = two real signals of equal length n packed into one complex transform. */
enum { MS_OP_NONE = 0, MS_OP_GRAIN = 1, MS_OP_TILT = 2, MS_OP_ROT = 3 };

typedef struct {
    double lo_f0, lo_f1;     /* rising skirt, Hz   */
    double hi_f0, hi_f1;     /* falling skirt, Hz  */
    int32_t lo_mode, hi_mode;/* 0 none, 1 brick wall, 2 raised cosine */
    int32_t zero;            /* band contributes nothing */
    int32_t _pad;
} ms_band_edge;

typedef struct {
    int32_t kind;            /* MS_OP_* */
    int32_t n_bands;         /* 0 or 3 (multiband unfold) */
    int32_t lp_on;           /* low-pass present */
    int32_t stretch_on;      /* spectral stretch present */
    double df;               /* bin spacing, Hz: 1.0 / (n * (1.0 / sr)) */
    double factor;           /* stretch factor */
    double alpha;            /* MS_OP_TILT exponent, MS_OP_ROT angle */
    double warp_exp;         /* fft_warp_power (main_v2.py:103-115): 1 / max(1e-6, power); 0 = no warp.  Order of the
                                grain operator: low-pass -> power warp -> stretch -> multiband */
    ms_band_edge lp;
    ms_band_edge mb[3];
} ms_spec_op;

typedef struct {
    int32_t n;               /* signal length (any n >= 1) */
    int32_t _pad;
    int64_t in_a, in_b;      /* offsets into src; in_b < 0: no second signal */
    int64_t out_a, out_b;    /* offsets into dst; out_b < 0: discard second signal */
    ms_spec_op op[2];        /* operator for signal a and for signal b */
} ms_spec_job;

/* One-shot: plan + run + release. */
/* ms_spectral_workspace_bytes_f32 / ms_spectral_workspace_bytes_f64: declared below by MS_DECLARE_API */
/* ms_spectral_apply_f32 / ms_spectral_apply_f64: declared below by MS_DECLARE_API */
/* Planned: job descriptors are uploaded into `workspace` once; ms_spectral_run() only launches kernels
 * (CUDA-graph capturable).  src/dst/workspace must stay valid for the life of the handle. */
/* ms_spectral_create_f32 / ms_spectral_create_f64: declared below by MS_DECLARE_API */
/* ms_spectral_run_f32 / ms_spectral_run_f64: declared below by MS_DECLARE_API */
/* ms_spectral_destroy_f32 / ms_spectral_destroy_f64: declared below by MS_DECLARE_API */
/* The two halves of ms_spectral_run, for stages that work on the spectra in between (spectral imprint):
 * ms_spectral_forward leaves job i's natural-order spectrum (n complex values; for a single-signal job simply the
 * DFT of the signal) at workspace + z_base_bytes + 2 * sizeof(REAL) * z_offset[i]  (ms_spectral_z_table, offsets in
 * complex elements, in the order the jobs were given); ms_spectral_inverse applies the jobs' operators to whatever
 * is there and transforms back. */
/* ms_spectral_forward_f32/_f64, ms_spectral_inverse_f32/_f64, ms_spectral_z_table_f32/_f64: declared below */
/* SpectralImprint.apply (main_v2.py:565-581) on the spectra of one render's grains, in event order: an exponential
 * moving average of |X| per bin (restarted when the spectrum length changes) blended into the magnitudes, phases
 * kept.  One record per imprinted grain, grouped by render in event order. */
typedef struct { int64_t z; int32_t n, _pad; } ms_imprint_evt;               /* z: offset of the grain's spectrum, complex elements */
typedef struct { int32_t ev_begin, ev_end; double amount, smooth; } ms_imprint_render;
/* ms_imprint_f32 / ms_imprint_f64: declared below by MS_DECLARE_API */
/* Event feedback (main_v2.py:731-734): dst = (1 - fb) cur + fb prev over the first min(n_cur, n_prev) samples, cur beyond.
 * prev is the PREVIOUS event's final grain of the same render, so the events of a render are processed rank by rank
 * (the host launches rank e of all renders together).  With the spectral imprint on, ms_imprint_step advances the
 * per-render moving average by exactly one grain (state: `mem`, max_bins REALs per render slot; prev_bins per slot). */
typedef struct { int64_t cur, prev, dst; int32_t n_cur, n_prev; double fb; } ms_feedback_evt;
typedef struct { int64_t z; int32_t n, slot; double amount, smooth; } ms_imprint_step_evt;
/* ms_feedback_f32/_f64, ms_imprint_step_f32/_f64: declared below by MS_DECLARE_API */
/* resonator_bank (main_v2.py:369-384) on time-domain grains: dst = 0.55 src + 0.45 bank sign(src), bank = the
 * peak-normalised sum of decaying sinusoids whose frequencies / phases the host drew.  One CTA per grain. */
typedef struct { double f_over_sr, phase, weight; } ms_res_mode;
typedef struct {
    int64_t src, dst;        /* pool offsets */
    int32_t n, mode_begin, mode_count, _pad;
    double decay;            /* 1 / (tau * sr): env[j] = exp(-j * decay) */
} ms_res_evt;
/* ms_resonator_f32 / ms_resonator_f64: declared below by MS_DECLARE_API */
/* waveguide_splinters (main_v2.py:386-402) on time-domain grains: a cascade of feedback combs, per line
 * v[t] = y[t] + g v[t - d], y[t] <- (1 - mix) y[t] + mix v[t].  dst may equal src.  One CTA per grain. */
typedef struct { int32_t d, _pad; double g, mix; } ms_wg_line;
typedef struct { int64_t src, dst, tmp; int32_t n, line_begin, line_count, _pad; } ms_wg_evt;   /* tmp: n REALs of scratch */
/* ms_waveguide_f32 / ms_waveguide_f64: declared below by MS_DECLARE_API */
/* partial_lock_stretch (main_v2.py:130-148) on the spectrum of one grain (single-signal job, after
 * ms_spectral_forward): W = low-pass / power warp of the grain's spectrum (`pre`), the top_n strongest bins of W
 * (DC excluded) are moved to round(k * factor) with a triangular spread over +-neigh bins on top of 0.12 W, and the
 * result replaces the spectrum in place; ms_spectral_inverse (operator: multiband only) finishes.  `scratch`:
 * offset (REAL elements) of 3 * (n/2 + 1) REALs of per-grain scratch in the `scratch` buffer. */
typedef struct {
    int64_t z;               /* offset of the grain's spectrum, complex elements */
    int64_t scratch;
    int32_t n, top_n, neigh, _pad;
    double factor;
    ms_spec_op pre;
} ms_plock_evt;
/* ms_partial_lock_f32 / ms_partial_lock_f64: declared below by MS_DECLARE_API */
/* cepstral_warp (main_v2.py:150-163) around three spectral stages of single-signal jobs: (1) forward of the grain;
 * ms_cepstral(step 0): X = low-pass / power warp of its spectrum (`pre`) is kept in scratch and log(|X| + 1e-12)
 * becomes the spectrum of stage 2; (2) inverse of stage 2 -> cepstrum; ms_cepstral(step 1): the cepstrum resampled at
 * t / factor; (3) forward of stage 3; ms_cepstral(step 2): exp(Re Z3) with the phases of X replaces the spectrum of
 * stage 1, whose inverse (operator: stretch, multiband) finishes.  Offsets z1/z2/z3 in complex elements of the three
 * stages' spectra, xp/cep/cep2 in REAL elements of `scratch`. */
typedef struct {
    int64_t z1, z2, z3;
    int64_t xp, cep, cep2;
    int32_t n, _pad;
    double factor;
    ms_spec_op pre;
} ms_cep_evt;
/* ms_cepstral_f32 / ms_cepstral_f64: declared below by MS_DECLARE_API */
/* test entry: Z[k] = sum_j (a[j] + i b[j]) exp(-2 pi i jk/n), interleaved re/im, natural order */
/* ms_fft_pair_forward_f32 / ms_fft_pair_forward_f64: declared below by MS_DECLARE_API */
/* ms_fft_pair_workspace_bytes_f32 / ms_fft_pair_workspace_bytes_f64: declared below by MS_DECLARE_API */

/* ---- transient synthesis: gen_basic (main_v2.py:219-269).  One record per event; the array lives in
 *      DEVICE memory.  The PCG64 state is numpy's `PCG64(seed).state` right after seeding. */
enum { MS_SY_GAUSS = 0, MS_SY_DUST = 1, MS_SY_NOISE = 2, MS_SY_SKEW = 3, MS_SY_RES = 4, MS_SY_PLAIN = 5, MS_SY_WAVELET = 6,
       MS_SY_IRFRAG = 7, MS_SY_SCANLINE = 8, MS_SY_SILENT = 9, MS_SY_CHAOS = 10, MS_SY_STICK = 11 };
typedef struct {
    uint64_t s_hi, s_lo, i_hi, i_lo;
    int32_t n, mode;
    int32_t fade, sigma;      /* max(8,int(.01n)) ; max(1,int(.0025n)) */
    int64_t out;              /* offset into the float pool where this event's signal is written */
    double f_over_sr;         /* MS_SY_RES: max(10, ring_hz) / gen_sr */
    double inv_fade;          /* 1 / fade */
    double ring_decay;        /* MS_SY_RES: 1 / (tau * gen_sr) */
    double env_decay;         /* 1 / (T * gen_sr) of the mode's exponential envelope */
    int64_t dust_begin;       /* MS_SY_DUST: range in the impulse arrays */
    int32_t dust_count, ker_len;
    int64_t aux;              /* MS_SY_NOISE / MS_SY_SKEW: pool offset of the tilted noise */
    int64_t atom_begin;       /* MS_SY_WAVELET: range in the atom arrays */
    int32_t atom_count, _pad;
} ms_synth_evt;
/* gen_wavelet_atoms (main_v2.py:317-331) + morlet_atom (:165-170): per atom the host-drawn scalars, as
 * (f0 / gen_sr, 1 / (sigma * gen_sr), phase, weight) and the circular shift in samples. */
typedef struct { double f0_over_sr, inv_sigma, phase, weight; } ms_wavelet_atom;
/* normals + closed-form modes (GAUSS, RES, PLAIN) and raw normals for NOISE/SKEW (written at `out`) */
/* ms_synth_normal_f32 / ms_synth_normal_f64: declared below by MS_DECLARE_API */
/* ms_synth_dust_f32 / ms_synth_dust_f64: declared below by MS_DECLARE_API */
/* NOISE / SKEW: envelope, rectified difference and fades applied to the tilted noise at `aux` */
/* ms_synth_tilt_finish_f32 / ms_synth_tilt_finish_f64: declared below by MS_DECLARE_API */
/* MS_SY_IRFRAG (gen_ir_fragment, main_v2.py:333-348), MS_SY_SCANLINE (gen_image_scanline, :350-362), MS_SY_SILENT:
 * a short host-chosen table (dust_val[dust_begin .. +dust_count]) stretched to n samples by linear interpolation
 * under a Hann window, then peak-normalised to 0.9 (IR fragment) or smoothed by exp(-linspace(0,5,ker_len))
 * (scanline; `aux` = n samples of scratch in the pool).  One CTA per event. */
/* MS_SY_CHAOS (gen_micro_chaos, main_v2.py:303-315) also runs in ms_synth_table: f_over_sr = r, ring_decay = gate,
 * env_decay = y0 = (seed % 10000) / 10000, the PCG64 state as for the normal modes, `aux` = n samples of scratch. */
/* MS_SY_STICK (gen_stick_slip, main_v2.py:283-301): ms_synth_normal first leaves the event's n raw normals at `aux`
 * (the model draws exactly one per sample), ms_synth_table then walks the two-state friction model sequentially with
 * the reference's float64 operation order: f_over_sr = threshold, ring_decay = build, env_decay = decay, inv_fade = noise. */
/* ms_synth_table_f32 / ms_synth_table_f64: declared below by MS_DECLARE_API */
/* MS_SY_WAVELET events: sum of shifted Gaussian-windowed cosines under a Hann window (float64 phase) */
/* ms_synth_wavelet_f32 / ms_synth_wavelet_f64: declared below by MS_DECLARE_API */

/* ---- overlap-add placement + ADSR (main_v2.py:742-764, 172-195) ---- */
typedef struct {
    int64_t out;              /* offset of the render's mono buffer */
    int32_t out_n;
    int32_t ev_begin, ev_end; /* placed events, ascending */
    int32_t max_len;
    int32_t A, D_end, sus_end;
    int32_t has_release;
    double inv_A, inv_D, inv_R;
    double S, curve;
    int64_t env;              /* >= 0: offset in envpool of a precomputed envelope shared by several renders
                                 (ms_adsr_tables); < 0: evaluate make_adsr in closed form per sample */
} ms_ola_render;
typedef struct {
    int64_t grain;            /* pool offset of grain[offset] */
    int32_t start, len;
    double amp;
} ms_ola_evt;
/* ms_adsr_tables: make_adsr (main_v2.py:172-195) evaluated once per distinct envelope of the batch (a preset
 * sweep shares one); dev_reps[i].env is where table i goes, its other fields describe the envelope. */
/* ms_adsr_tables_f32 / ms_adsr_tables_f64: declared below by MS_DECLARE_API */
/* ms_overlap_add_f32 / ms_overlap_add_f64: declared below by MS_DECLARE_API */

/* ---- early-reflection cloud + short IR as one FIR (main_v2.py:409-421, 438-445), applied by
 *      FFT overlap-save ---- */
typedef struct {
    int64_t ir;               /* offset of the IR taps in irpool */
    int32_t ir_len;
    int32_t h_len;            /* ir_len + max tap delay */
    int64_t h;                /* unused (kept for layout stability) */
    int32_t tap_begin, tap_end;
    int64_t x, y;             /* offsets of the render's mono input / output */
    int32_t out_n;
    int32_t x_begin, x_end;   /* support of the input: samples outside [x_begin, x_end) are exactly zero */
    int32_t _pad;
} ms_fir_render;
/* The cloud and the IR are both causal LTI filters.  Route by row: ir_len <= 8192 -- the library keeps the spectrum of
 * every distinct IR (computed once in ms_fir_create) and composes IRspec * (1 + FFT(cloud taps)) per render;
 * 8192 < ir_len <= 2^21 (EXTENSION: the reference cuts at 8192) -- the cloud runs first as its own pass into the workspace,
 * then the IR as uniformly partitioned overlap-save with partition spectra computed once per distinct (ir, ir_len,
 * partition length), using only min(ir_len, out_n - x_begin) taps (the others cannot reach y[:out_n]).  A batch may mix
 * both; longer IRs fail in ms_fir_workspace_bytes / ms_fir_create.  ms_fir_run allocates nothing and never synchronises. */
/* ms_fir_workspace_bytes_f32 / ms_fir_workspace_bytes_f64: declared below by MS_DECLARE_API */
/* ms_fir_create_f32 / ms_fir_create_f64: declared below by MS_DECLARE_API */
/* ms_fir_run_f32 / ms_fir_run_f64: declared below by MS_DECLARE_API */
/* ms_fir_destroy_f32 / ms_fir_destroy_f64: declared below by MS_DECLARE_API */

/* ---- stereo diffusion + soft clip + normalise (main_v2.py:423-436, 31-34, 26-29) ---- */
#define MS_POST_K 12
typedef struct {
    int64_t y;                /* mono input offset */
    int64_t out;              /* output offset in frames */
    int64_t rbuf;             /* offset in `mono` of the right channel: written by ms_post (modes 1, 3), read (mode 2) */
    int32_t n;
    int32_t stereo_mode;      /* 0 duplicate, 1 Bessel FIR of y (even n), 2 precomputed, 3 Bessel FIR (even n) of the n
                                 samples at rbuf - n (a second mono signal: the right channel's own FIR output under
                                 space_ir_stereo), written at rbuf; the left channel is roll(y, dl) in modes 1-3 */
    int32_t dl, dr;
    double drive, inv_tanh_drive, peak;
    double coef[2 * MS_POST_K + 1];  /* J_m(theta), m = -K..K */
} ms_post_render;
/* ms_post_f32 / ms_post_f64: declared below by MS_DECLARE_API */
/* ms_roll_f32 / ms_roll_f64: declared below by MS_DECLARE_API */
/* EXTENSION (the reference delivers every render at base_sr): an export sample rate.  ms_post_export runs the max pass of
 * ms_post (the same kernel) on the renders of `dev_renders`, then, instead of its write pass, resamples each channel of the
 * clipped and normalised signal x = soft_clip(.) * scale, in the working precision, by up / down as
 * scipy.signal.resample_poly(x, up, down) defines it:
 *     out[m] = sum_j x[j] g[m down - j up + half],  0 <= m < ceil(n up / down),
 * g = up * firwin(2 half + 1, 1 / max(up, down), window=("kaiser", 5.0)), half = 10 max(up, down), g zero outside
 * [0, 2 half].  The filter arrives as a polyphase bank: phase p = (m down) mod up holds `taps` = rate[3] coefficients,
 * entry s + A of phase p being g[p + half - s up] (zero outside g) for s = -A .. taps - 1 - A, A = half / up; with
 * q = (m down) div up, out[m] = sum_s x[q + s] bank[p][s + A].  The output is interleaved float32 stereo at `out`; there is
 * no renormalisation after the resampler, so inter-sample peaks may exceed `peak`.  Row i of dev_export belongs to row i of
 * dev_renders.  max_n: largest n, max_out_n: largest out_end - out.  Allocates nothing, never synchronises. */
typedef struct {
    int64_t out, out_end;     /* output frames [out, out_end); under ms_post_pcm, out is the first slot and out_end - out the
                                 frame count */
    int64_t bank, bank_end;   /* the render's polyphase bank in the bank pool: up * taps coefficients */
    int32_t rate[4];          /* up, down, half, taps per phase */
} ms_export_render;
/* ms_post_export_f32 / ms_post_export_f64: declared below by MS_DECLARE_API */
/* EXTENSION (the reference delivers float samples): integer PCM output.  ms_post_pcm runs the max pass of ms_post (the
 * same kernel) on the renders of `dev_renders`, then a write pass that stores each output frame as signed `bits`-bit PCM
 * instead of float32.  The input of the quantiser is the value the float path rounds to float32 -- soft_clip(.) * scale,
 * or the resampler's sum when `dev_export` is not NULL (then row i of dev_export belongs to row i of dev_renders, and
 * out_end - out is its frame count) -- widened to double.  With S = 2^(bits - 1), each channel of output frame i becomes
 *     q = clamp(rint(x S + d), -S, S - 1)      (rint: round half to even; x S is exact, so one rounding)
 * d = 0 without dither.  With dither, d is TPDF from Philox4x32-10 (Random123), a pure function of the key and i:
 * counter (i mod 2^32, i >> 32, 0x64697468, 0), key (key[0], key[1]); of the output words w0..w3, d_L = (w0 - w1) 2^-32,
 * d_R = (w2 - w3) 2^-32.  Stored form, at byte 8 * out of `out` (`out` counted in 8-byte slots, as a float frame is): little-
 * endian two's complement, interleaved L, R -- 4 bytes a frame (bits 16) or 6 (bits 24).  A render of n frames (n of
 * its ms_post_render row, or out_end - out of its export row) owns ceil(n / 2) (16) or ceil(3 n / 4) (24) slots; the
 * bytes of those slots past its last frame are written as zero.  Every row must carry the call's `bits` (16 or 24) and
 * `dither` (0 or 1) in `fmt`; a row that does not is left unwritten.  max_n: largest n, max_out_n: largest out_end - out
 * (with dev_export).  Allocates nothing, never synchronises. */
typedef struct {
    uint32_t key[2];          /* Philox key: low and high 32 bits of the render's seed mod 2^64 */
    int32_t fmt[2];           /* bits (16 or 24), dither (1: TPDF, 0: none) */
} ms_pcm_render;
/* ms_post_pcm_f32 / ms_post_pcm_f64: declared below by MS_DECLARE_API */

/* ---- EXTENSION, not on the reference's path (SURVEY a14): band-limited polyphase decimation.  render() never decimates:
 *      the rate change is a relabel (main_v2.py:489-490), the band-limit is lowpass_fft (main_v2.py:39-59).  This stage
 *      exists because the task statement names it; its oracle is scipy.signal.upfirdn / resample_poly in float64, and it
 *      is "parity unpinned" by the reference.  y[s][m] = sum_k h[k] x[s][m q - k] (zero-extended), m < ceil((n + taps - 1) / q);
 *      taps <= 4096; x_stride / y_stride: elements between consecutive signals. ---- */
/* ms_polyphase_decimate_f32 / ms_polyphase_decimate_f64: declared below by MS_DECLARE_API */
/* ---- EXTENSION (the reference plays an impulse response at base_sr whatever its file rate): a batched rational
 *      resampler.  `space_ir_sr` resamples the IR to base_sr with it before the convolution.  For each of n_signals signals
 *      of n samples (x_stride / y_stride: elements between consecutive signals) and 0 <= m < n_out,
 *          y[s][m] = sum_j x[s][j] g[m down - j up + half]      (x zero outside [0, n); g zero outside [0, 2 half]),
 *      scipy.signal.resample_poly(x, up, down)'s sum when g is its filter and n_out = ceil(n up / down); a smaller n_out
 *      computes only the first outputs, each bitwise as in the full call.  `bank` is g as the polyphase bank of
 *      ms_export_render: phase p holds `taps` = half / up + (up - 1 + half) / up + 1 coefficients, entry t + A being
 *      g[p + half - t up] for t = -A .. taps - 1 - A, A = half / up; with q = (m down) div up, p = (m down) mod up,
 *      y[s][m] = sum_t x[s][q + t] bank[p][t + A], added in ascending t.  Allocates nothing, never synchronises; bad
 *      arguments (up, down < 1, half, n, n_signals, n_out < 0, taps that do not match, strides shorter than the signals)
 *      return -1 with ms_last_error(). ---- */
/* ms_resample_poly_f32 / ms_resample_poly_f64: declared below by MS_DECLARE_API */

/* ---- entry points.  Every stage exists in two precisions with identical signatures except for the
 *      element type of the signal buffers: suffix _f32 (float) and _f64 (double).  The interleaved stereo
 *      output of ms_post is float in both. ---- */
#define MS_DECLARE_API(SFX, REAL) \
    size_t ms_spectral_workspace_bytes##SFX(const ms_spec_job* host_jobs, int njobs); \
    int ms_spectral_apply##SFX(const ms_spec_job* host_jobs, int njobs, const REAL* src, REAL* dst, \
    void* workspace, size_t workspace_bytes, void* stream); \
    int ms_spectral_create##SFX(const ms_spec_job* host_jobs, int njobs, const REAL* src, REAL* dst, \
    void* workspace, size_t workspace_bytes, void* stream, void** handle); \
    int ms_spectral_run##SFX(void* handle, void* stream); \
    int ms_spectral_forward##SFX(void* handle, void* stream); \
    int ms_spectral_inverse##SFX(void* handle, void* stream); \
    int ms_spectral_z_table##SFX(void* handle, int64_t* host_z_offsets, size_t* z_base_bytes); \
    int ms_feedback##SFX(const ms_feedback_evt* dev_evts, int n_evts, int max_n, REAL* pool, void* stream); \
    int ms_imprint_step##SFX(const ms_imprint_step_evt* dev_evts, int n_evts, int max_bins, REAL* z_base, REAL* mem, \
    int32_t* prev_bins, void* stream); \
    int ms_waveguide##SFX(const ms_wg_evt* dev_evts, int n_evts, const ms_wg_line* dev_lines, REAL* pool, void* stream); \
    int ms_resonator##SFX(const ms_res_evt* dev_evts, int n_evts, const ms_res_mode* dev_modes, REAL* pool, void* stream); \
    int ms_partial_lock##SFX(const ms_plock_evt* dev_evts, int n_evts, REAL* z_base, REAL* scratch, void* stream); \
    int ms_cepstral##SFX(int step, const ms_cep_evt* dev_evts, int n_evts, int max_n, REAL* z1_base, REAL* z2_base, \
    REAL* z3_base, REAL* scratch, void* stream); \
    int ms_imprint##SFX(const ms_imprint_evt* dev_evts, const ms_imprint_render* dev_renders, int n_renders, int max_bins, \
    REAL* z_base, void* stream); \
    void ms_spectral_destroy##SFX(void* handle); \
    int ms_fft_pair_forward##SFX(const REAL* a, const REAL* b, int n, REAL* z_out, \
    void* workspace, size_t workspace_bytes, void* stream); \
    size_t ms_fft_pair_workspace_bytes##SFX(int n); \
    int ms_synth_normal##SFX(const ms_synth_evt* dev_evts, int n_evts, REAL* pool, void* stream); \
    int ms_synth_dust##SFX(const ms_synth_evt* dev_evts, int n_evts, const int32_t* dust_pos, const REAL* dust_val, \
    REAL* pool, void* stream); \
    int ms_synth_tilt_finish##SFX(const ms_synth_evt* dev_evts, int n_evts, REAL* pool, void* stream); \
    int ms_synth_table##SFX(const ms_synth_evt* dev_evts, int n_evts, const REAL* dust_val, REAL* pool, void* stream); \
    int ms_synth_wavelet##SFX(const ms_synth_evt* dev_evts, int n_evts, const ms_wavelet_atom* atoms, const int32_t* shifts, \
    REAL* pool, void* stream); \
    int ms_adsr_tables##SFX(const ms_ola_render* dev_reps, int n_tables, int max_out_n, REAL* envpool, void* stream); \
    int ms_overlap_add##SFX(const ms_ola_render* dev_renders, int n_renders, int max_out_n, const ms_ola_evt* dev_evts, \
    const REAL* pool, const REAL* envpool, REAL* mono, void* stream); \
    size_t ms_fir_workspace_bytes##SFX(const ms_fir_render* host_renders, int n_renders); \
    int ms_fir_create##SFX(const ms_fir_render* host_renders, int n_renders, const REAL* irpool, const int32_t* tap_off, \
    const REAL* tap_gain, const REAL* mono_in, REAL* mono_out, void* workspace, size_t workspace_bytes, void* stream, \
    void** handle); \
    int ms_fir_run##SFX(void* handle, void* stream); \
    void ms_fir_destroy##SFX(void* handle); \
    int ms_post##SFX(const ms_post_render* dev_renders, int n_renders, int max_n, REAL* mono, uint64_t* maxbits, \
    float* out, void* stream); \
    int ms_post_export##SFX(const ms_post_render* dev_renders, const ms_export_render* dev_export, int n_renders, int max_n, \
    int max_out_n, REAL* mono, uint64_t* maxbits, const REAL* bank, float* out, void* stream); \
    int ms_post_pcm##SFX(const ms_post_render* dev_renders, const ms_pcm_render* dev_pcm, const ms_export_render* dev_export, \
    int n_renders, int max_n, int max_out_n, int bits, int dither, REAL* mono, uint64_t* maxbits, const REAL* bank, void* out, \
    void* stream); \
    int ms_roll##SFX(const REAL* src, REAL* dst, int n, int shift, void* stream); \
    int ms_polyphase_decimate##SFX(const REAL* x, int64_t x_stride, int n, int n_signals, const REAL* h, int taps, int q, \
    REAL* y, int64_t y_stride, void* stream); \
    int ms_resample_poly##SFX(const REAL* x, int64_t x_stride, int n, int n_signals, const REAL* bank, int up, int down, \
    int half, int taps, REAL* y, int64_t y_stride, int n_out, void* stream);
MS_DECLARE_API(_f32, float)
MS_DECLARE_API(_f64, double)

#ifdef __cplusplus
}
#endif
#endif
