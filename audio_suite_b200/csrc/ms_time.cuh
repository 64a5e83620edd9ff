// ms_time.cuh -- time-domain stages of render(): overlap-add placement + ADSR (main_v2.py:742-764,
// 172-195), the reflection-cloud / impulse-response FIR builder (main_v2.py:409-421, 438-445), and the
// stereo / soft-clip / normalise tail (main_v2.py:423-436, 31-34, 26-29, 775-781).

#define OLA_TILE 1024
#define OLA_NTHR 256
#define POST_K MS_POST_K          // Bessel taps -K..K of the stereo rotation
#define POST_NC (2 * POST_K + 1)
#define POST_HALF (OLA_TILE / 2 + 2 * POST_K + 4)            // samples of one parity in a tile's window (+ quad slack)
#define POST_PAR (POST_HALF + POST_HALF / 4 + 2)             // ... with the one-in-four skew

// ---- overlap-add ("unfold" placement) + ADSR --------------------------------------------------------
typedef ms_ola_render OlaRender;
typedef ms_ola_evt OlaEvt;


MS_DEV real adsr_gain(const OlaRender& R, int i) {      // (kept inline: an out-of-line call was measured slower, 1.56 -> 2.05 ms)
    // Evaluated in the working precision: an error relative to a loud sample is still an error relative
    // to the peak, and the FIR gain + soft clip downstream turn 1e-7 of that into 1e-5 (DESIGN.md, precision).
    const real S = (real)R.S, curve = (real)R.curve;
    if (i < R.A) return r_pow((real)((double)i * R.inv_A), curve);
    if (i < R.D_end) return (real)1.0 - ((real)1.0 - S) * r_pow((real)((double)(i - R.A) * R.inv_D), curve);
    if (i < R.sus_end || !R.has_release) return S;
    const real r = (i == R.out_n - 1 && R.out_n - R.sus_end > 1) ? (real)1.0 : (real)((double)(i - R.sus_end) * R.inv_R);
    return S * ((real)1.0 - r_pow(r, curve));
}

// grid = (ceil(max out_n / OLA_TILE), renders), block = OLA_NTHR.  Gather form: every output sample
// sums the events that cover it, in event order, so no atomics and each output is written once.
// envelope tables: one per distinct ADSR description that several renders of the batch share
MS_DEV void adsr_table_body(const OlaRender* MS_RESTRICT reps, real* MS_RESTRICT envpool, const Ctx& c) {
    const OlaRender R = reps[c.by];
    const int t0 = c.bx * OLA_TILE;
    const int t1 = (t0 + OLA_TILE) < R.out_n ? (t0 + OLA_TILE) : R.out_n;
    for (int i = t0 + c.tid; i < t1; i += c.nthr) envpool[R.env + i] = adsr_gain(R, i);
}

// (ncu has this kernel waiting on its chain of dependent global loads -- render record, event record, grain samples,
//  envelope: long scoreboard 18.6 warps per issue, 27 % of the issue slots.  Tiles of 2048 samples, i.e. half as many
//  chains, were measured SLOWER on B200: 1.52 -> 1.58 ms on the C5 sweep.)
#define OLA_ATILE OLA_TILE
MS_DEV void ola_adsr_body(const OlaRender* MS_RESTRICT renders, const OlaEvt* MS_RESTRICT evts,
                          const real* MS_RESTRICT pool, const real* MS_RESTRICT envpool, real* MS_RESTRICT mono, const Ctx& c) {
    const OlaRender R = renders[c.by];
    const int t0 = c.bx * OLA_ATILE;
    if (t0 >= R.out_n) return;
    const int t1 = (t0 + OLA_ATILE) < R.out_n ? (t0 + OLA_ATILE) : R.out_n;
    // candidates: start < t1 and start > t0 - max_len
    int lo = R.ev_begin, hi = R.ev_end;
    while (lo < hi) { const int m = (lo + hi) >> 1; if (evts[m].start >= t1) hi = m; else lo = m + 1; }
    const int eb = lo;
    lo = R.ev_begin; hi = eb;
    while (lo < hi) { const int m = (lo + hi) >> 1; if (evts[m].start > t0 - R.max_len) hi = m; else lo = m + 1; }
    const int ea = lo;
    real* out = mono + R.out;
    // every thread owns OLA_ATILE / OLA_NTHR samples (i = t0 + tid + q * nthr) and keeps their sums in registers;
    // events are the outer loop (one descriptor fetch per event, not per sample) and are added in event order,
    // so each output sample sees the same sequence of additions as out[start:start+L] += amp * g (main_v2.py:755)
    real acc[OLA_ATILE / OLA_NTHR];
#pragma unroll
    for (int q = 0; q < OLA_ATILE / OLA_NTHR; ++q) acc[q] = (real)0.;
    for (int e = ea; e < eb; ++e) {
        const int st = __ldg(&evts[e].start), ln = __ldg(&evts[e].len);
        const real amp = (real)__ldg(&evts[e].amp);
        const real* g = pool + evts[e].grain;
#pragma unroll
        for (int q = 0; q < OLA_ATILE / OLA_NTHR; ++q) {
            const int k = t0 + c.tid + q * OLA_NTHR - st;
            if (k >= 0 && k < ln) acc[q] += amp * __ldg(&g[k]);
        }
    }
#pragma unroll
    for (int q = 0; q < OLA_ATILE / OLA_NTHR; ++q) {
        const int i = t0 + c.tid + q * OLA_NTHR;
        if (i < t1) out[i] = acc[q] * (R.env >= 0 ? __ldg(&envpool[R.env + i]) : adsr_gain(R, i));
    }
}

// ---- reflection cloud as a dense tap vector: e[off_t] += g_t  (early_reflection_cloud, main_v2.py:413-420) ----
// The cloud and the impulse response are both causal LTI filters, so they are applied as ONE filter whose
// spectrum is IRspec * (1 + FFT(e)); e is only max_off + 1 samples long.
typedef ms_fir_render FirRender;
struct ErJob { long long e; int elen, tap_begin, tap_end; };
MS_DEV void er_scatter_body(const ErJob* MS_RESTRICT jobs, const int* MS_RESTRICT tap_off, const real* MS_RESTRICT tap_gain,
                            real* ebase, const Ctx& c) {
    const ErJob J = jobs[c.by];
    real* e = ebase + J.e;
    for (int i = c.tid; i < J.elen; i += c.nthr) e[i] = (real)0.;
    c.sync();
    // Several taps may share a delay.  No atomics: the FIRST tap of a delay sums every later tap of that delay in tap
    // order and writes the sum, so the result does not depend on the thread schedule (O(taps^2) compares per render,
    // taps <= 4096; the tap table is L1-resident).
    for (int t = J.tap_begin + c.tid; t < J.tap_end; t += c.nthr) {
        const int off = __ldg(&tap_off[t]);
        if (off < 0 || off >= J.elen) continue;
        bool first = true;
        for (int u = J.tap_begin; u < t; ++u) if (__ldg(&tap_off[u]) == off) { first = false; break; }
        if (!first) continue;
        real sum = __ldg(&tap_gain[t]);
        for (int u = t + 1; u < J.tap_end; ++u) if (__ldg(&tap_off[u]) == off) sum += __ldg(&tap_gain[u]);
        e[off] = sum;
    }
}

// ---- stereo diffusion + soft clip + normalise -----------------------------------------------------------
typedef ms_post_render PostRender;
MS_DEV int wrap_idx(long long i, int n) { long long r = i % n; if (r < 0) r += n; return (int)r; }
// the clipped value is stored as float32, so tanh is evaluated in float32 (argument rounded once: 6e-8 relative)
MS_DEV real soft_clip(real v, real drive, real inv_t) { return drive > (real)0. ? (real)tanhf((float)(v * drive)) * inv_t : v; }

// The right channel of an even-length render over one tile: R[i] = sum_m J_m y[(i + dr + 2 m) mod n] (25 Bessel taps at
// even lags).  The tile's input window (1024 + 4K samples, circular) is staged in shared memory de-interleaved into
// its even and odd samples (each parity is a dense 25-tap FIR of its own), every four samples skewed by one slot so
// that threads working on quads of outputs hit distinct banks; results land in `res` (slot of output j: j + (j >> 3)).
// Pass 1 keeps the result at rbuf for pass 2.  (Recomputing the taps in pass 2 instead -- 40 N -> 24 N bytes of HBM
// traffic per render -- was measured SLOWER on B200: max pass 2.66 -> 2.40 ms but write pass 2.18 -> 3.00 ms.  These
// passes are bound by the per-tile latency chain (stage, barrier, taps, barrier), not by bandwidth.)
MS_DEV void post_right_tile(const PostRender& R, const real* MS_RESTRICT y, int t0, int len, real* win, real* coef, real* res, const Ctx& c) {
    const int n = R.n;
    const int W = len + 4 * POST_K;
    const int w0 = wrap_idx((long long)t0 + R.dr - 2 * POST_K, n);          // one 64-bit modulo per thread
    {
        // every load of the window is issued before the first store (ncu: one loop body per sample made each STS wait
        // out its own LDG)
        constexpr int NQ = (OLA_TILE + 4 * POST_K + OLA_NTHR - 1) / OLA_NTHR;
        real tmp[NQ];
#pragma unroll
        for (int q = 0; q < NQ; ++q) {
            const int j = c.tid + OLA_NTHR * q;
            int idx = w0 + j;
            if (idx >= n) { idx -= n; if (idx >= n) idx %= n; }              // second wrap only for n < tile
            tmp[q] = j < W ? y[idx] : (real)0.;
        }
#pragma unroll
        for (int q = 0; q < NQ; ++q) {
            const int j = c.tid + OLA_NTHR * q, mm = j >> 1;
            if (j < W) win[(j & 1) * POST_PAR + mm + (mm >> 2)] = tmp[q];
        }
    }
    for (int j = c.tid; j < POST_NC; j += c.nthr) coef[j] = (real)R.coef[j];
    c.sync();
    // thread -> parity (warp-uniform) and a quad of consecutive outputs of that parity: 28 loads per 4 outputs
    for (int u = c.tid; u < OLA_TILE / 4; u += c.nthr) {
        const int par = u / (OLA_TILE / 8), t = u - par * (OLA_TILE / 8);
        if (8 * t + par >= len) continue;
        const real* w = win + par * POST_PAR + 5 * t;     // slot of sample m0 = 4t: 4t + t
        real a0 = (real)0., a1 = (real)0., a2 = (real)0., a3 = (real)0.;
        real x0 = w[0], x1 = w[1], x2 = w[2];
        struct alignas(2 * sizeof(real)) CoefPair { real a, b; };
        const CoefPair* cp = (const CoefPair*)coef;          // two coefficients per (broadcast) load: coef sits at an even offset, POST_NC + 1 entries
#pragma unroll
        for (int k = 0; k < POST_NC; ++k) {
            const real x3 = w[(k + 3) + ((k + 3) >> 2)];
            const CoefPair pr = cp[k >> 1];
            const real ck = (k & 1) ? pr.b : pr.a;
            a0 += ck * x0; a1 += ck * x1; a2 += ck * x2; a3 += ck * x3;
            x0 = x1; x1 = x2; x2 = x3;
        }
        const int j0 = 9 * t + par;                  // slot of output j = 8t + par + 2q is j + (j >> 3): stride 9, conflict-free
        res[j0] = a0; res[j0 + 2] = a1; res[j0 + 4] = a2; res[j0 + 6] = a3;
    }
    c.sync();
}
// block-wide maximum of non-negative values: warp shuffles, then one value per warp through shared memory
MS_DEV real block_max(real m, real* red, const Ctx& c) {
#ifdef MS_HOST_EMUL
    red[c.tid] = m;
    c.sync();
    for (int s = c.nthr >> 1; s > 0; s >>= 1) {
        if (c.tid < s) red[c.tid] = r_max(red[c.tid], red[c.tid + s]);
        c.sync();
    }
    const real r = red[0];
    c.sync();
    return r;
#else
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = r_max(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((c.tid & 31) == 0) red[c.tid >> 5] = m;
    c.sync();
    real r = (c.tid & 31) < (c.nthr >> 5) ? red[c.tid & 31] : (real)0.;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) r = r_max(r, __shfl_xor_sync(0xffffffffu, r, o));
    c.sync();
    return r;
#endif
}
// pass 1: per-render max(|L|, |R|) before the clip (tanh is monotonic, so the clipped max follows).
MS_DEV void post_max_body(const PostRender* MS_RESTRICT renders, real* mono, unsigned long long* MS_RESTRICT maxbits, const Ctx& c) {
    const PostRender& R = renders[c.by];
    const int n = R.n, mode = R.stereo_mode;
    const int t0 = c.bx * OLA_TILE;
    if (t0 >= n) return;
    const int t1 = (t0 + OLA_TILE) < n ? (t0 + OLA_TILE) : n;
    const real* y = mono + R.y;
    real* win = (real*)c.smem;                       // 2 * POST_PAR
    real* coef = win + 2 * POST_PAR;                  // POST_NC (+1)
    real* red = coef + POST_NC + 1;                  // nthr
    real* res = red + OLA_NTHR;                      // OLA_TILE results, stream order
    const int len = t1 - t0;
    real m = (real)0.;
    if (mode == 1 || mode == 3) {                    // mode 3: the right channel is made from the n samples before rbuf
        post_right_tile(R, mode == 3 ? mono + R.rbuf - n : y, t0, len, win, coef, res, c);
        real yv[OLA_TILE / OLA_NTHR];
#pragma unroll
        for (int q = 0; q < OLA_TILE / OLA_NTHR; ++q) { const int j = c.tid + OLA_NTHR * q; yv[q] = j < len ? y[t0 + j] : (real)0.; }
#pragma unroll
        for (int q = 0; q < OLA_TILE / OLA_NTHR; ++q) {
            const int j = c.tid + OLA_NTHR * q;
            if (j < len) {
                const real r = res[j + (j >> 3)];
                mono[R.rbuf + t0 + j] = r;
                m = r_max(m, r_max(r_abs(r), r_abs(yv[q])));
            }
        }
    } else {
        for (int i = t0 + c.tid; i < t1; i += c.nthr) {
            m = r_max(m, r_abs(y[i]));
            if (mode == 2) m = r_max(m, r_abs(mono[R.rbuf + i]));
        }
    }
    m = block_max(m, red, c);
    if (c.tid == 0) {
        union { double f; unsigned long long u; } cv; cv.f = (double)m;
#ifdef MS_HOST_EMUL
        if (cv.u > maxbits[c.by]) maxbits[c.by] = cv.u;
#else
        atomicMax(&maxbits[c.by], cv.u);       // non-negative doubles order like their bit patterns
#endif
    }
}
// ---- EXTENSION: integer PCM output (include/microsound_b200.h, ms_post_pcm) ----
// The write passes below take the store as a compile-time policy: BITS 0 stores float2 frames (ms_post, ms_post_export:
// the code they always had), BITS 16 / 24 store PCM, with DITHER on or off (the dither-off passes hold no Philox code).
typedef ms_pcm_render PcmRender;
#define PCM_TILE_BYTES (6 * OLA_TILE)        // pcm24: one tile of 1024 frames staged in shared memory
// Philox4x32-10 (Salmon et al., SC'11; Random123's philox4x32 with 10 rounds): the counter c becomes the output words
MS_DEV void philox4x32_10(uint32_t c[4], uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        if (r) { k0 += 0x9E3779B9u; k1 += 0xBB67AE85u; }
        const uint32_t hi0 = __umulhi(0xD2511F53u, c[0]), lo0 = 0xD2511F53u * c[0];
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c[2]), lo1 = 0xCD9E8D57u * c[2];
        c[0] = hi1 ^ c[1] ^ k0; c[1] = lo1; c[2] = hi0 ^ c[3] ^ k1; c[3] = lo0;
    }
}
// q = clamp(rint(x S + d), -S, S - 1), S = 2^(BITS - 1), in double: x S is exact, so there is one rounding
template <int BITS> MS_DEV int pcm_quant(double x, double d) {
    const double S = (double)(1 << (BITS - 1));
    return (int)fmin(fmax(rint(x * S + d), -S), S - 1.0);
}
// output frame i of a PCM render of n frames: dither, quantise, store (pcm16: one 32-bit word per frame at o; pcm24: 6 bytes
// at slot j of the staged tile, written as three 16-bit halves)
template <int BITS, bool DITHER>
MS_DEV void pcm_frame(const PcmRender& P, long long n, long long i, double l, double r, unsigned char* o, char* stage, int j) {
    double dl = 0.0, dr = 0.0;
    if (DITHER) {
        uint32_t w[4] = {(uint32_t)i, (uint32_t)((unsigned long long)i >> 32), 0x64697468u, 0u};
        philox4x32_10(w, P.key[0], P.key[1]);
        dl = ((double)w[0] - (double)w[1]) * 2.3283064365386963e-10;     // 2^-32: exact, triangular on (-1, 1)
        dr = ((double)w[2] - (double)w[3]) * 2.3283064365386963e-10;
    }
    const uint32_t ql = (uint32_t)pcm_quant<BITS>(l, dl), qr = (uint32_t)pcm_quant<BITS>(r, dr);
    if (BITS == 16) {
        ((uint32_t*)o)[i] = (ql & 0xffffu) | (qr << 16);
        if (i == n - 1 && (n & 1)) ((uint32_t*)o)[i + 1] = 0u;                      // the rest of the last slot
    } else {
        unsigned short* s = (unsigned short*)(stage + 6 * j);
        s[0] = (unsigned short)ql; s[1] = (unsigned short)(((ql >> 16) & 0xffu) | ((qr & 0xffu) << 8)); s[2] = (unsigned short)(qr >> 8);
    }
}
// pcm24: the staged tile of cnt frames, from frame f0 (a multiple of OLA_TILE, so byte 6 f0 is 8-aligned), as 8-byte words;
// the last word's bytes past the tile are zero (they lie in the render's own last slot)
MS_DEV void pcm24_flush(char* stage, unsigned char* o, long long f0, int cnt, const Ctx& c) {
    const int nb = 6 * cnt, nw = (nb + 7) >> 3;
    if (c.tid < 8 * nw - nb) stage[nb + c.tid] = 0;
    c.sync();
    unsigned long long* d = (unsigned long long*)(o + 6 * f0);
    const unsigned long long* s = (const unsigned long long*)stage;
    for (int w = c.tid; w < nw; w += c.nthr) d[w] = s[w];
}
// pass 2: write interleaved stereo, clipped and scaled to the requested peak (modes 1-3 read the right channel at rbuf)
template <int BITS, bool DITHER>
MS_DEV void post_write_body(const PostRender* MS_RESTRICT renders, const PcmRender* MS_RESTRICT pcms, const real* MS_RESTRICT mono,
                            const unsigned long long* MS_RESTRICT maxbits, float2* MS_RESTRICT out, const Ctx& c) {
    const PostRender& R = renders[c.by];
    const int t0 = c.bx * OLA_TILE;
    if (t0 >= R.n) return;
    const int t1 = (t0 + OLA_TILE) < R.n ? (t0 + OLA_TILE) : R.n;
    const real* y = mono + R.y;
    const int mode = R.stereo_mode;
    union { double f; unsigned long long u; } cv; cv.u = maxbits[c.by];
    const real drive = (real)R.drive, inv_t = (real)R.inv_tanh_drive;
    const real top = soft_clip((real)cv.f, drive, inv_t);
    const real scale = top > (real)0. ? (real)R.peak / top : (real)1.0;
    float2* o = out + R.out;
    const int dlm = mode ? wrap_idx((long long)R.dl, R.n) : 0;          // left channel = roll(y, dl)
    real lv[OLA_TILE / OLA_NTHR], rv[OLA_TILE / OLA_NTHR];
    const real* rsrc = mode ? mono + R.rbuf : y;
#pragma unroll
    for (int q = 0; q < OLA_TILE / OLA_NTHR; ++q) {
        const int i = t0 + c.tid + OLA_NTHR * q;
        int li = i - dlm; if (li < 0) li += R.n;
        lv[q] = i < t1 ? y[li] : (real)0.;
        rv[q] = i < t1 ? rsrc[i] : (real)0.;
    }
    if constexpr (BITS == 0) {
#pragma unroll
        for (int q = 0; q < OLA_TILE / OLA_NTHR; ++q) {
            const int i = t0 + c.tid + OLA_NTHR * q;
            if (i < t1) o[i] = make_float2((float)(soft_clip(lv[q], drive, inv_t) * scale), (float)(soft_clip(rv[q], drive, inv_t) * scale));
        }
    } else {
        const PcmRender P = pcms[c.by];
        if (P.fmt[0] != BITS || P.fmt[1] != (DITHER ? 1 : 0)) return;
        unsigned char* ob = (unsigned char*)o;
#pragma unroll
        for (int q = 0; q < OLA_TILE / OLA_NTHR; ++q) {
            const int i = t0 + c.tid + OLA_NTHR * q;
            if (i < t1) pcm_frame<BITS, DITHER>(P, R.n, i, (double)(soft_clip(lv[q], drive, inv_t) * scale), (double)(soft_clip(rv[q], drive, inv_t) * scale),
                                                ob, c.smem, i - t0);
        }
        if (BITS == 24) pcm24_flush(c.smem, ob, t0, t1 - t0, c);
    }
}
// ---- EXTENSION: export sample rate, the write pass of an exporting render (include/microsound_b200.h, ms_post_export) ----
// out[m] = sum_s x[q + s] bank[p][s + A], q = (m down) div up, p = (m down) mod up, x = soft_clip(.) * scale of each channel
// (zero outside [0, n)).  grid = (ceil(max output frames / EXP_TILE), renders), OLA_NTHR threads; a thread owns the outputs
// m0 + tid + OLA_NTHR k (stores of a warp are consecutive float2).  The tile's input window -- both channels, clipped and
// scaled on load -- goes through shared memory in rounds of EXP_CH frames; every output adds the taps that fall in the
// round, in ascending s, into the same two accumulators, so the sum does not depend on the rounds (heavy decimation
// spans many rounds: at 1/640 a tile of outputs reads 655360 input frames).  One bank load (read through L1) feeds both
// channels.  Products m down reach 4e10 (C4 at 640/147): 64-bit until the offsets inside the tile.
typedef ms_export_render ExportRender;
#define EXP_TILE 1024                // output frames per CTA
#define EXP_CH 2048                  // input frames per round of the staged window
template <int BITS, bool DITHER>
MS_DEV void post_export_body(const PostRender* MS_RESTRICT renders, const ExportRender* MS_RESTRICT exps, const PcmRender* MS_RESTRICT pcms,
                             const real* MS_RESTRICT mono, const unsigned long long* MS_RESTRICT maxbits, const real* MS_RESTRICT bank,
                             float2* MS_RESTRICT out, const Ctx& c) {
    const PostRender& R = renders[c.by];
    const ExportRender E = exps[c.by];
    const long long out_n = E.out_end - E.out;
    const long long m0 = (long long)c.bx * EXP_TILE;
    if (m0 >= out_n) return;
    const int cnt = (int)(out_n - m0 < EXP_TILE ? out_n - m0 : EXP_TILE);
    const long long up = E.rate[0], down = E.rate[1];
    const int taps = E.rate[3], A = E.rate[2] / E.rate[0];
    const int n = R.n, mode = R.stereo_mode;
    union { double f; unsigned long long u; } cv; cv.u = maxbits[c.by];
    const real drive = (real)R.drive, inv_t = (real)R.inv_tanh_drive;
    const real top = soft_clip((real)cv.f, drive, inv_t);
    const real scale = top > (real)0. ? (real)R.peak / top : (real)1.0;
    const real* y = mono + R.y;
    const real* rsrc = mode ? mono + R.rbuf : y;
    const int dlm = mode ? wrap_idx((long long)R.dl, n) : 0;           // left channel = roll(y, dl)
    const long long w0 = m0 * down / up - A;                            // input frame of window slot 0
    const int wlen = (int)((m0 + cnt - 1) * down / up + (taps - A) - w0);
    constexpr int NQ = EXP_TILE / OLA_NTHR, NL = EXP_CH / OLA_NTHR;
    int rq[NQ];                                  // window slot of q(m), -1: no output
    const real* tp[NQ];                          // taps of the output's phase, at s = 0
    real aL[NQ], aR[NQ];
#pragma unroll
    for (int k = 0; k < NQ; ++k) {
        const int i = c.tid + OLA_NTHR * k;
        const long long md = (m0 + i) * down, q = md / up;
        rq[k] = i < cnt ? (int)(q - w0) : -1;
        tp[k] = bank + E.bank + (md - q * up) * taps + A;
        aL[k] = aR[k] = (real)0.;
    }
    real* wl = (real*)c.smem;                    // EXP_CH frames of each channel
    real* wr = wl + EXP_CH;
    for (int c0 = 0; c0 < wlen; c0 += EXP_CH) {
        const int clen = wlen - c0 < EXP_CH ? wlen - c0 : EXP_CH;
        // every load of the round is issued before the first store
        real lv[NL], rv[NL];
#pragma unroll
        for (int k = 0; k < NL; ++k) {
            const int j = c.tid + OLA_NTHR * k;
            const long long J = w0 + c0 + j;
            lv[k] = rv[k] = (real)0.;
            if (j < clen && J >= 0 && J < n) {
                int li = (int)J - dlm; if (li < 0) li += n;
                lv[k] = y[li];
                rv[k] = rsrc[J];
            }
        }
        if (c0) c.sync();                        // the previous round has been read
#pragma unroll
        for (int k = 0; k < NL; ++k) {
            const int j = c.tid + OLA_NTHR * k;
            if (j < clen) { wl[j] = soft_clip(lv[k], drive, inv_t) * scale; wr[j] = soft_clip(rv[k], drive, inv_t) * scale; }
        }
        c.sync();
#pragma unroll
        for (int k = 0; k < NQ; ++k) {
            if (rq[k] < 0) continue;
            const int d = rq[k] - c0;            // slot of x[q] in this round
            const int s_lo = -A > -d ? -A : -d;
            const int s_hi = taps - 1 - A < clen - 1 - d ? taps - 1 - A : clen - 1 - d;
            real l = aL[k], r = aR[k];
            for (int s = s_lo; s <= s_hi; ++s) {
                const real h = __ldg(&tp[k][s]);
                l += h * wl[d + s];
                r += h * wr[d + s];
            }
            aL[k] = l; aR[k] = r;
        }
    }
    if constexpr (BITS == 0) {
        float2* o = out + E.out + m0;
#pragma unroll
        for (int k = 0; k < NQ; ++k)
            if (rq[k] >= 0) o[c.tid + OLA_NTHR * k] = make_float2((float)aL[k], (float)aR[k]);
    } else {
        // the dither is drawn here, after the accumulation: its registers do not compete with the tap loop's
        const PcmRender P = pcms[c.by];
        if (P.fmt[0] != BITS || P.fmt[1] != (DITHER ? 1 : 0)) return;
        unsigned char* ob = (unsigned char*)(out + E.out);
        if (BITS == 24) c.sync();                // the staged window is read by every thread: its space becomes the tile's
#pragma unroll
        for (int k = 0; k < NQ; ++k)
            if (rq[k] >= 0) pcm_frame<BITS, DITHER>(P, out_n, m0 + c.tid + OLA_NTHR * k, (double)aL[k], (double)aR[k], ob, c.smem, c.tid + OLA_NTHR * k);
        if (BITS == 24) pcm24_flush(c.smem, ob, m0, cnt, c);
    }
}
// ---- EXTENSION: batched rational resampler (include/microsound_b200.h, ms_resample_poly; `space_ir_sr` resamples the IR) ----
// y[s][m] = sum_t x[s][q + t] bank[p][t + A], q = (m down) div up, p = (m down) mod up (zero outside [0, n)): the tap loop of
// post_export_body for one plain signal.  grid = (ceil(n_out / RS_TILE), signals), OLA_NTHR threads; a thread owns the outputs
// m0 + tid + OLA_NTHR k.  The window goes through shared memory in rounds of RS_CH samples, every load of a round issued
// before its first store; each output adds the taps that fall in the round, in ascending t, into one accumulator, so the
// sum does not depend on the rounds.  (A separate body, not post_export_body with a load policy: that one clips, scales and
// reads two channels with the stereo roll on load, and keeping the post kernels' SASS unchanged forbids reshaping it.)
#define RS_TILE 1024                 // outputs per CTA
#define RS_CH 2048                   // input samples per round of the staged window
MS_DEV void resample_poly_body(const real* MS_RESTRICT x, long long x_stride, int n, const real* MS_RESTRICT bank, int up, int down,
                               int half, int taps, real* MS_RESTRICT y, long long y_stride, int n_out, const Ctx& c) {
    const long long m0 = (long long)c.bx * RS_TILE;
    if (m0 >= n_out) return;
    const int cnt = (int)(n_out - m0 < RS_TILE ? n_out - m0 : RS_TILE);
    const real* xs = x + (long long)c.by * x_stride;
    const int A = half / up;
    const long long w0 = m0 * down / up - A;                            // input sample of window slot 0
    const int wlen = (int)((m0 + cnt - 1) * down / up + (taps - A) - w0);
    constexpr int NQ = RS_TILE / OLA_NTHR, NL = RS_CH / OLA_NTHR;
    int rq[NQ];                                  // window slot of q(m), -1: no output
    const real* tp[NQ];                          // taps of the output's phase, at t = 0
    real acc[NQ];
#pragma unroll
    for (int k = 0; k < NQ; ++k) {
        const int i = c.tid + OLA_NTHR * k;
        const long long md = (m0 + i) * down, q = md / up;
        rq[k] = i < cnt ? (int)(q - w0) : -1;
        tp[k] = bank + (md - q * up) * taps + A;
        acc[k] = (real)0.;
    }
    real* win = (real*)c.smem;                   // RS_CH samples
    for (int c0 = 0; c0 < wlen; c0 += RS_CH) {
        const int clen = wlen - c0 < RS_CH ? wlen - c0 : RS_CH;
        real v[NL];
#pragma unroll
        for (int k = 0; k < NL; ++k) {
            const int j = c.tid + OLA_NTHR * k;
            const long long J = w0 + c0 + j;
            v[k] = (j < clen && J >= 0 && J < n) ? __ldg(&xs[J]) : (real)0.;
        }
        if (c0) c.sync();                        // the previous round has been read
#pragma unroll
        for (int k = 0; k < NL; ++k) {
            const int j = c.tid + OLA_NTHR * k;
            if (j < clen) win[j] = v[k];
        }
        c.sync();
#pragma unroll
        for (int k = 0; k < NQ; ++k) {
            if (rq[k] < 0) continue;
            const int d = rq[k] - c0;            // slot of x[q] in this round
            const int t_lo = -A > -d ? -A : -d;
            const int t_hi = taps - 1 - A < clen - 1 - d ? taps - 1 - A : clen - 1 - d;
            real a = acc[k];
            for (int t = t_lo; t <= t_hi; ++t) a += __ldg(&tp[k][t]) * win[d + t];
            acc[k] = a;
        }
    }
    real* ys = y + (long long)c.by * y_stride + m0;
#pragma unroll
    for (int k = 0; k < NQ; ++k)
        if (rq[k] >= 0) ys[c.tid + OLA_NTHR * k] = acc[k];
}
// circular shift used by the odd-length stereo path: dst[i] = src[(i + shift) mod n]
MS_DEV void roll_body(const real* MS_RESTRICT src, real* MS_RESTRICT dst, int n, int shift, const Ctx& c) {
    for (int i = c.bx * c.nthr + c.tid; i < n; i += c.nthr * 64) dst[i] = src[wrap_idx((long long)i + shift, n)];
}

// ---- spectral imprint (SpectralImprint.apply, main_v2.py:565-581) ----------------------------------------------
// grid = (ceil(max_bins / nthr), renders): a thread owns one rfft bin of one render and walks that render's grains
// in event order, carrying the moving average of the magnitude in a register.  The average restarts whenever the
// spectrum length differs from the previous imprinted grain's (M:575).  Spectra are those of single-signal jobs
// (Z = DFT of the real grain); only bins 0..n/2 are rewritten, the inverse transform mirrors them (irfft).
typedef ms_imprint_evt ImprintEvt;
typedef ms_imprint_render ImprintRender;
MS_DEV void imprint_body(const ImprintEvt* MS_RESTRICT evts, const ImprintRender* MS_RESTRICT renders, cpx* zbase, const Ctx& c) {
    const ImprintRender R = renders[c.by];
    const int k = c.bx * c.nthr + c.tid;
    const real amount = (real)R.amount, smooth = (real)R.smooth;
    real mem = (real)0.;
    int prev_bins = -1;
    for (int e = R.ev_begin; e < R.ev_end; ++e) {
        const int n = evts[e].n, bins = n / 2 + 1;
        if (k < bins) {
            cpx* Z = zbase + evts[e].z;
            const cpx X = Z[k];
            const real mag = (real)hypot((double)X.x, (double)X.y);
            mem = (bins != prev_bins) ? mag : smooth * mem + ((real)1.0 - smooth) * mag;
            const real mag2 = ((real)1.0 - amount) * mag + amount * mem;
            Z[k] = mag > (real)0. ? c_scale(X, mag2 / mag) : mk(mag2, (real)0.);     // angle(0) = 0
        }
        prev_bins = bins;
    }
}

// ---- partial lock (partial_lock_stretch, main_v2.py:130-148) ------------------------------------------------------
// One CTA per grain.  (1) W[k] = low-pass / power-warp of the grain's spectrum and its magnitude, for every rfft bin;
// (2) the magnitude of the top_n-th strongest bin (k >= 1) by bisection on the bit pattern of the non-negative
// magnitudes (monotone), a block-wide count per step; (3) Y = 0.12 W, then every selected bin adds
// W[k] * (1 - |d| / (neigh + 1)) at round-half-even(k * factor) + d; (4) Y replaces the spectrum's bins 0..n/2.
typedef ms_plock_evt PlockEvt;
#define PLOCK_NTHR 256
#define PLOCK_SEL_MAX 1024               // selected bins kept (pl_top_n is at most 200 in the reference's UI; exact ties may add a few)
MS_DEV int plock_block_sum(int v, int* red, const Ctx& c) {
    red[c.tid] = v;
    c.sync();
    for (int s = c.nthr >> 1; s > 0; s >>= 1) {
        if (c.tid < s) red[c.tid] += red[c.tid + s];
        c.sync();
    }
    const int r = red[0];
    c.sync();
    return r;
}
MS_DEV void partial_lock_body(const PlockEvt* MS_RESTRICT evts, cpx* zbase, real* scratch, const Ctx& c) {
    const PlockEvt& E = evts[c.bx];
    const SpecOp& op = *(const SpecOp*)&E.pre;
    const int n = E.n, bins = n / 2 + 1;
    cpx* Z = zbase + E.z;
    cpx* W = (cpx*)(scratch + E.scratch);
    real* M = (real*)(W + bins);
    int* red = (int*)c.smem;
    for (int k = c.tid; k < bins; k += c.nthr) {
        const cpx w = warp_bin(op, Z, n, k, 0, 0);
        W[k] = w;
        M[k] = (real)hypot((double)w.x, (double)w.y);
    }
    c.sync();
    const int want = E.top_n < bins - 1 ? E.top_n : bins - 1;
    // largest threshold T (as bits of a double) such that count(M[k] >= T, k >= 1) >= want
    unsigned long long lo = 0ull, hi = 0x7ff0000000000000ull;          // count(lo) >= want always; hi = +inf: count = 0
    while (hi - lo > 1ull) {
        const unsigned long long mid = lo + ((hi - lo) >> 1);
        union { unsigned long long u; double d; } cv; cv.u = mid;
        int cnt = 0;
        for (int k = 1 + c.tid; k < bins; k += c.nthr) cnt += ((double)M[k] >= cv.d) ? 1 : 0;
        if (plock_block_sum(cnt, red, c) >= want) lo = mid; else hi = mid;
    }
    union { unsigned long long u; double d; } th; th.u = lo;
    // The selected bins in ascending k, compacted into shared memory (a thread owns a contiguous chunk of bins; an
    // exclusive scan of the chunk counts gives its slot), then a GATHER: every output bin adds the selected bins that
    // land within +-neigh of it, in k order.  No atomics, the result does not depend on the thread schedule.
    int* sel_k2 = red + PLOCK_NTHR + 1;                       // PLOCK_SEL_MAX target bins (round-half-even(k * factor))
    int* sel_k = sel_k2 + PLOCK_SEL_MAX;                      // ... and their source bins
    const int chunk = (bins - 1 + c.nthr - 1) / c.nthr;
    const int k_lo = 1 + c.tid * chunk, k_hi = (k_lo + chunk) < bins ? (k_lo + chunk) : bins;
    int mine = 0;
    if (want > 0) for (int k = k_lo; k < k_hi; ++k) mine += ((double)M[k] >= th.d) ? 1 : 0;
    red[c.tid] = mine;
    c.sync();
    if (c.tid == 0) { int acc = 0; for (int i = 0; i < c.nthr; ++i) { const int v = red[i]; red[i] = acc; acc += v; } red[c.nthr] = acc; }
    c.sync();
    const int n_sel = red[c.nthr] < PLOCK_SEL_MAX ? red[c.nthr] : PLOCK_SEL_MAX;
    {
        int at = red[c.tid];
        if (want > 0) for (int k = k_lo; k < k_hi; ++k) {
            if ((double)M[k] < th.d) continue;
            if (at < PLOCK_SEL_MAX) { sel_k[at] = k; sel_k2[at] = (int)rint((double)k * E.factor); }     // Python round(): half to even
            ++at;
        }
    }
    c.sync();
    const int nb = E.neigh;
    const real inv = (real)1.0 / (real)(nb + 1);
    for (int kk = c.tid; kk < bins; kk += c.nthr) {
        cpx y = c_scale(W[kk], (real)0.12);
        if (kk >= 1) {
            for (int i = 0; i < n_sel; ++i) {
                const int k2 = sel_k2[i];
                int d = kk - k2;
                if (d < 0) d = -d;
                if (d > nb || k2 < 1 || k2 >= bins) continue;
                const real w = (real)1.0 - (real)d * inv;
                const cpx x = W[sel_k[i]];
                y.x += x.x * w; y.y += x.y * w;
            }
        }
        Z[kk] = y;
    }
}

// ---- cepstral warp (cepstral_warp, main_v2.py:150-163): the three elementwise steps between its transforms ---------
// grid = (ceil(max_n / nthr), grains).  step 0: X = low-pass / warp of the grain's spectrum -> scratch, log(|X| + 1e-12)
// -> spectrum of the cepstrum transform;  step 1: cepstrum resampled at t / factor (np.interp, zeros to the right);
// step 2: exp(Re rfft(warped cepstrum)) with the phases of X -> the grain's spectrum.
typedef ms_cep_evt CepEvt;
template <int STEP>
MS_DEV void cepstral_body(const CepEvt* MS_RESTRICT evts, cpx* z1, cpx* z2, const cpx* MS_RESTRICT z3, real* scratch, const Ctx& c) {
    const CepEvt& E = evts[c.by];
    const int n = E.n, bins = n / 2 + 1;
    const int i = c.bx * c.nthr + c.tid;
    if (STEP == 0) {
        if (i >= bins) return;
        const SpecOp& op = *(const SpecOp*)&E.pre;
        const cpx x = warp_bin(op, z1 + E.z1, n, i, 0, 0);
        ((cpx*)(scratch + E.xp))[i] = x;
        z2[E.z2 + i] = mk((real)log(hypot((double)x.x, (double)x.y) + 1e-12), (real)0.);
    } else if (STEP == 1) {
        if (i >= n) return;
        const real* cep = scratch + E.cep;
        const double pos = (double)i / fmax(1e-12, E.factor);
        real v = (real)0.;
        if (pos <= (double)(n - 1)) {
            int i0 = (int)pos;
            if (i0 >= n - 1) v = cep[n - 1];
            else { const real fr = (real)(pos - (double)i0); v = cep[i0] + (cep[i0 + 1] - cep[i0]) * fr; }
        }
        scratch[E.cep2 + i] = v;
    } else {
        if (i >= bins) return;
        const cpx x = ((const cpx*)(scratch + E.xp))[i];
        const double mag = hypot((double)x.x, (double)x.y);
        const double g = exp((double)z3[E.z3 + i].x);
        z1[E.z1 + i] = mag > 0.0 ? mk((real)(g * ((double)x.x / mag)), (real)(g * ((double)x.y / mag))) : mk((real)g, (real)0.);
    }
}

// ---- resonator bank (resonator_bank, main_v2.py:369-384) ------------------------------------------------------------
// One CTA per grain: pass 1 writes the bank (sum of decaying sinusoids, float64 phase) to dst and takes its peak,
// pass 2 overwrites dst with 0.55 x + 0.45 (bank / peak) sign(x).
typedef ms_res_evt ResEvt;
typedef ms_res_mode ResMode;
MS_DEV void resonator_body(const ResEvt* MS_RESTRICT evts, const ResMode* MS_RESTRICT modes, real* pool, const Ctx& c) {
    const ResEvt E = evts[c.bx];
    const real* x = pool + E.src;
    real* y = pool + E.dst;
    const ResMode* Mo = modes + E.mode_begin;
    real* red = (real*)c.smem;
    real mx = (real)0.;
    for (int j = c.tid; j < E.n; j += c.nthr) {
        double acc = 0.0;
        for (int k = 0; k < E.mode_count; ++k) {
            double cyc = (double)j * Mo[k].f_over_sr;
            cyc -= floor(cyc);
            acc += Mo[k].weight * sin(6.283185307179586476925286766559 * cyc + Mo[k].phase);
        }
        const real v = (real)(acc * exp(-(double)j * E.decay));
        y[j] = v;
        mx = r_max(mx, r_abs(v));
    }
    red[c.tid] = mx;
    c.sync();
    for (int s = c.nthr >> 1; s > 0; s >>= 1) { if (c.tid < s) red[c.tid] = r_max(red[c.tid], red[c.tid + s]); c.sync(); }
    const real inv = (real)1.0 / r_max((real)1e-12, red[0]);
    for (int j = c.tid; j < E.n; j += c.nthr) {
        const real xv = x[j];
        const real sg = xv > (real)0. ? (real)1. : (xv < (real)0. ? (real)-1. : (real)0.);
        y[j] = (real)0.55 * xv + (real)0.45 * (y[j] * inv) * sg;
    }
}

// ---- waveguide (waveguide_splinters, main_v2.py:386-402) ---------------------------------------------------------------
// One CTA per grain, lines one after the other.  Within a line v[t] = y[t] + g v[t - d] couples only samples d apart:
// a thread owns a residue r < d and walks t = r, r + d, ... (d is 0.4..8 ms at the design rate, so the chains are short).
typedef ms_wg_evt WgEvt;
typedef ms_wg_line WgLine;
MS_DEV void waveguide_body(const WgEvt* MS_RESTRICT evts, const WgLine* MS_RESTRICT lines, real* pool, const Ctx& c) {
    const WgEvt E = evts[c.bx];
    const real* x = pool + E.src;
    real* y = pool + E.dst;
    const int n = E.n;
    if (E.src != E.dst) {
        for (int j = c.tid; j < n; j += c.nthr) y[j] = x[j];
        c.sync();
    }
    for (int l = 0; l < E.line_count; ++l) {
        const WgLine Ln = lines[E.line_begin + l];
        const int d = Ln.d;
        const real g = (real)Ln.g, mix = (real)Ln.mix, dry = (real)1.0 - (real)Ln.mix;
        const int chains = d < n ? d : n;
        for (int r = c.tid; r < chains; r += c.nthr) {
            real v = (real)0.;
            for (int t = r; t < n; t += d) {
                const real yt = y[t];
                v = yt + g * v;                           // v[t - d] of the same chain (0 before the first sample)
                y[t] = dry * yt + mix * v;
            }
        }
        c.sync();
    }
}

// ---- event feedback (main_v2.py:731-734) and the one-grain step of the spectral imprint that goes with it ----------------
typedef ms_feedback_evt FeedbackEvt;
typedef ms_imprint_step_evt ImprintStepEvt;
MS_DEV void feedback_body(const FeedbackEvt* MS_RESTRICT evts, real* pool, const Ctx& c) {
    const FeedbackEvt E = evts[c.by];
    const int j = c.bx * c.nthr + c.tid;
    if (j >= E.n_cur) return;
    const real cur = pool[E.cur + j];
    const real fb = (real)E.fb;
    pool[E.dst + j] = j < E.n_prev ? ((real)1.0 - fb) * cur + fb * pool[E.prev + j] : cur;
}
// mem: max_bins reals per render slot; prev_bins: spectrum length of the slot's previous imprinted grain (-1: none).
// prev_bins is updated by a second tiny launch (imprint_commit_body) so that every thread of this one sees the old value.
MS_DEV void imprint_step_body(const ImprintStepEvt* MS_RESTRICT evts, cpx* zbase, real* mem, const int* MS_RESTRICT prev_bins,
                              int max_bins, const Ctx& c) {
    const ImprintStepEvt E = evts[c.by];
    const int bins = E.n / 2 + 1;
    const int k = c.bx * c.nthr + c.tid;
    if (k >= bins) return;
    cpx* Z = zbase + E.z;
    real* m = mem + (long long)E.slot * max_bins;
    const cpx X = Z[k];
    const real mag = (real)hypot((double)X.x, (double)X.y);
    const real amount = (real)E.amount, smooth = (real)E.smooth;
    const real mm = (prev_bins[E.slot] != bins) ? mag : smooth * m[k] + ((real)1.0 - smooth) * mag;
    m[k] = mm;
    const real mag2 = ((real)1.0 - amount) * mag + amount * mm;
    Z[k] = mag > (real)0. ? c_scale(X, mag2 / mag) : mk(mag2, (real)0.);
}
MS_DEV void imprint_commit_body(const ImprintStepEvt* MS_RESTRICT evts, int n_evts, int* prev_bins, const Ctx& c) {
    for (int e = c.bx * c.nthr + c.tid; e < n_evts; e += c.nthr * 64) prev_bins[evts[e].slot] = evts[e].n / 2 + 1;
}

// ---- EXTENSION (no reference counterpart; SURVEY a14): band-limited polyphase decimation ---------------------------------
// Nothing in render() decimates -- the rate change is a relabel (main_v2.py:489-490) and the band-limit is lowpass_fft
// (main_v2.py:39-59) -- so this stage is OFF the parity path; it exists because north_star names it, and is checked
// against scipy.signal.upfirdn / resample_poly in float64 ("parity unpinned by the reference").
//   y[m] = sum_k h[k] x[m q - k]   (upfirdn(h, x, up = 1, down = q): zero-extended input, m < ceil((n + taps - 1) / q))
// i.e. only the q-th outputs of the FIR are ever formed (the polyphase identity), never the full-rate signal.
// grid = (ceil(n_out / DEC_OUT), signals), DEC_NTHR threads.  The taps and the tile's input window live in shared
// memory; a warp forms one output at a time: its lanes stride over the taps (conflict-free: consecutive lanes read
// consecutive taps and consecutive input samples) and the 32 partial sums are reduced with warp shuffles.
#define DEC_NTHR 256
#define DEC_OUT 256                  // outputs per CTA
#define DEC_TAPS_MAX 4096
MS_DEV real warp_sum(real v, real* scratch, const Ctx& c) {
#ifdef MS_HOST_EMUL
    scratch[c.tid] = v;
    c.syncwarp();
    real s = (real)0.;
    const int w0 = c.tid & ~31;
    for (int i = 0; i < 32; ++i) s += scratch[w0 + (i ^ 0)];      // same value in every lane, like the xor butterfly
    c.syncwarp();
    return s;
#else
    (void)scratch; (void)c;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
#endif
}
MS_DEV void decimate_body(const real* MS_RESTRICT x, long long x_stride, int n, const real* MS_RESTRICT h, int taps, int q,
                          real* MS_RESTRICT y, long long y_stride, int n_out, const Ctx& c) {
    real* sh = (real*)c.smem;                        // taps
    real* sx = sh + taps;                            // window: (DEC_OUT - 1) q + taps samples, oldest first
    real* scratch = sx + (DEC_OUT - 1) * q + taps;   // emulator only
    const real* xs = x + (long long)c.by * x_stride;
    real* ys = y + (long long)c.by * y_stride;
    const int m0 = c.bx * DEC_OUT;
    if (m0 >= n_out) return;
    const int mcnt = (n_out - m0) < DEC_OUT ? (n_out - m0) : DEC_OUT;
    const long long first = (long long)m0 * q - (taps - 1);              // input index of window slot 0
    const int wlen = (mcnt - 1) * q + taps;
    for (int i = c.tid; i < taps; i += c.nthr) sh[i] = __ldg(&h[i]);
    for (int i = c.tid; i < wlen; i += c.nthr) {
        const long long j = first + i;
        sx[i] = (j >= 0 && j < n) ? __ldg(&xs[j]) : (real)0.;
    }
    c.sync();
    const int lane = c.tid & 31, warp = c.tid >> 5, nwarps = c.nthr >> 5;
    for (int mm = warp; mm < mcnt; mm += nwarps) {
        // x[m q - k] sits at window slot (m - m0) q + taps - 1 - k
        const real* w = sx + mm * q + taps - 1;
        real acc = (real)0.;
        for (int k = lane; k < taps; k += 32) acc += sh[k] * w[-k];
        acc = warp_sum(acc, scratch, c);
        if (lane == 0) ys[m0 + mm] = acc;
    }
}
