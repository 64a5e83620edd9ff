"""Kernel-level checks shared by the CPU (block emulator) and GPU test files: the same assertions run
against the same C ABI; only the device differs."""
import ctypes as C

import numpy as np

from audio_suite_b200 import _abi, configs, engine, plan
from oracle import microsound_np as O


def _api(dev, precision):
    return _abi.Api(dev.lib, precision)


def _real(precision):
    return np.float32 if precision == "f32" else np.float64


def _to_host(dev, buf, n, dtype):
    out = dev.download(buf, 0, n)
    return np.asarray(out).view(dtype) if np.asarray(out).dtype != dtype else np.asarray(out)


def fft_pair(dev, precision, a, b):
    api, real = _api(dev, precision), _real(precision)
    n = len(a)
    need = api.ms_fft_pair_workspace_bytes(n)
    assert need > 0, dev.lib.ms_last_error()
    ws = dev.empty(need, np.uint8)
    da, db = dev.upload(np.asarray(a, real)), dev.upload(np.asarray(b, real))
    z = dev.empty(2 * n, real)
    rc = api.ms_fft_pair_forward(dev.ptr(da), dev.ptr(db), n, dev.ptr(z), dev.ptr(ws), need, dev.stream_ptr())
    assert rc == 0, dev.lib.ms_last_error()
    dev.synchronize()
    zz = np.asarray(dev.download(z, 0, 2 * n), dtype=np.float64)
    return zz[0::2] + 1j * zz[1::2]


def check_fft_lengths(dev, precision, lengths, tol):
    rng = np.random.default_rng(0)
    real = _real(precision)
    for n in lengths:
        a, b = rng.standard_normal(n).astype(real), rng.standard_normal(n).astype(real)
        got = fft_pair(dev, precision, a, b)
        want = np.fft.fft(a.astype(np.float64) + 1j * b.astype(np.float64))
        err = np.max(np.abs(got - want)) / np.max(np.abs(want))
        assert err < tol, (n, err)


def spectral_apply(dev, precision, jobs, src, dst_len):
    api, real = _api(dev, precision), _real(precision)
    arr = (_abi.SpecJob * len(jobs))(*jobs)
    need = api.ms_spectral_workspace_bytes(C.addressof(arr), len(jobs))
    assert need > 0, dev.lib.ms_last_error()
    ws = dev.empty(need, np.uint8)
    dsrc = dev.upload(np.asarray(src, real))
    dst = dev.zeros(dst_len, real)
    rc = api.ms_spectral_apply(C.addressof(arr), len(jobs), dev.ptr(dsrc), dev.ptr(dst), dev.ptr(ws), need, dev.stream_ptr())
    assert rc == 0, dev.lib.ms_last_error()
    dev.synchronize()
    return np.asarray(dev.download(dst, 0, dst_len), dtype=np.float64)


def _ref_grain(x, sr, p):
    g = x
    if p["bandlimit_on"]:
        g = O.fft_lowpass(g, sr, p["cut"], roll=p["bandlimit_roll_hz"])
    g = O.spectrum_stretch(g, p["st"])
    if p["unfold_mode"] != "Classic reinterpret":
        b1, b2, b3 = p["mb_b1"], p["mb_b2"], p["mb_b3"]
        g = O.multiband_unfold(g, sr, [(0, b1), (b1, b2), (b2, b3)], [p["mb_u1"], p["mb_u2"], p["mb_u3"]], p["mb_roll"])
    return g


def check_spectral_ops(dev, precision, tol, big=True):
    """Pairs of signals with *different* operators in one complex transform, against the oracle."""
    rng = np.random.default_rng(5)
    real = _real(precision)
    base = configs.with_defaults()

    def Pm(**kw):
        p = dict(base)
        p.update(kw)
        return p
    cases = [
        (7680, 768000, Pm(cut=18000 * 16, st=1.0), Pm(cut=18000 * 16, st=2.5)),
        (3301, 48000 * 30, Pm(cut=18000 * 30., st=1.3, unfold_mode="Multi-band unfold"),
         Pm(cut=9000 * 30., st=1.0, unfold_mode="Multi-band unfold", mb_roll=0.0)),
        (1690, 48000 * 30, Pm(cut=18000 * 30., st=0.3), Pm(cut=1e9, st=1.0)),
        (4001, 48000 * 30, Pm(cut=18000 * 30., st=2.0), Pm(cut=1e9, st=0.9)),
        (999, 48000 * 30, Pm(cut=18000 * 30., st=4.0, bandlimit_roll_hz=0.0), Pm(cut=5e5, st=0.25)),
    ]
    if big:
        cases += [
            (48000, 4800000, Pm(cut=1.8e6, st=4.0), Pm(cut=0.9e6, st=0.5, bandlimit_roll_hz=0.0)),
            (12480, 48000 * 26, Pm(cut=18000 * 26, st=3.36), Pm(cut=18000 * 26, st=0.77, bandlimit_on=False)),
            (30000, 3000000, Pm(cut=1e6, st=2.5), Pm(cut=1e6, st=2.5)),
        ]
    for n, sr, pa, pb in cases:
        a = rng.standard_normal(n).astype(real).astype(np.float64)
        b = rng.standard_normal(n).astype(real).astype(np.float64)
        j = _abi.SpecJob()
        j.n, j.in_a, j.in_b, j.out_a, j.out_b = n, 0, n, 0, n
        oa = plan.grain_spec_op(pa, sr, n, pa["cut"], pa["st"])
        ob = plan.grain_spec_op(pb, sr, n, pb["cut"], pb["st"])
        j.op[0] = oa if oa is not None else _abi.SpecOp()
        j.op[1] = ob if ob is not None else _abi.SpecOp()
        out = spectral_apply(dev, precision, [j], np.concatenate([a, b]), 2 * n)
        ra, rb = _ref_grain(a, sr, pa), _ref_grain(b, sr, pb)
        sc = max(np.max(np.abs(ra)), np.max(np.abs(rb)))
        assert np.max(np.abs(out[:n] - ra)) / sc < tol, (n, "a")
        assert np.max(np.abs(out[n:] - rb)) / sc < tol, (n, "b")
        j2 = _abi.SpecJob()
        j2.n, j2.in_a, j2.in_b, j2.out_a, j2.out_b = n, 0, -1, 0, -1
        j2.op[0] = j.op[0]
        out2 = spectral_apply(dev, precision, [j2], a, n)
        assert np.max(np.abs(out2 - ra)) / sc < tol, (n, "single")


def check_identity_ops(dev, precision, tol):
    """OP_NONE round trip is the identity for direct, two-pass and Bluestein lengths."""
    rng = np.random.default_rng(9)
    real = _real(precision)
    jobs, src, off = [], [], 0
    for n in (16, 17, 480, 625, 1000, 4099, 9000, 12345):
        a, b = rng.standard_normal(n).astype(real), rng.standard_normal(n).astype(real)
        j = _abi.SpecJob()
        j.n, j.in_a, j.in_b, j.out_a, j.out_b = n, off, off + n, off, off + n
        jobs.append(j)
        src += [a, b]
        off += 2 * n
    src = np.concatenate(src)
    out = spectral_apply(dev, precision, jobs, src, off)
    assert np.max(np.abs(out - src.astype(np.float64))) < tol * 10


def synth_plain(dev, precision, seed, n):
    """Raw normals * 0.1 with fades (gen_basic's fallback branch, main_v2.py:263-269)."""
    p = configs.with_defaults(gen_mode="Noise burst")     # planner needs a valid mode; we override below
    rp = plan.plan_render(p)
    api, real = _api(dev, precision), _real(precision)
    rec = np.zeros(1, dtype=np.dtype(_abi.SynthEvt))
    st = np.random.PCG64(seed).state["state"]
    rec[0]["s_hi"], rec[0]["s_lo"] = st["state"] >> 64, st["state"] & 0xFFFFFFFFFFFFFFFF
    rec[0]["i_hi"], rec[0]["i_lo"] = st["inc"] >> 64, st["inc"] & 0xFFFFFFFFFFFFFFFF
    rec[0]["n"], rec[0]["mode"] = n, plan.MODE_NOISE     # NOISE writes the raw normals
    rec[0]["fade"], rec[0]["inv_fade"], rec[0]["sigma"] = 8, 1.0 / 8, 1
    d = dev.upload(rec)
    pool = dev.zeros(n, real)
    rc = api.ms_synth_normal(dev.ptr(d), 1, dev.ptr(pool), dev.stream_ptr())
    assert rc == 0, dev.lib.ms_last_error()
    dev.synchronize()
    return np.asarray(dev.download(pool, 0, n))


def check_normals_bit_exact(dev, precision, cases):
    real = _real(precision)
    for seed, n in cases:
        got = synth_plain(dev, precision, seed, n)
        want = np.random.default_rng(seed).standard_normal(n).astype(real)
        assert got.dtype == want.dtype
        if precision == "f32":
            assert np.array_equal(got, want), (seed, n, int(np.argmax(got != want)))
        else:
            # identical stream positions everywhere; the ~3e-4 of draws that come from the ziggurat tail
            # go through log1p, where the device libm and glibc may differ in the last bit
            diff = got != want
            assert diff.mean() < 1e-3 and np.max(np.abs(got - want)) < 1e-14, (seed, n, int(diff.sum()))


def render_error(dev, params, precision, taps=None):
    ref, mref = O.render(params, taps=taps)
    out, meta = engine.render(params, device=dev, precision=precision)
    assert out.dtype == np.float64 and out.shape == ref.shape
    assert meta["out_sr"] == mref["out_sr"] and meta["design_sr_base"] == mref["design_sr_base"]
    err = float(np.max(np.abs(out - ref)))
    rms_db = 20 * np.log10(max(1e-30, float(np.sqrt(np.mean((out - ref) ** 2)))))
    gm = np.max(np.abs(meta["grain_last"] - mref["grain_last"])) / max(1e-30, np.max(np.abs(mref["grain_last"])))
    mm = np.max(np.abs(meta["micro_last"] - mref["micro_last"])) / max(1e-30, np.max(np.abs(mref["micro_last"])))
    return err, rms_db, float(gm), float(mm)


# tolerance north_star states: 1e-5 max-abs and -100 dBFS RMS residual against the numpy path
MAX_ABS_TOL = 1e-5
RMS_DB_TOL = -100.0


def reference_noise_floor(params, taps):
    """The reference's own float64 rounding, where it is visible: spectral_diffusion_stereo (main_v2.py:432-435)
    runs a full-length rfft/irfft over the pre-clip signal, which leaves ~eps * peak of noise in samples
    whose exact value is 0 (silence after the last grain), and tanh has unit slope there.  With a
    +12 dB/oct noise tilt the pre-clip peak reaches 1e11, i.e. 2e-5 of reference noise.  Our right
    channel is an exact time-domain identity (Bessel taps), so that noise shows up as a difference."""
    if not params["stereo_on"] or params["sat_drive"] <= 0:
        return 0.0
    return 8.0 * np.finfo(np.float64).eps * float(np.max(np.abs(taps["after_ir"]))) * float(params["sat_drive"])


VACUOUS = 0.05          # 4 x floor above this: the end-to-end tolerance cannot fail on a +-0.98 output


def check_render(dev, params, precision="auto", floor=None):
    taps = {}
    err, rms_db, gm, mm = render_error(dev, params, precision, taps)
    # cepstral warp / spectral imprint / resonator sign keep the phase of bins that hold only rounding noise: that share
    # of the reference's own output is not reproducible by any other FFT (oracle.rounding_noise_floor measures it by a
    # 1e-15 jitter).  Where that makes the end-to-end tolerance vacuous the stages themselves are verified on the
    # device's own input (check_stages) -- no silent pass.
    floor = O.rounding_noise_floor(params) if floor is None else floor
    assert err < MAX_ABS_TOL + reference_noise_floor(params, taps) + 4.0 * floor, (err, floor)
    assert rms_db < RMS_DB_TOL or floor > 1e-6, rms_db
    assert (gm < 2e-6 or floor > 1e-6) and mm < 2e-6, (gm, mm)
    if floor > 1e-6:
        staged = check_stages(dev, params)
        print("rounding-noise floor %.3e (4 x floor %s the vacuous bound %.2f): stage-level checks %s" % (
            floor, ">" if 4.0 * floor > VACUOUS else "<=", VACUOUS, staged))
        assert staged, "ill-conditioned render with no stage-level coverage"
    return err


def preset_like(name):
    """Parameter sets shaped like the shipped presets that need only accelerated rows (values copied from
    microsound_0.2.1/presets/<name>.json; the files themselves stay in the reference)."""
    p = configs.with_defaults(PRESET_LIKE[name])
    if isinstance(p.get("_ir_audio"), str):            # what on_load_ir hands over: mono, peak 0.9 (main_v2.py:1401-1413)
        ir = configs.synth_ir(0.25, 48000, 11, channels=1)
        p["_ir_audio"] = ir * (0.9 / np.max(np.abs(ir)))
    if isinstance(p.get("_img_gray"), str):
        p["_img_gray"] = np.random.default_rng(5).integers(0, 256, (40, 300)).astype(np.uint8)
    return p


PRESET_LIKE = {
    "opal_airfold": dict(gen_mode="Wavelet atoms", micro_ms=1.6, wav_base_hz=1800, wav_count=10, wav_spread=0.9,
                         unfold_mode="Multi-band unfold", mb_u1=60, mb_u2=32, mb_u3=16, event_process="Poisson",
                         grains_per_sec=10, stereo_on=True, stereo_width=0.85, er_cloud_on=True, er_taps=300, er_max_ms=48),
    "opal_oval_breath": dict(gen_mode="Wavelet atoms", micro_ms=2.6, wav_base_hz=900, wav_count=5, wav_spread=0.3,
                             event_process="Poisson", grains_per_sec=6, bp_density="0:4, 8:9, 16:4", partial_stretch=1.08,
                             er_cloud_on=True, er_taps=300, er_max_ms=52, stereo_width=0.85),
    "basinski_melodic_loop": dict(gen_mode="Gaussian click", micro_ms=3.6, event_process="Poisson", grains_per_sec=4,
                                  spectral_imprint_on=True, spectral_imprint_amt=0.35, spectral_imprint_smooth=0.99,
                                  partial_stretch=0.9, er_cloud_on=False, stereo_width=0.5),
    "micro_carillon": dict(gen_mode="Wavelet atoms", micro_ms=1.1, wav_base_hz=660, wav_count=6, wav_spread=0.15,
                           event_process="Clustered", grains_per_sec=18, cluster_size=3, cluster_spread_ms=10,
                           partial_lock_on=True, er_cloud_on=True, er_taps=200, er_max_ms=32),      # lock at factor 1: identity
    "oval_glass_orbit": dict(gen_mode="Wavelet atoms", micro_ms=1.9, wav_base_hz=1400, wav_count=6, wav_spread=0.4,
                             partial_lock_on=True, partial_stretch=1.05, event_process="Poisson", grains_per_sec=7,
                             bp_unfold="0:28, 6:34, 14:30", bp_density="0:6, 10:9, 18:6", er_cloud_on=True, er_taps=260,
                             er_max_ms=48, stereo_width=0.7),
    "01_corona_glass_fog": dict(stereo_width=0.7, gen_mode="Crackle / corona", micro_ms=1.0, seed=14001, crackle_alpha=1.35,
                                crackle_density=260.0, crackle_kernel=72, unfold_mode="Multi-band unfold", nl_warp_on=True,
                                nl_warp_power=1.35, mb_u1=40.0, mb_u2=22.0, mb_u3=12.0, mb_roll=2500.0, event_process="Hawkes",
                                hawkes_gain=0.8, hawkes_decay_s=0.22, bp_density="0:12, 3:24, 8:14", bp_unfold="0:18, 4:35, 8:20",
                                spectral_imprint_on=True, spectral_imprint_amt=0.32, spectral_imprint_smooth=0.93,
                                er_cloud_on=True, er_taps=420, er_max_ms=55.0),
    "corona_memory_glass": dict(gen_mode="Crackle / corona", micro_ms=0.7, crackle_alpha=1.35, crackle_density=260,
                                crackle_kernel=48, event_process="Hawkes", grains_per_sec=16, hawkes_gain=0.85,
                                hawkes_decay_s=0.18, unfold_mode="Multi-band unfold", mb_u1=48, mb_u2=26, mb_u3=14,
                                partial_lock_on=True, partial_stretch=1.12, spectral_imprint_on=True,
                                spectral_imprint_amt=0.42, spectral_imprint_smooth=0.94, er_cloud_on=True, er_taps=420, er_max_ms=55),
    "melodic_dust_chime": dict(gen_mode="Crackle / corona", micro_ms=0.9, crackle_alpha=1.25, crackle_density=120,
                               partial_lock_on=True, partial_stretch=0.98, event_process="Clustered", grains_per_sec=14,
                               cluster_size=4, cluster_spread_ms=16, er_cloud_on=False),
    "glass_harmonic_arc": dict(gen_mode="Wavelet atoms", micro_ms=1.4, wav_base_hz=330, wav_count=8, wav_spread=0.25,
                               partial_lock_on=True, partial_stretch=1.0, event_process="Poisson", grains_per_sec=9,
                               spectral_imprint_on=True, spectral_imprint_amt=0.18, er_cloud_on=True, er_taps=240, er_max_ms=45),
    "oval_room_trace": dict(gen_mode="IR fragment", micro_ms=2.0, event_process="Poisson", grains_per_sec=6,
                            spectral_imprint_on=True, spectral_imprint_amt=0.28, space_ir_on=True, space_ir_max_samps=11000,
                            er_cloud_on=False, _ir_audio="synthetic mono 250 ms"),
    "image_grain_hallucination": dict(gen_mode="Image scanline", micro_ms=0.8, partial_stretch=1.35, event_process="Clustered",
                                      grains_per_sec=26, cluster_size=10, cluster_spread_ms=12, nl_warp_on=True,
                                      nl_warp_power=1.9, er_cloud_on=True, er_taps=220, er_max_ms=35,
                                      _img_gray="synthetic 40 x 300"),
    "closed_curve_air": dict(gen_mode="Noise burst", micro_ms=1.8, noise_tilt=-9.0, cep_warp_on=True, cep_factor=1.25,
                             event_process="Poisson", grains_per_sec=7, partial_stretch=0.98, er_cloud_on=True, er_taps=190,
                             er_max_ms=44),
    "ghost_formants": dict(gen_mode="Noise burst", micro_ms=1.1, noise_tilt=-6.0, cep_warp_on=True, cep_factor=1.45,
                           partial_stretch=0.92, event_process="Poisson", grains_per_sec=12, bp_cutoff="0:16000, 6:9000, 12:6000",
                           er_cloud_on=True, er_taps=260, er_max_ms=42),
    "chaotic_dustfield": dict(gen_mode="Micro-chaos", micro_ms=0.9, chaos_r=3.97, chaos_gate=0.42, event_process="Poisson",
                              grains_per_sec=9, bp_density="0:6, 3:14, 5:28, 9:10", nl_warp_on=True, nl_warp_power=1.6,
                              bandlimit_out_hz=14000, er_taps=180, er_max_ms=38),
    "elliptical_insect_hum": dict(gen_mode="Micro-chaos", micro_ms=1.4, chaos_r=3.91, chaos_gate=0.22,
                                  unfold_mode="Multi-band unfold", mb_u1=34, mb_u2=22, mb_u3=14, event_process="Poisson",
                                  grains_per_sec=8, nl_warp_on=True, nl_warp_power=1.2, er_taps=210, er_max_ms=36),
    "infra_mechanical_choir": dict(gen_mode="Resonant strike", micro_ms=3.5, ring_hz=420, ring_decay_ms=90, res_bank_on=True,
                                   res_modes=36, res_fmin=90, res_fmax=4200, res_decay_ms=160, partial_lock_on=True,
                                   partial_stretch=0.88, event_process="Clustered", grains_per_sec=8, cluster_spread_ms=40,
                                   bp_unfold="0:18, 6:40, 14:22"),
    "infra_tone_lattice": dict(gen_mode="Resonant strike", micro_ms=2.8, ring_hz=180, ring_decay_ms=120, res_bank_on=True,
                               res_fmin=90, res_fmax=1800, res_decay_ms=220, partial_lock_on=True, partial_stretch=1.02,
                               event_process="Poisson", grains_per_sec=6, spectral_imprint_on=True, spectral_imprint_amt=0.22,
                               er_taps=300, er_max_ms=60),
    "friction_lattice": dict(gen_mode="Stick–slip friction", micro_ms=2.4, ss_threshold=0.85, ss_build=0.08, ss_decay=0.72,
                             ss_noise=0.06, wg_on=True, wg_lines=14, wg_max_ms=6.5, wg_fb=0.78, partial_stretch=1.18,
                             partial_lock_on=True, event_process="Clustered", grains_per_sec=22, cluster_size=8,
                             cluster_spread_ms=18, er_cloud_on=False, stereo_width=0.35),
    "orbital_friction_loop": dict(gen_mode="Stick–slip friction", micro_ms=3.2, ss_threshold=0.55, ss_build=0.035, ss_decay=0.88,
                                  ss_noise=0.04, wg_on=True, wg_lines=6, wg_max_ms=5.5, wg_fb=0.6, event_process="Poisson",
                                  grains_per_sec=5, partial_stretch=1.03, er_cloud_on=False),
    "wavelet_mist": dict(out_dur_s=12.0, time_unfold=30.0, sat_drive=1.05, stereo_width=0.75, gen_mode="Wavelet atoms", micro_ms=1.6,
                         seed=33009, noise_tilt=-5.0, wav_base_hz=1700.0, wav_count=14, wav_spread=1.1,
                         unfold_mode="Multi-band unfold", partial_stretch=0.92, nl_warp_on=True, nl_warp_power=1.35,
                         cep_warp_on=True, cep_factor=1.35, mb_b1=1800.0, mb_b2=7000.0, mb_u1=55.0, mb_u2=28.0, mb_u3=10.0,
                         mb_roll=2500.0, bandlimit_out_hz=17500.0, bandlimit_roll_hz=3200.0, event_process="Poisson",
                         grains_per_sec=14.0, max_grains=5500, grain_amp_rand=0.25, grain_offset_max_ms=120.0,
                         bp_density="0:10, 5:18, 12:12", bp_unfold="0:45, 6:22, 12:35", bp_cutoff="0:16000, 7:11000, 12:17500",
                         bp_stretch="0:0.85, 12:0.95", res_bank_on=True, res_modes=30, res_fmin=90.0, res_fmax=9000.0,
                         res_decay_ms=110.0, event_feedback_on=True, event_feedback_amt=0.22, spectral_imprint_on=True,
                         spectral_imprint_amt=0.25, spectral_imprint_smooth=0.94, er_taps=520, er_max_ms=60.0,
                         space_ir_on=True, space_ir_max_samps=16000, env_a=80.0, env_d=450.0, env_s=0.7, env_r=3800.0,
                         env_curve=1.6),
    "soft_ellipse_memory": dict(gen_mode="Noise burst", micro_ms=2.2, noise_tilt=-8.0, event_process="Poisson",
                                grains_per_sec=6, spectral_imprint_on=True, spectral_imprint_amt=0.25,
                                spectral_imprint_smooth=0.97, partial_stretch=0.95, bp_cutoff="0:14000, 12:9000, 24:6000",
                                er_cloud_on=True, er_taps=180, er_max_ms=40),
}




# ---- stage-level parity where the reference's own output is decided by rounding noise -------------------------------------
# cepstral_warp (main_v2.py:150-163) and SpectralImprint (565-581) keep the PHASE of every bin and give it a new
# magnitude; resonator_bank (369-384) multiplies by sign(x).  After a band-limit (every shipped cepstral preset has one)
# the emptied bins hold ~1e-16 of rounding noise whose phase / sign no other FFT reproduces, so a time-domain comparison
# of the whole render cannot fail there (oracle.rounding_noise_floor up to 1.9 on a +-0.98 output).  What IS determined
# is each stage as a function of ITS input: these checks read the device buffers around the stage (engine.run's probe
# hook), hand the oracle the SAME input and compare magnitudes in every bin and phases where the input is above 1e-9 of
# its peak, at 1e-9.
STAGE_TOL = 1e-9


def _ws_complex(dev, stage, zbase, z_off, n):
    raw = np.asarray(dev.download(stage.ws, int(zbase) + 16 * int(z_off), 16 * int(n)))
    return raw.view(np.complex128).copy()


def _phase_close(y, x, tol):
    big = np.abs(x) > 1e-9 * max(1e-300, float(np.max(np.abs(x))))
    if not np.any(big):
        return 0.0
    ok = big & (np.abs(y) > 0)
    return float(np.max(np.abs(y[ok] / np.abs(y[ok]) - x[ok] / np.abs(x[ok])))) if np.any(ok) else 0.0


def check_stages(dev, params):
    """Runs one render (float64) with probes around the ill-conditioned stages and checks each against the oracle on
    the device's own input.  Returns the names of the stages it verified."""
    br = engine.BatchRenderer([params], device=dev, precision="f64")
    rp = br.plans[0]
    seen, hold = [], {}

    def spectra(stage, zbase, evs, zname="z"):
        return [_ws_complex(dev, stage, zbase, e[zname], e["n"]) for e in evs]

    def probe(name, item=None):
        dev.synchronize()
        if name == "cep_x":
            ev = br.h_cep_evt
            scr = np.asarray(dev.download(br.cep_scratch, 0, br.cep_scratch.shape[0] if hasattr(br.cep_scratch, "shape") else len(br.cep_scratch)))
            hold["cep_x"] = [scr[int(e["xp"]):int(e["xp"]) + 2 * (int(e["n"]) // 2 + 1)].view(np.complex128).copy() for e in ev]
        elif name == "cep_y":
            ev = br.h_cep_evt
            ys = spectra(br.cep_stages[0], br.cep_zb[0], ev, "z1")
            for e, x, y in zip(ev, hold["cep_x"], ys):
                n = int(e["n"]); bins = n // 2 + 1
                want = O.cepstrum_warp_magnitudes(x, n, float(e["factor"]))
                got = np.abs(y[:bins])
                assert np.max(np.abs(got - want) / want) < STAGE_TOL, ("cepstral magnitudes", n, float(np.max(np.abs(got - want) / want)))
                assert _phase_close(y[:bins], x, STAGE_TOL) < STAGE_TOL, ("cepstral phases", n)
            seen.append("cepstral_warp[%d]" % len(ev))
        elif name == "imprint_x":
            hold["imp_x"] = spectra(br.imprint_stage, br.imprint_zbase, br.h_imp_evt)
        elif name == "imprint_y":
            ys = spectra(br.imprint_stage, br.imprint_zbase, br.h_imp_evt)
            for r in br.h_imp_render:
                mem = O.ImprintMemory()
                for k in range(int(r["ev_begin"]), int(r["ev_end"])):
                    n = int(br.h_imp_evt[k]["n"]); bins = n // 2 + 1
                    x, y = hold["imp_x"][k][:bins], ys[k][:bins]
                    want = mem.blend(np.abs(x), float(r["amount"]), float(r["smooth"]))
                    sc = max(1e-300, float(np.max(want)))
                    assert np.max(np.abs(np.abs(y) - want)) / sc < STAGE_TOL, ("imprint magnitudes", k)
                    assert _phase_close(y, x, STAGE_TOL) < STAGE_TOL, ("imprint phases", k)
            seen.append("spectral_imprint[%d]" % len(ys))
        elif name == "seq_imprint_x":
            hold["seq_x"] = spectra(item["stage"], item["zbase"], item["h_imp"])
        elif name == "seq_imprint_y":
            ys = spectra(item["stage"], item["zbase"], item["h_imp"])
            mems = hold.setdefault("seq_mem", {})
            for e, x, y in zip(item["h_imp"], hold["seq_x"], ys):
                n = int(e["n"]); bins = n // 2 + 1
                mem = mems.setdefault(int(e["slot"]), O.ImprintMemory())
                want = mem.blend(np.abs(x[:bins]), float(e["amount"]), float(e["smooth"]))
                sc = max(1e-300, float(np.max(want)))
                assert np.max(np.abs(np.abs(y[:bins]) - want)) / sc < STAGE_TOL, ("imprint step magnitudes", n)
                assert _phase_close(y[:bins], x[:bins], STAGE_TOL) < STAGE_TOL, ("imprint step phases", n)
            seen.append("imprint_step")
        elif name == "res_x":
            hold["res_x"] = [np.asarray(dev.download(br.pool, int(e["src"]), int(e["n"]))).astype(np.float64) for e in br.h_res_evt]
        elif name == "res_y":
            evs = [ev for ev in rp.events if ev.res is not None]
            assert len(evs) == len(br.h_res_evt)
            for e, pe, x in zip(br.h_res_evt, evs, hold["res_x"]):
                y = np.asarray(dev.download(br.pool, int(e["dst"]), int(e["n"]))).astype(np.float64)
                want = O.resonator_bank(x, pe.gen_sr, int(params["res_modes"]), float(params["res_fmin"]), float(params["res_fmax"]),
                                        float(params["res_decay_ms"]), pe.seed)
                sc = max(1e-300, float(np.max(np.abs(want))))
                assert np.max(np.abs(y - want)) / sc < STAGE_TOL, ("resonator bank", int(e["n"]), float(np.max(np.abs(y - want)) / sc))
            seen.append("resonator_bank[%d]" % len(evs))
    br.run(probe=probe)
    dev.synchronize()
    br.close()
    return seen


# ---- the 27 shipped presets, from the fixture the unmodified reference wrote (oracle/make_golden_presets.py) ----------------
def preset_fixture():
    """{name: (params, audio[::step] float32, step, rounding-noise floor, [(pct, msg), ...])} for every shipped preset:
    parameters exactly as on_load_preset merges them (main_v2.py:1286-1291), 2 s renders of the reference."""
    import json
    import os
    from conftest import GOLDEN
    g = np.load(os.path.join(GOLDEN, "presets.npz"))
    out = {}
    for name in json.loads(str(g["names"])):
        p = json.loads(str(g["params_" + name]))
        p["_ir_audio"], p["_img_gray"] = None, None
        ir = str(g["ir_of_" + name])
        if ir:
            p["_ir_audio"] = np.array(g["ir_" + ir])
        if p["gen_mode"] == "Image scanline":
            p["_img_gray"] = np.array(g["img_gray"])
        out[name] = (p, np.array(g["audio_" + name]), int(g["step"]), float(g["floor_" + name]),
                     [tuple(x) for x in json.loads(str(g["progress_" + name]))])
    return out


def shipped_irs(directory):
    """The shipped impulse responses the preset fixture carries -- each as the array the reference's on_load_ir rule made
    of it (main_v2.py:1401-1413: int16 / 32768, mean over channels, normalised to 0.9) -- written back to `directory` as
    16-bit mono WAV files that this rule maps to exactly that array: the samples are a * peak / 0.9 for the one int16
    peak that makes every sample an integer.  Returns {path: array}."""
    import os
    import wave
    from conftest import GOLDEN
    g = np.load(os.path.join(GOLDEN, "presets.npz"))
    out = {}
    for key in sorted(k for k in g.files if k.startswith("ir_") and not k.startswith("ir_of_")):
        a = np.array(g[key])
        peak = next(q for q in range(1, 32768) if np.max(np.abs(a / 0.9 * q - np.round(a / 0.9 * q))) < 1e-6)
        path = os.path.join(str(directory), key[3:])
        with wave.open(path, "wb") as w:
            w.setnchannels(1)
            w.setsampwidth(2)
            w.setframerate(48000)
            w.writeframes(np.round(a / 0.9 * peak).astype("<i2").tobytes())
        out[path] = a
    assert out
    return out


def check_preset(dev, name, fixture=None):
    """One shipped preset through render(): audio against the reference's, progress messages identical, and -- where
    the reference's own output is decided by rounding noise -- the stage-level checks on the device's own input."""
    p, want, step, floor, msgs = (fixture or preset_fixture())[name]
    seen = []
    out, meta = engine.render(p, progress=lambda pct, msg: seen.append((int(pct), str(msg))), device=dev)
    assert seen == msgs, (name, seen[:3], msgs[:3])
    assert out.shape[0] == int(round(p["out_dur_s"] * p["base_sr"])) and meta["out_sr"] == int(p["base_sr"])
    err = float(np.max(np.abs(out[::step] - want.astype(np.float64))))
    assert err < MAX_ABS_TOL + 1e-7 + 4.0 * floor, (name, err, floor)          # 1e-7: the fixture stores float32
    staged = []
    if floor > 1e-6:
        staged = check_stages(dev, p)
        assert staged, name
    print("preset %-28s max-abs %.2e  floor %.2e  stage checks %s" % (name, err, floor, staged or "-"))
    return err
