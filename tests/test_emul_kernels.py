"""CPU tests of the *kernel bodies* through the block emulator (tests/host_emul): same C ABI, same
engine, CUDA threads emulated by fibres.  Sizes are kept small; the GPU tests repeat these at full size."""
import numpy as np
import pytest

import kernel_checks as K
from audio_suite_b200 import configs
from oracle import microsound_np as O


@pytest.mark.parametrize("precision,tol", [("f32", 2e-6), ("f64", 1e-13)])
def test_fft_direct_twopass_bluestein(emul, precision, tol):
    K.check_fft_lengths(emul, precision, [16, 60, 125, 243, 480, 1000, 7680, 8192, 17, 97, 1690, 3301, 4097,
                                           9000, 12480, 20011, 51900, 83040, 15360, 19200], tol)   # 51900 = 173 * 300, 83040 = 173 * 480: in-tile Bluestein of 512


@pytest.mark.parametrize("precision,tol", [("f32", 3e-6), ("f64", 1e-12)])
def test_spectral_ops_on_packed_pairs(emul, precision, tol):
    K.check_spectral_ops(emul, precision, tol, big=False)


@pytest.mark.parametrize("precision,tol", [("f32", 1e-6), ("f64", 1e-13)])
def test_identity_round_trip(emul, precision, tol):
    K.check_identity_ops(emul, precision, tol)


@pytest.mark.parametrize("precision", ["f32", "f64"])
def test_normals_bit_exact_vs_numpy(emul, precision):
    # 40000 normals cross ~20 rounds of the block scan and contain wedge rejections and tail draws
    K.check_normals_bit_exact(emul, precision, [(12345, 16), (1, 2047), (7, 2049), (2026, 40000)])


@pytest.mark.parametrize("name,precision", [("C1b", "f32"), ("C1b", "f64"), ("C2", "f32")])
def test_render_small_configs(emul, name, precision):
    K.check_render(emul, configs.canonical(name), precision)


def test_render_c3_auto_precision(emul):
    p = configs.canonical("C3")
    p["out_dur_s"] = 0.25
    K.check_render(emul, p, "auto")


@pytest.mark.parametrize("mode", configs.BASIC_MODES)
def test_render_every_generator(emul, mode):
    p = configs.with_defaults(gen_mode=mode, event_process="Poisson", out_dur_s=0.4, grains_per_sec=25.0,
                              time_unfold=40.0, micro_ms=2.0, partial_stretch=1.7, space_ir_on=True,
                              _ir_audio=configs.synth_ir(0.05, 48000, 3))
    K.check_render(emul, p, "auto")


def test_render_lanes_multiband_odd_stereo(emul):
    p = configs.with_defaults(event_process="Clustered", out_dur_s=0.30003, base_sr=44100, grains_per_sec=30.0,
                              bp_unfold="0:20, 0.2:33.3", bp_stretch="0:0.5, 0.3:2", bp_cutoff="0:9000,0.3:18000",
                              unfold_mode="Multi-band unfold", gen_mode="Resonant strike")
    assert int(round(p["out_dur_s"] * p["base_sr"])) % 2 == 1        # odd length: FFT rotation path
    K.check_render(emul, p, "auto")


def test_identities_from_the_reference_code(emul):
    from audio_suite_b200 import engine
    base = dict(out_dur_s=0.1, event_process="Single", er_cloud_on=False, gen_mode="Gaussian click")
    # stereo_on False -> L == R (M:778); final max|out| == peak (M:781)
    out, meta = engine.render(configs.with_defaults(base, stereo_on=False, peak=0.5), device=emul)
    assert np.array_equal(out[:, 0], out[:, 1]) and abs(np.max(np.abs(out)) - 0.5) < 1e-6
    # bandlimit off and stretch 1 -> grain_last == micro_last (M:688-729)
    out, meta = engine.render(configs.with_defaults(base, bandlimit_on=False, partial_stretch=1.0), device=emul)
    assert np.array_equal(meta["grain_last"], meta["micro_last"])
    assert meta["micro_last"][0] == 0.0                                  # fade-in starts at exactly 0 (M:267)
    # unit-impulse IR leaves the output unchanged; an IR shorter than 8 samples is skipped (M:439)
    ref, _ = engine.render(configs.with_defaults(base), device=emul, precision="f64")
    imp = np.zeros(64); imp[0] = 1.0
    a, _ = engine.render(configs.with_defaults(base, space_ir_on=True, _ir_audio=imp), device=emul, precision="f64")
    b, _ = engine.render(configs.with_defaults(base, space_ir_on=True, _ir_audio=np.ones(7)), device=emul, precision="f64")
    assert np.max(np.abs(a - ref)) < 1e-6 and np.array_equal(b, ref)


def test_progress_call_shapes(emul):
    from audio_suite_b200 import engine
    from oracle import microsound_np as O
    p = configs.with_defaults(event_process="Poisson", out_dur_s=0.5, grains_per_sec=300.0, micro_ms=0.5)
    a, b = [], []
    engine.render(p, progress=lambda pct, msg: a.append((pct, msg)), device=emul)
    O.render(p, progress=lambda pct, msg: b.append((pct, msg)))
    assert a == b and a[0][0] == 0 and a[-1] == (100, "Done.")


def test_batch_equals_single_renders(emul):
    from audio_suite_b200 import engine
    ps = [configs.with_defaults(seed=s, out_dur_s=0.1, gen_mode=m, time_unfold=u)
          for s, m, u in ((1, "Gaussian click", 25.0), (2, "Noise burst", 30.0), (3, "Gaussian click", 25.0))]
    batch = engine.render_batch(ps, device=emul, precision="f64")
    for p, got in zip(ps, batch):
        one, _ = engine.render(p, device=emul, precision="f64")
        assert np.max(np.abs(got.astype(np.float64) - one)) < 1e-6     # pairing changes rounding only


def test_pooled_and_streamed_planning_match_in_process(emul):
    """Large batches are planned and packed by worker processes in relocatable chunks, streamed (render_batch) or as one
    batch (plan_and_pack); the merged tables must render exactly what the single-chunk path renders."""
    from audio_suite_b200 import engine, tables as T
    ps = [configs.with_defaults(seed=10 + s, out_dur_s=0.05 + 0.01 * (s % 2), gen_mode=m, time_unfold=u, space_ir_on=True,
                                _ir_audio=configs.synth_ir(0.02, 48000, 3))
          for s, (m, u) in enumerate([("Gaussian click", 25.0), ("Noise burst", 30.0), ("Dust impulses", 25.0),
                                      ("Resonant strike", 30.0), ("Skewed transient", 25.0), ("Gaussian click", 30.0),
                                      ("Resonant strike", 25.0)])]
    ps[3]["base_sr"], ps[3]["out_dur_s"] = 44100, 0.05003          # odd length -> FFT rotation path
    # the stages outside the native planner's family, split across pieces
    extra = dict(event_process="Poisson", out_dur_s=0.15, grains_per_sec=30.0, micro_ms=2.0, er_cloud_on=False, bandlimit_on=False)
    ps += [configs.with_defaults(extra, seed=40, cep_warp_on=True, cep_factor=1.2, gen_mode="Resonant strike"),
           configs.with_defaults(extra, seed=41, res_bank_on=True, wg_on=True, wg_max_ms=1.0, partial_lock_on=True, partial_stretch=1.1,
                                 unfold_mode="Multi-band unfold", gen_mode="Stick–slip friction"),
           configs.with_defaults(extra, seed=42, event_feedback_on=True, spectral_imprint_on=True, res_bank_on=True, gen_mode="Gaussian click"),
           configs.with_defaults(extra, seed=43, spectral_imprint_on=True, gen_mode="Wavelet atoms")]
    one = engine.render_batch(ps, device=emul)
    streamed = engine.render_batch(ps, device=emul, chunk=5, workers=3, piece=2)     # slices of 5 = pieces of 2+2+1, 2
    ramped = engine.render_batch(ps, device=emul, chunk=[1, 2, 3], workers=2, piece=2)  # slice schedule 1, 2, 3, 3: short first slices
    for a, c in zip(one, ramped):
        assert a.shape == c.shape and np.max(np.abs(a.astype(np.float64) - c.astype(np.float64))) < 1e-6
    tb, plans = T.plan_and_pack(ps, workers=3, min_batch=2)                          # through the pool
    assert plans is None
    br = engine.BatchRenderer(device=emul, tables=tb)
    br.run()
    pooled = [br.output(r) for r in range(br.n_renders)]
    br.close()
    for a, b, c in zip(one, pooled, streamed):
        assert a.shape == b.shape and np.max(np.abs(a.astype(np.float64) - b.astype(np.float64))) < 1e-6
        assert a.shape == c.shape and np.max(np.abs(a.astype(np.float64) - c.astype(np.float64))) < 1e-6


@pytest.mark.parametrize("name", list(K.PRESET_LIKE))
def test_preset_rows_wavelet_atoms_and_imprint(emul, name):
    """SURVEY 8(f) rows now accelerated: the wavelet-atom generator and the spectral imprint (sequential across the
    events of a render), on shortened versions of the shipped presets that need nothing else."""
    p = K.preset_like(name)
    p["out_dur_s"] = 0.3 if p["event_process"] == "Hawkes" else 1.2          # the Hawkes presets fire hundreds of events per second
    K.check_render(emul, p, "f64")


def test_imprint_restarts_when_the_grain_length_changes(emul):
    p = K.preset_like("soft_ellipse_memory")
    p["out_dur_s"], p["bp_unfold"], p["grains_per_sec"] = 1.0, "0:25, 0.5:25, 0.51:31, 1:31", 20.0
    K.check_render(emul, p, "f64")


@pytest.mark.parametrize("power,stretch,odd", [(1.25, 1.0, False), (0.6, 2.3, False), (3.0, 0.7, True)])
def test_power_warp_fused_into_the_grain_operator(emul, power, stretch, odd):
    """fft_warp_power (main_v2.py:103-115) between the low-pass and the stretch: a gather of a gather."""
    p = configs.with_defaults(nl_warp_on=True, nl_warp_power=power, partial_stretch=stretch, event_process="Poisson",
                              out_dur_s=0.6, grains_per_sec=20.0, gen_mode="Resonant strike", er_cloud_on=False,
                              bp_unfold="0:25, 0.6:25.013" if odd else "")
    K.check_render(emul, p, "f64")


@pytest.mark.parametrize("kw", [dict(partial_stretch=1.05), dict(partial_stretch=1.0),
                                dict(partial_stretch=0.7, pl_top_n=60, pl_neigh=9, unfold_mode="Multi-band unfold"),
                                dict(partial_stretch=1.3, nl_warp_on=True, bandlimit_roll_hz=0.0, gen_mode="Noise burst")])
def test_partial_lock(emul, kw):
    """partial_lock_stretch (main_v2.py:130-148): top-N bin selection, triangular scatter, 12 % dry spectrum."""
    base = dict(partial_lock_on=True, event_process="Poisson", out_dur_s=0.6, grains_per_sec=20.0,
                gen_mode="Resonant strike", er_cloud_on=False)
    base.update(kw)
    K.check_render(emul, configs.with_defaults(base), "f64")


@pytest.mark.parametrize("kw", [dict(gen_mode="Crackle / corona"),
                                dict(gen_mode="Crackle / corona", crackle_density=900, crackle_kernel=8, micro_ms=4.0),
                                dict(gen_mode="IR fragment", _ir_audio=configs.synth_ir(0.25, 48000, 11, channels=1)),
                                dict(gen_mode="IR fragment"),                                     # no IR loaded: silence
                                dict(gen_mode="Image scanline", _img_gray=np.random.default_rng(5).integers(0, 256, (40, 300)).astype(np.uint8)),
                                dict(gen_mode="Image scanline"),
                                dict(gen_mode="Micro-chaos"),
                                dict(gen_mode="Micro-chaos", chaos_r=3.99, chaos_gate=0.9, micro_ms=3.0, seed=20000),
                                dict(gen_mode="Stick–slip friction"),
                                dict(gen_mode="Stick–slip friction", ss_threshold=0.5, ss_build=0.2, ss_decay=0.9, ss_noise=0.3, micro_ms=3.0)])
def test_next_row_generators(emul, kw):
    """gen_crackle (main_v2.py:271-281), gen_ir_fragment (:333-348), gen_image_scanline (:350-362), gen_micro_chaos
    (:303-315; the logistic map must stay bit-identical over thousands of iterations)."""
    p = configs.with_defaults(event_process="Poisson", out_dur_s=0.6, grains_per_sec=20.0, er_cloud_on=False, **kw)
    K.check_render(emul, p, "f64")


@pytest.mark.parametrize("kw", [dict(cep_factor=1.45, gen_mode="Resonant strike", nl_warp_on=True, unfold_mode="Multi-band unfold",
                                     partial_stretch=1.3),
                                dict(cep_factor=0.8, gen_mode="Gaussian click", bp_unfold="0:25,0.6:25.013"),
                                dict(cep_factor=1.2, gen_mode="Wavelet atoms", partial_lock_on=True),
                                dict(cep_factor=1.1, partial_lock_on=True, partial_stretch=0.8, unfold_mode="Multi-band unfold",
                                     res_bank_on=True, nl_warp_on=True),
                                dict(cep_factor=1.25, gen_mode="Noise burst", bandlimit_on=True)])
def test_cepstral_warp(emul, kw):
    """cepstral_warp (main_v2.py:150-163) as forward / log / inverse / resample / forward / exp / inverse.  Without the
    band-limit the reference is well conditioned and the match is at float32-output level; after a band-limit its own
    output is decided by rounding noise (oracle.rounding_noise_floor), which is what the last case documents."""
    base = dict(event_process="Poisson", out_dur_s=0.6, grains_per_sec=20.0, er_cloud_on=False, cep_warp_on=True, bandlimit_on=False)
    base.update(kw)
    p = configs.with_defaults(base)
    err = K.check_render(emul, p, "f64")
    if not p["bandlimit_on"]:
        assert err < 1e-6
    else:
        assert O.rounding_noise_floor(p) > 1e-3          # the reference itself moves by this much under a 1e-15 jitter


@pytest.mark.parametrize("kw", [dict(), dict(unfold_mode="Multi-band unfold", partial_stretch=1.2),
                                dict(partial_lock_on=True, partial_stretch=0.88, res_modes=36, res_fmin=90, res_fmax=4200,
                                     res_decay_ms=160, micro_ms=3.5),
                                dict(gen_mode="Wavelet atoms", nl_warp_on=True, unfold_mode="Multi-band unfold", spectral_imprint_on=True)])
def test_resonator_bank(emul, kw):
    """resonator_bank (main_v2.py:369-384) between the stretch / partial lock and the multiband unfold."""
    base = dict(event_process="Poisson", out_dur_s=0.6, grains_per_sec=20.0, er_cloud_on=False, res_bank_on=True, gen_mode="Resonant strike")
    base.update(kw)
    assert K.check_render(emul, configs.with_defaults(base), "f64") < 1e-6


@pytest.mark.parametrize("kw", [dict(gen_mode="Resonant strike", wg_max_ms=1.0),
                                dict(res_bank_on=True, unfold_mode="Multi-band unfold", gen_mode="Stick–slip friction", wg_lines=12,
                                     wg_max_ms=0.6, partial_lock_on=True, partial_stretch=1.1)])
def test_waveguide(emul, kw):
    """waveguide_splinters (main_v2.py:386-402): feedback combs walked chain by chain (samples d apart)."""
    base = dict(event_process="Poisson", out_dur_s=0.6, grains_per_sec=20.0, er_cloud_on=False, wg_on=True)
    base.update(kw)
    assert K.check_render(emul, configs.with_defaults(base), "f64") < 1e-6


@pytest.mark.parametrize("kw", [dict(gen_mode="Resonant strike", bp_unfold="0:25,0.3:40,0.6:25", event_feedback_amt=0.8),
                                dict(gen_mode="Wavelet atoms", spectral_imprint_on=True, bandlimit_on=False, bp_unfold="0:25,0.3:40,0.6:25"),
                                dict(gen_mode="Gaussian click", spectral_imprint_on=True, bandlimit_on=False, res_bank_on=True,
                                     nl_warp_on=True, unfold_mode="Multi-band unfold")])
def test_event_feedback(emul, kw):
    """Event feedback (main_v2.py:731-740): every grain is mixed with the previous event's FINAL grain (after feedback
    and imprint), so a render's events run rank by rank; the imprint's moving average advances one grain per rank."""
    base = dict(event_process="Poisson", out_dur_s=0.6, grains_per_sec=20.0, er_cloud_on=False, event_feedback_on=True)
    base.update(kw)
    assert K.check_render(emul, configs.with_defaults(base), "f64") < 1e-6


def test_every_shipped_preset_shape_is_accepted():
    """All 27 shipped presets now plan (no NotImplementedError left on the SURVEY 8(f) list)."""
    from audio_suite_b200 import plan as P
    for name in K.PRESET_LIKE:
        P.plan_render(K.preset_like(name))


# ---- round 2 ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kw", [dict(), dict(gen_mode="Crackle / corona"), dict(gen_mode="Micro-chaos")])
def test_first_placed_sample_survives_the_fir_stage(emul, kw):
    """ADVICE r1 (tables.py x_begin): Poisson events, no grain offset, reflection cloud on -- the first placed sample is
    not an exact zero after the band-limit or for generators without a fade-in, and must come through the FIR stage."""
    p = configs.with_defaults(dict(event_process="Poisson", grain_offset_on=False, er_cloud_on=True, out_dur_s=0.5, grains_per_sec=14.0), **kw)
    assert K.check_render(emul, p, "f64") < 1e-6


def test_fused_fir_blocks_of_65536(emul):
    """8192-tap IR + reflection cloud -> 65536-point blocks: the fused three-phase FIR path (ms_fir_fused.cuh), one and
    several block pairs, with and without taps."""
    p = configs.c5_params(3)
    p["out_dur_s"] = 0.5
    assert K.check_render(emul, p, "f64") < 1e-6
    p = configs.c5_params(7)
    p.update(out_dur_s=2.6, event_process="Poisson", grains_per_sec=4.0, grain_offset_on=False)        # three blocks -> two units
    assert K.check_render(emul, p, "f64") < 1e-6
    p = configs.c5_params(5)
    p.update(out_dur_s=3.0, er_cloud_on=False, event_process="Poisson", grains_per_sec=3.0)            # IR only, long output
    assert K.check_render(emul, p, "f64") < 1e-6


@pytest.mark.parametrize("name", ["oval_room_trace", "image_grain_hallucination", "closed_curve_air", "02_friction_lattice",
                                  "basinski_oval_decay", "room_as_particle"])
def test_shipped_presets_from_the_reference_fixture(emul, name):
    """A subset of the 27 shipped presets on the block emulator (the GPU suite runs all of them): audio against the
    reference's 2 s render, progress messages with their notes, stage-level checks where the floor demands them."""
    fx = K.preset_fixture()
    p = fx[name][0]
    if name in ("closed_curve_air", "02_friction_lattice"):
        # (kept short on the CPU: compare against the oracle instead of the 2 s fixture)
        p = dict(p, out_dur_s=0.5)
        K.check_render(emul, p, "f64")
        return
    K.check_preset(emul, name, fx)


def test_results_do_not_depend_on_the_thread_schedule():
    """Race check without compute-sanitizer (closed on the GPU pool, profiles/r02_compute_sanitizer_closed.log): the block
    emulator visits the fibres of a block in a fresh pseudo-random order between every two barriers (MS_EMUL_SHUFFLE); a
    shared-memory race -- a read that is not separated from a write by a barrier -- changes the result with the order.
    Covers the warp-local FFTs and the fused FIR phases, the block-wide in-place passes, in-tile and global Bluestein, the
    post passes, overlap-add, every generator; bitwise equality across schedules."""
    import subprocess
    import sys
    code = r'''
import sys, hashlib
sys.path.insert(0, %r); sys.path.insert(0, %r); sys.path.insert(0, %r)
import numpy as np
from emul_device import EmulDevice
from audio_suite_b200 import configs, engine
dev = EmulDevice()
W = configs.with_defaults
ir = configs.synth_ir(0.05, 48000, 3)
ps = [configs.canonical("C1b")]
p = configs.c5_params(3); p["out_dur_s"] = 0.3; ps.append(p)
for mode in configs.BASIC_MODES:
    ps.append(W(gen_mode=mode, event_process="Poisson", out_dur_s=0.2, grains_per_sec=25.0, time_unfold=40.0, micro_ms=2.0, partial_stretch=1.7,
                space_ir_on=True, _ir_audio=ir))
ps.append(W(event_process="Clustered", out_dur_s=0.10003, base_sr=44100, grains_per_sec=30.0, bp_unfold="0:20, 0.1:33.3", unfold_mode="Multi-band unfold"))
ps.append(W(cep_warp_on=True, bandlimit_on=False, res_bank_on=True, wg_on=True, wg_max_ms=1.0, event_feedback_on=True, spectral_imprint_on=True,
            event_process="Poisson", out_dur_s=0.2, grains_per_sec=25.0, micro_ms=2.0, gen_mode="Micro-chaos"))
ps.append(W(partial_lock_on=True, partial_stretch=1.3, pl_top_n=60, pl_neigh=9, event_process="Poisson", out_dur_s=0.2, grains_per_sec=25.0,
            gen_mode="Resonant strike", er_taps=2000))              # lock: compaction + gather; cloud: many taps sharing a delay
h = hashlib.sha256()
for p in ps:
    out, meta = engine.render(p, device=dev, precision="f64")
    h.update(out.tobytes()); h.update(meta["grain_last"].tobytes())
print(h.hexdigest())
'''
    import os
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = code % (root, os.path.join(root, "tests"), os.path.join(root, "tests", "host_emul"))
    digests = []
    for seed in (None, "1", "2", "12345"):
        env = dict(os.environ)
        env.pop("MS_EMUL_SHUFFLE", None)
        if seed:
            env["MS_EMUL_SHUFFLE"] = seed
        digests.append(subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, check=True).stdout.strip().splitlines()[-1])
    assert len(set(digests)) == 1, digests
