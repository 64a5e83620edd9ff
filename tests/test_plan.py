"""Host planner vs the oracle's scalar decisions: every integer (grain length, design rate, start,
offset, length, tap delay, roll) must be bit-exact; float64 scalars must be identical."""
import numpy as np
import pytest

from audio_suite_b200 import configs, plan as P
from oracle import microsound_np as O


def _param_sets():
    W = configs.with_defaults
    for name in ("C1", "C1b", "C2", "C3"):
        yield name, configs.canonical(name)
    for i in (0, 1, 2, 17, 100, 4095):
        yield f"C5[{i}]", configs.c5_params(i)
    yield "poisson", W(event_process="Poisson", out_dur_s=3.0, bp_unfold="0:20, 1:33.3, 2:25", bp_stretch="0:.5,3:2")
    yield "clustered", W(event_process="Clustered", out_dur_s=3.0)
    yield "hawkes", W(event_process="Hawkes", out_dur_s=1.0)
    yield "offset_small", W(event_process="Poisson", out_dur_s=2.0, grain_offset_max_ms=0.4)
    yield "past_end", W(event_process="Poisson", out_dur_s=0.3, micro_ms=40.0)
    c4 = configs.canonical("C4")
    c4["out_dur_s"] = 30.0
    yield "C4_30s", c4


@pytest.mark.parametrize("name,params", list(_param_sets()))
def test_segment_map_is_bit_exact(name, params):
    want = O.plan_events(params)
    got = P.plan_render(params)
    assert (got.base_sr, got.out_n, got.design_sr_base) == (want["base_sr"], want["out_n"], want["design_sr_base"])
    assert len(got.events) == len(want["events"])
    for g, w in zip(got.events, want["events"]):
        assert (g.index, g.gen_sr, g.n, g.start, g.offset, g.length, g.placed) == \
               (w["index"], w["gen_sr"], w["n"], w["start"], w["offset"], w["length"], w["placed"])
        assert g.amp == w["amp"] and g.t0 == w["t0"] and g.stretch == w["stretch"] and g.cutoff_gen == w["cutoff_gen"]


def test_c4_design_rate_clip():
    p = configs.canonical("C4")
    p["out_dur_s"] = 5.0
    rp = P.plan_render(p)
    assert rp.design_sr_base == 30_000_000 and all(e.n == 300000 and e.gen_sr == 30_000_000 for e in rp.events)
    assert all(e.cutoff_gen == 18000.0 * 500.0 for e in rp.events)      # unclipped unfold in the cutoff (M:691)


def test_reflection_taps_and_stereo_shifts():
    for sr, seed in ((48000, 12345), (96000, 7), (44100, 99)):
        o1, g1 = P.reflection_taps(sr, 320, 45.0, seed)
        o2, g2 = O.reflection_taps(sr, 320, 45.0, seed)
        assert np.array_equal(o1, o2) and np.array_equal(g1, g2)
    rp = P.plan_render(configs.canonical("C3"))
    dl, dr, w = O.stereo_shifts(48000, 0.65)
    assert (rp.stereo_dl, rp.stereo_dr) == (dl, dr) and rp.stereo_theta == 0.9 * w


def test_half_to_even_rounding_everywhere():
    p = configs.with_defaults(base_sr=48000, out_dur_s=0.05001, time_unfold=1.00001, micro_ms=0.3333)
    assert P.plan_render(p).out_n == O.plan_events(p)["out_n"]
    assert P.grain_length(44100, 2.5 / 44.1) == int(max(16, round(44100 * (2.5 / 44.1) / 1000.0)))


def test_missing_key_raises_keyerror_like_reference():
    p = configs.with_defaults()
    del p["env_a"]
    with pytest.raises(KeyError):
        P.plan_render(p)


def test_every_next_row_is_accepted_now():
    """SURVEY 8(f): nothing on the reference's render path raises NotImplementedError any more."""
    P.plan_render(configs.with_defaults(event_feedback_on=True, spectral_imprint_on=True, event_process="Poisson"))
    P.plan_render(configs.with_defaults(cep_warp_on=True, partial_lock_on=True, partial_stretch=1.2))
    P.plan_render(configs.with_defaults(gen_mode="Stick–slip friction", wg_on=True, res_bank_on=True, cep_warp_on=True))
    P.plan_render(configs.with_defaults(partial_lock_on=True, nl_warp_on=True))
    P.plan_render(configs.with_defaults(gen_mode="Wavelet atoms"))          # accelerated since (SURVEY 8f ranks 1-2)
    P.plan_render(configs.with_defaults(spectral_imprint_on=True))


def test_mask_edges_follow_reference_branching():
    e = P.lowpass_edge(4_800_000.0, 1.8e6, 0.0)
    assert (e.hi_mode, e.hi_f0) == (1, 1.8e6)
    e = P.lowpass_edge(48000.0, 30000.0, 2500.0)           # cutoff clipped to nyquist
    assert (e.hi_mode, e.hi_f0, e.hi_f1) == (2, 24000.0, 24000.0)
    e = P.bandpass_edge(48000.0, 0.0, 0.0, 100.0)
    assert e.zero == 1
    e = P.bandpass_edge(48000.0, 1000.0, 30000.0, 500.0)
    assert (e.lo_mode, e.lo_f0, e.lo_f1, e.hi_mode) == (2, 500.0, 1000.0, 0)


def test_bessel_taps_reproduce_the_rotation_filter():
    from audio_suite_b200.tables import bessel_coeffs as _bessel_coeffs
    rng = np.random.default_rng(1)
    for n, sr, width in ((4800, 48000, 0.65), (960, 96000, 1.0)):
        x = rng.standard_normal(n)
        want = O.stereo_diffuse(x, sr, width)[:, 1]
        dl, dr, w = O.stereo_shifts(sr, width)
        c = _bessel_coeffs(0.9 * w)
        K = (len(c) - 1) // 2
        got = sum(c[K + m] * np.roll(x, -(dr + 2 * m)) for m in range(-K, K + 1))
        assert np.max(np.abs(got - want)) < 1e-12


# ---- round 2 ---------------------------------------------------------------------------------------------------------------
def test_malformed_lane_raises_like_the_reference():
    """'a:b:c' makes the reference's `t, v = part.split(":")` raise ValueError (main_v2.py:461 sits outside its try)."""
    from oracle import ref_loader
    for fn in (P.parse_breakpoints, O.parse_lane) + ((ref_loader.load().parse_breakpoints,) if ref_loader.available() else ()):
        with pytest.raises(ValueError):
            fn("0:1:2, 3:4")
        assert list(fn("0:1, x:2, 3, 4:5")) == [(0.0, 1.0), (4.0, 5.0)]


def test_pooled_planning_keeps_the_whole_ir_for_the_fragment_generator():
    """ADVICE r1 (plan.py _slim_params): gen_ir_fragment draws its 256-sample piece from the WHOLE mono mix, not from the
    8192 taps the convolution keeps; a 2-D IR of 4..7 rows passes the reference's size >= 8 test (rows x channels)."""
    from audio_suite_b200 import tables as T
    ir = configs.synth_ir(1.0, 48000, 21)                       # 48000 x 2
    for kw in (dict(gen_mode="IR fragment", space_ir_on=True), dict(gen_mode="IR fragment", space_ir_max_samps=0, space_ir_on=True),
               dict(gen_mode="Gaussian click", space_ir_on=True, _ir_audio=np.ones((5, 2))), dict(gen_mode="IR fragment", _ir_audio=np.ones((5, 2)))):
        p = configs.with_defaults(dict(event_process="Poisson", out_dur_s=0.5, _ir_audio=ir), **kw)
        a = T.pack_chunk([P.plan_render(p)])
        b = T.pack_chunk([P.plan_render(P._slim_params(p))])
        for name in ("sy1", "ola_e", "fir", "dust_val", "irs", "tap_gain"):
            x, y = getattr(a, name), getattr(b, name)
            assert x.shape == y.shape and x.tobytes() == y.tobytes(), (kw, name)


def test_streamed_planning_does_not_deadlock_on_large_requests():
    """ADVICE r1 (tables.py plan_stream): requests larger than the pipe (a 4 MB `_img_gray` per piece) used to block the
    parent on a write while the worker blocked on its answer.  Requests now leave from a feeder thread, for streamed
    batches and for the pooled batches of plan_and_pack (BatchRenderer(params_list)) alike."""
    import threading
    from audio_suite_b200 import tables as T
    img = np.random.default_rng(3).integers(0, 256, (2048, 2048)).astype(np.uint8)
    ps = [configs.with_defaults(gen_mode="Image scanline", seed=i, out_dur_s=0.05, _img_gray=img) for i in range(300)]
    for plan, renders, slices in ((lambda: T.plan_stream(ps[:96], 32, workers=2, piece=16), 96, 3),
                                  (lambda: [T.plan_and_pack(ps, workers=2)[0]], 300, 1)):
        got = []
        th = threading.Thread(target=lambda: got.extend(plan()), daemon=True)
        th.start()
        th.join(120)
        stuck = th.is_alive()
        if stuck:                        # a writer blocked on a full pipe holds its lock: closing the pipe would hang too
            for proc in T._POOL.procs:
                proc.kill()
        T.shutdown_pool()
        assert not stuck and len(got) == slices and sum(len(t.post) for t in got) == renders
