"""Long impulse responses (EXTENSION; the reference keeps 8192 taps, main_v2.py:443): the optional key `space_ir_tap_cap`
through both planners, and the FIR stage's uniformly partitioned overlap-save route for rows with more than 8192 IR taps,
against float64 convolution.

The CPU tests drive ms_fir_* on the block emulator with MS_FIR_PART forcing small partitions, so every branch of the route
(head entries, partial last partition, skipped blocks, the clip to out_n - x_begin taps) runs at emulator sizes.  The GPU
tests repeat the stage at full size (one subprocess per MS_FIR_PART: the CUDA build reads it once per process), run C4 with
its whole 10 s IR, and check that capped renders do not change when uncapped renders share their batch.

Worst errors relative to max|ref|, measured: block emulator f64 1.1e-15, f32 7.6e-7 (P forced to 64 and 4096); NVIDIA B200
(1000 W power limit) f64 1.5e-15, f32 8.7e-7 (IRs of 240000 and 960000 taps, P by the rule, 4096 and 32768), C4 with its whole
IR 1.1e-15 in situ.  So the short route's tolerances (stage_checks.FIR_TOL, 1e-13 / 3e-6) hold for this route as well."""
import functools
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import stage_checks as S
from audio_suite_b200 import configs, engine, hostplan, plan as P, tables as T
from oracle import microsound_np as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _ir_params(ir, **kw):
    base = dict(gen_mode="Resonant strike", micro_ms=5.0, time_unfold=30.0, out_dur_s=0.25, event_process="Poisson",
                grains_per_sec=20.0, bp_density="", space_ir_on=True, space_ir_max_samps=40000, er_cloud_on=True, er_taps=40,
                stereo_on=True, _ir_audio=ir)
    base.update(kw)
    return configs.with_defaults(base)


def _same_tables(a, b):
    for name in a.__dataclass_fields__:
        x, y = getattr(a, name), getattr(b, name)
        if isinstance(x, np.ndarray):
            assert x.dtype == y.dtype and x.shape == y.shape and x.tobytes() == y.tobytes(), name
        else:
            assert x == y, name


# ---- planners -------------------------------------------------------------------------------------------------------------
def test_default_cap_tables_unchanged():
    ir = configs.synth_ir(0.1, 48000, 5)                        # 4800 rows: below every cap tried
    want = T.pack_chunk([P.plan_render(_ir_params(ir))])
    for cap in (8192, 20000, None):
        _same_tables(want, T.pack_chunk([P.plan_render(_ir_params(ir, space_ir_tap_cap=cap))]))
    long_ir = configs.synth_ir(0.5, 48000, 6)
    assert P.plan_render(_ir_params(long_ir)).ir.size == 8192
    _same_tables(T.pack_chunk([P.plan_render(_ir_params(long_ir))]),
                 T.pack_chunk([P.plan_render(_ir_params(long_ir, space_ir_tap_cap=8192))]))


def test_cap_rule_slice_cut_mix():
    ir = configs.synth_ir(0.7, 48000, 7)                        # 33600 x 2
    rp = P.plan_render(_ir_params(ir, space_ir_max_samps=20000, space_ir_tap_cap=None))
    assert np.array_equal(rp.ir, ir[:20000].astype(np.float64).mean(axis=1))
    rp = P.plan_render(_ir_params(ir, space_ir_max_samps=20000, space_ir_tap_cap=12345))
    assert np.array_equal(rp.ir, ir[:12345].astype(np.float64).mean(axis=1))
    assert P.plan_render(_ir_params(ir[:3], space_ir_tap_cap=None)).ir is None       # "< 8 values" on the slice: 6 values
    assert P.plan_render(_ir_params(ir, space_ir_max_samps=3, space_ir_tap_cap=None)).ir is None


def test_pooled_digest_carries_cap():
    ir = configs.synth_ir(0.7, 48000, 8)
    for cap, n in ((None, 30000), (10000, 10000), (8192, 8192)):
        p = _ir_params(ir, space_ir_max_samps=30000, space_ir_tap_cap=cap)
        q = P._slim_params(p)
        assert q["_ir_audio"] is None and q["_ir_digest"]["taps"].size == n
        _same_tables(T.pack_chunk([P.plan_render(p)]), T.pack_chunk([P.plan_render(q)]))


def test_native_planner_long_ir():
    subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "audio_suite_b200", "csrc"), "libms_hostplan.so"])
    hostplan._lib = None
    assert hostplan.lib() is not None
    ir = configs.synth_ir(1.0, 48000, 9)
    ps = [_ir_params(ir, seed=11 + i, space_ir_tap_cap=cap, space_ir_max_samps=msamp)
          for i, (cap, msamp) in enumerate([(None, 48000), (30000, 48000), (8192, 48000), (None, 20000), (9000, 9000)])]
    want = T.pack_chunk([P.plan_render(p) for p in ps])
    got = hostplan.plan_chunk(ps)
    for name in want.__dataclass_fields__:
        a, b = getattr(want, name), getattr(got, name)
        if isinstance(a, np.ndarray) and a.dtype.names:
            for f in a.dtype.names:
                if not f.startswith("_pad") and f != "h":
                    assert np.array_equal(a[f], b[f]), (name, f)
        elif isinstance(a, np.ndarray):
            assert np.array_equal(a, b), name
        else:
            assert a == b, name
    assert sorted(set(int(v) for v in got.fir["ir_len"])) == [8192, 9000, 20000, 30000, 48000]


def test_preset_carries_cap(tmp_path):
    from audio_suite_b200 import frontend
    path = tmp_path / "hall.json"
    path.write_text(json.dumps({"space_ir_on": True, "space_ir_tap_cap": None}))
    p = frontend.load_preset(str(path))
    assert "space_ir_tap_cap" in p and p["space_ir_tap_cap"] is None
    assert frontend.load_preset({"space_ir_tap_cap": 20000})["space_ir_tap_cap"] == 20000
    assert "space_ir_tap_cap" not in frontend.load_preset({}) and "space_ir_tap_cap" not in configs.FACTORY_DEFAULTS


def test_cache_keys_differ_by_cap():
    ir = configs.synth_ir(0.3, 48000, 10)
    keys = {engine._cache_key(_ir_params(ir, **kw), None, "f64") for kw in ({}, dict(space_ir_tap_cap=8192),
                                                                             dict(space_ir_tap_cap=None), dict(space_ir_tap_cap=9000))}
    assert len(keys) == 4                                       # (absent and 8192 render the same bits, but are distinct keys)


@pytest.mark.parametrize("cap", [True, False, 0, -5, 1.5, 8192.0, "8192", [8192]])
def test_invalid_cap_raises(cap):
    p = _ir_params(configs.synth_ir(0.3, 48000, 12), space_ir_tap_cap=cap)
    with pytest.raises(ValueError, match="space_ir_tap_cap"):
        P.plan_render(p)
    with pytest.raises(ValueError, match="space_ir_tap_cap"):
        P._slim_params(p)
    if hostplan.lib() is not None:
        with pytest.raises(ValueError, match="space_ir_tap_cap"):
            hostplan.plan_chunk([p])


def test_over_limit_ir_raises():
    ir = np.zeros((P.IR_TAP_LIMIT + 1, 2))
    ir[::1000] = 0.1
    p = _ir_params(ir, space_ir_max_samps=P.IR_TAP_LIMIT + 10, space_ir_tap_cap=None)
    with pytest.raises(ValueError, match="outside the accelerated path"):
        P.plan_render(p)
    with pytest.raises(ValueError, match="outside the accelerated path"):
        P._slim_params(p)
    p["space_ir_tap_cap"] = P.IR_TAP_LIMIT                    # at the limit: accepted
    assert P.plan_render(p).ir.size == P.IR_TAP_LIMIT


# ---- stage: ms_fir_* with long rows ---------------------------------------------------------------------------------------
def _zero_input(cs):
    cs = dict(cs, name=cs["name"] + "-zero-input")
    cs["x"] = np.zeros_like(cs["x"])
    return cs


def long_cases(part, big=False):
    """Hand-built rows around partition length `part` (what MS_FIR_PART forces)."""
    rng = np.random.default_rng(31 if big else 3)
    P_, c = part, []
    k = 8192 // P_ + 1                                           # first multiple of P above 8192
    if not big:
        c += [
            S.fir_case("ir8193-taps", rng, 20000, 8193, 40, 300, 0, x_begin=100, x_end=15000),
            S.fir_case("ir-kP-no-taps", rng, 12000 + P_ // 2, k * P_, 0, 0, 0),
            S.fir_case("ir-kP+1-taps", rng, 15000, k * P_ + 1, 20, 2 * P_ + 3, 0, x_begin=7, x_end=14000),
            S.fir_case("ir-kP-1-late-start", rng, 16000, k * P_ - 1, 12, 500, 0, x_begin=9000, x_end=16000),
            S.fir_case("ir-longer-than-out", rng, 9000, 12000, 10, 200, 0, x_begin=500, x_end=3000),
            S.fir_case("out-shorter-than-P", rng, P_ - 7 if P_ > 16 else 9, 8300, 3, 4, 0, x_begin=1, x_end=P_ - 9 if P_ > 16 else 8),
            S.fir_case("early-end", rng, 30000, 9000, 30, 700, 0, x_begin=2000, x_end=2600),
        ]
        c.append(_zero_input(S.fir_case("ir9100", rng, 14000, 9100, 10, 100, 0, x_begin=40, x_end=13000)))
        c.append(dict(S.fir_case("shared-IR", rng, 18000, 8193, 25, 900, 0, x_begin=3, x_end=17000), ir=c[0]["ir"], share="ir8193-taps"))
        c.append(S.fir_case("second-IR", rng, 11000, 10000, 0, 0, 0, x_begin=0, x_end=11000))
    else:
        c += [
            S.fir_case("ir240000-60s-taps", rng, 5_760_000, 240000, 320, 4320, 0, x_begin=1000, x_end=5_600_000, dup=8),
            S.fir_case("ir960000-no-taps", rng, 2_000_000, 960000, 0, 0, 0, x_begin=300_000, x_end=1_500_000),
            S.fir_case("ir960000-clip", rng, 700_000, 960000, 100, 4320, 0, x_begin=50_000, x_end=400_000),
            S.fir_case("ir8193-early-end", rng, 1_000_000, 8193, 40, 2000, 0, x_begin=100, x_end=20_000),
        ]
        c.append(dict(S.fir_case("shared-960000", rng, 1_200_000, 960000, 50, 3000, 0, x_begin=7, x_end=1_100_000),
                      ir=c[1]["ir"], share="ir960000-no-taps"))
    return c


def short_cases(big=False):
    rng = np.random.default_rng(5)
    s = 3 if big else 1
    return [S.fir_case("short-B8192", rng, 20000 * s, 1000, 40, 2000, 8192, x_begin=300, x_end=15000 * s, dup=3),
            S.fir_case("short-B65536", rng, 150000, 6000, 320, 2160, 65536, x_begin=30, x_end=140000)]


def _refs(cases, precision, fft=False):
    ref = S.fir_reference_fft if fft else S.fir_reference
    return [ref(S._as_ref(cs["ir"], precision), cs["offs"], S._as_ref(cs["gains"], precision), S._as_ref(cs["x"], precision),
                cs["x_begin"], cs["x_end"]) for cs in cases]


def _direct_samples(cs, precision, at):
    """float64 direct sums y[i] = sum_t h[t] x_er[i - t] at the positions `at` (x_er: input + reflection cloud)."""
    x = S._as_ref(cs["x"], precision)
    ir = S._as_ref(cs["ir"], precision)
    xer = x.copy()
    g = S._as_ref(cs["gains"], precision)
    for off, gg in zip(cs["offs"].tolist(), g.tolist()):
        xer[off:] += gg * x[:len(x) - off]
    out = []
    for i in at.tolist():
        lo = max(0, i - len(ir) + 1)
        out.append(float(np.dot(ir[:i - lo + 1], xer[lo:i + 1][::-1])))
    return np.array(out)


def check_long(dev, precision, part, big=False):
    """Long rows alone and mixed with short rows (short rows bitwise equal to running them alone), two runs per handle
    (bitwise equal), the kernels that ran.  Returns {"errors", "kernels"}."""
    cases = long_cases(part, big)
    refs = _refs(cases, precision, fft=big)
    errors = {}
    outs, starts, log = S.fir_run(dev, precision, cases, runs=2)
    assert np.array_equal(outs[0], outs[1], equal_nan=True), "second ms_fir_run on one handle differs"
    assert "FirLongMacK" in log.base() and "FirLongZeroK" in log.base(), sorted(log.base())
    errors.update(S.check_fir_outputs(precision, cases, outs[0], starts, refs=refs, label="long"))
    if big:                                                      # the FFT reference against direct sums
        rng = np.random.default_rng(99)
        for cs, s, r in zip(cases, starts, refs):
            n = len(cs["x"])
            at = np.unique(np.concatenate([rng.integers(cs["x_begin"], n, 24), [n - 1, min(n - 1, cs["x_begin"] + 5)]]))
            want = _direct_samples(cs, precision, at)
            scale = max(1e-300, float(np.max(np.abs(r))))
            e = float(np.max(np.abs(outs[0][s + at] - want))) / scale
            errors["direct:" + cs["name"]] = e
            assert e < S.FIR_TOL[precision], (precision, cs["name"], "direct sums", e)
    shorts = short_cases(big)
    alone, s_starts, slog = S.fir_run(dev, precision, shorts)
    assert "FirLongMacK" not in slog.base() and "FirLongZeroK" not in slog.base(), sorted(slog.base())
    mixed = [cases[0], shorts[0], cases[1], shorts[1]] + cases[2:]
    mouts, m_starts, _ = S.fir_run(dev, precision, mixed)
    for k, cs in ((1, shorts[0]), (3, shorts[1])):
        j = shorts.index(cs)
        n = len(cs["x"])
        assert np.array_equal(mouts[0][m_starts[k]:m_starts[k] + n], alone[0][s_starts[j]:s_starts[j] + n]), (precision, cs["name"])
    srefs = _refs(shorts, precision)
    mrefs = [refs[0], srefs[0], refs[1], srefs[1]] + refs[2:]
    merr = S.check_fir_outputs(precision, mixed, mouts[0], m_starts, refs=mrefs, label="mixed")
    errors.update({"mixed:" + k: v for k, v in merr.items()})
    return {"errors": errors, "kernels": sorted(log.names)}


@pytest.mark.parametrize("precision", ["f64", "f32"])
@pytest.mark.parametrize("part", [64, 256])
def test_long_stage_emulated(emul, precision, part, monkeypatch):
    monkeypatch.setenv("MS_FIR_PART", str(part))              # the emulator reads it at every ms_fir_create
    res = check_long(emul, precision, part)
    worst = max(res["errors"].values())
    print("long FIR %s P=%d: worst %.2e" % (precision, part, worst))


def test_long_stage_thread_schedule():
    """The route under MS_EMUL_SHUFFLE (fibres of a block in a fresh order between barriers): bitwise equal results."""
    code = ("import sys, hashlib; sys.path[:0] = [%r, %r, %r]\n"
            "from emul_device import EmulDevice; import test_long_ir as L, stage_checks as S\n"
            "dev = EmulDevice(); h = hashlib.sha256()\n"
            "for prec in ('f64', 'f32'):\n"
            "    outs, _, _ = S.fir_run(dev, prec, L.long_cases(64) + L.short_cases(), runs=1); h.update(outs[0].tobytes())\n"
            "print(h.hexdigest())\n") % (ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "tests", "host_emul"))
    digests = []
    for seed in (None, "1", "7"):
        env = dict(os.environ, MS_FIR_PART="64")
        env.pop("MS_EMUL_SHUFFLE", None)
        if seed:
            env["MS_EMUL_SHUFFLE"] = seed
        p = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, cwd=ROOT)
        assert p.returncode == 0, p.stderr[-4000:]
        digests.append(p.stdout.strip().splitlines()[-1])
    assert len(set(digests)) == 1, digests


def test_render_uncapped_emulated(emul, monkeypatch):
    """End to end on the emulator against the oracle's render with the same cap (the oracle's constant patched)."""
    import kernel_checks as K
    monkeypatch.setenv("MS_FIR_PART", "512")
    ir = configs.synth_ir(0.4, 48000, 13)                       # 19200 taps
    p = _ir_params(ir, space_ir_tap_cap=None)
    monkeypatch.setattr(O, "IR_TAP_CAP", 10 ** 9)
    K.check_render(emul, p, "f64")
    monkeypatch.setattr(O, "IR_TAP_CAP", 15000)
    K.check_render(emul, dict(p, space_ir_tap_cap=15000), "f64")


# ---- GPU ------------------------------------------------------------------------------------------------------------------
def long_stage_main():
    """Full-size stage checks on cuda:0 under the environment's MS_FIR_PART; prints one JSON line."""
    dev = engine.CudaDevice(0)
    part = int(os.environ.get("MS_FIR_PART", "0")) or 4096
    res = {p: check_long(dev, p, part, big=True) for p in ("f64", "f32")}
    print(json.dumps(res))


@functools.lru_cache(maxsize=None)
def _long_stage_run(part):
    code = "import sys; sys.path[:0] = [%r, %r]; import test_long_ir; test_long_ir.long_stage_main()" % (ROOT, os.path.join(ROOT, "tests"))
    env = dict(os.environ)
    env.pop("MS_FIR_PART", None)
    if part:
        env["MS_FIR_PART"] = str(part)
    p = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, cwd=ROOT)
    assert p.returncode == 0, "MS_FIR_PART=%s:\n%s" % (part, p.stderr[-6000:])
    return json.loads(p.stdout.strip().splitlines()[-1])


@pytest.mark.gpu
@pytest.mark.parametrize("part", [0, 4096, 32768])
def test_long_stage_gpu(cuda_dev, part):
    res = _long_stage_run(part)
    for precision in ("f64", "f32"):
        errs = res[precision]["errors"]
        print("long FIR %s MS_FIR_PART=%s: worst %.2e (%s)" % (precision, part or "rule", max(errs.values()), max(errs, key=errs.get)))


@pytest.mark.gpu
def test_c4_full_ir_in_situ(cuda_dev):
    """C4 with its whole 10 s IR (960000 taps, 57.6 M frames): the FIR stage's input and output read at the stage marks,
    the output compared with float64 direct sums at seeded positions; the post chain as in check_in_situ."""
    from scipy.signal import oaconvolve
    p = configs.canonical("C4")
    p["space_ir_tap_cap"] = None
    br = engine.BatchRenderer([p], device=cuda_dev, precision="f64")
    t = br.tables
    snap = {}

    def mark(name):
        if name == "overlap_add":
            snap["A"] = S._fetch(cuda_dev, br.mono, br.real, t.mono_n).astype(np.float64)
        elif name == "fir_overlap_save":
            snap["B"] = S._fetch(cuda_dev, br.mono, br.real, t.mono_n).astype(np.float64)
    try:
        br.run(mark=mark)
        cuda_dev.synchronize()
        f = t.fir[0]
        assert int(f["ir_len"]) == 960000
        n, x0 = int(f["out_n"]), int(f["x"])
        a = snap["A"][x0:x0 + n]
        y = snap["B"][int(f["y"]):int(f["y"]) + n]
        offs, gains = P.reflection_taps(int(p["base_sr"]), int(p["er_taps"]), float(p["er_max_ms"]), int(p["seed"]))
        keep = (offs > 0) & (offs < n)
        e = np.zeros(int(offs[keep].max()) + 1)
        e[0] = 1.0
        np.add.at(e, offs[keep], gains[keep])
        xer = oaconvolve(a, e)[:n]
        h = P._ir_taps(p["_ir_audio"], int(p["space_ir_max_samps"]), None)
        rng = np.random.default_rng(4)
        xb = int(f["x_begin"])
        at = np.unique(np.concatenate([rng.integers(xb, n, 48), [xb, n - 1]]))
        want = np.array([float(np.dot(h[:i - max(0, i - h.size + 1) + 1], xer[max(0, i - h.size + 1):i + 1][::-1])) for i in at.tolist()])
        scale = float(np.max(np.abs(y)))
        err = float(np.max(np.abs(y[at] - want))) / scale
        print("C4 full IR: FIR stage at %d positions, error %.2e of max|y|" % (at.size, err))
        assert err < S.FIR_TOL["f64"], err
        assert np.all(y[:xb] == 0.0)
        st = O.stereo_diffuse(y, int(p["base_sr"]), float(p["stereo_width"]))
        want = O.peak_normalize(O.soft_saturate(st, float(p["sat_drive"])), float(p["peak"]))
        e_post = float(np.max(np.abs(br.output(0).astype(np.float64) - want)))
        print("C4 full IR: post chain %.2e" % e_post)
        assert e_post < S.POST_OUT_TOL["f64"], e_post
    finally:
        br.close()


@pytest.mark.gpu
def test_batch_mixing_caps(cuda_dev):
    ps = [configs.c5_params(i) for i in range(12)]
    mixed = [dict(p, space_ir_tap_cap=None) if i % 3 == 1 else p for i, p in enumerate(ps)]
    capped = [p for i, p in enumerate(ps) if i % 3 != 1]
    a = [np.array(x) for x in engine.render_batch(mixed, device=cuda_dev)]          # (copies: the outputs are views)
    b = [np.array(x) for x in engine.render_batch(capped, device=cuda_dev)]
    got = [x for i, x in enumerate(a) if i % 3 != 1]
    assert len(got) == len(b)
    for x, y in zip(got, b):
        assert np.array_equal(x, y)
    full = [np.array(x) for x in engine.render_batch([p for i, p in enumerate(mixed) if i % 3 == 1], device=cuda_dev)]
    for x, y in zip([x for i, x in enumerate(a) if i % 3 == 1], full):
        assert np.array_equal(x, y)


@pytest.mark.gpu
def test_render_graph_replay_uncapped(cuda_dev):
    engine.clear_render_cache()
    p = dict(configs.c5_params(5), space_ir_tap_cap=None)
    a, _ = engine.render(p)                                     # eager
    b, _ = engine.render(p)                                     # captured and replayed
    c, _ = engine.render(p)                                     # replayed
    engine.clear_render_cache()
    assert np.array_equal(a, b) and np.array_equal(a, c)
    d, _ = engine.render(configs.c5_params(5), cache=False)
    assert not np.array_equal(a, d)                             # the cap reached the device
