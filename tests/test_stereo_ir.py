"""True-stereo impulse responses (EXTENSION; the reference mixes every IR to mono, main_v2.py:438-445): the optional key
`space_ir_stereo` through both planners, the front end, the FIR stage's pair units (one P1 and one forward row transform
for both channels of a render) and the post stage's stereo mode 3, against float64 restatements.

With u the mono mix after ADSR and the reflection cloud, a stereo render is yL = conv(u, h_L)[:n], yR = conv(u, h_R)[:n],
then L = roll(yL, dl) and R = the spectral rotation of roll(yR, -dr) (stereo on and n >= 64; else [yL, yR]), soft clip
and one joint peak normalisation.  With h_L == h_R == h this is exactly the mono render with h, bit for bit.

The CPU tests run the stage on the block emulator; the GPU tests repeat them in situ on real renders."""
import functools
import json
import os
import struct
import subprocess
import sys

import numpy as np
import pytest

import stage_checks as S
from audio_suite_b200 import configs, engine, frontend, hostplan, plan as P, tables as T
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


def _stereo_ir(seconds, sr, seed):
    """configs.synth_ir with its two channels made clearly different (the right one delayed and darker)."""
    ir = configs.synth_ir(seconds, sr, seed).astype(np.float64)
    ir[:, 1] = np.concatenate([np.zeros(37), ir[:-37, 1]]) * 0.7
    return ir


# ---- planners -------------------------------------------------------------------------------------------------------------
def test_tables_unchanged_without_stereo_ir():
    """Absent, False, and True with a 1-D or one-column IR: byte-identical tables, capped and uncapped."""
    st = _stereo_ir(0.3, 48000, 5)                              # 14400 x 2
    mono = st.mean(axis=1)
    for ir, flags in ((st, ({}, dict(space_ir_stereo=False), dict(space_ir_stereo=np.bool_(False)))),
                      (mono, ({}, dict(space_ir_stereo=False), dict(space_ir_stereo=True))),
                      (mono[:, None], ({}, dict(space_ir_stereo=True)))):
        for cap in ({}, dict(space_ir_tap_cap=None), dict(space_ir_tap_cap=10000)):
            want = T.pack_chunk([P.plan_render(_ir_params(ir, **cap))])
            for kw in flags:
                _same_tables(want, T.pack_chunk([P.plan_render(_ir_params(ir, **cap, **kw))]))


def test_pair_rule():
    ir = _stereo_ir(0.7, 48000, 7)                              # 33600 x 2
    rp = P.plan_render(_ir_params(ir, space_ir_max_samps=20000, space_ir_tap_cap=None, space_ir_stereo=True))
    assert np.array_equal(rp.ir, ir[:20000, 0]) and np.array_equal(rp.ir_r, ir[:20000, 1])
    assert rp.ir.dtype == np.float64 and rp.ir.flags.c_contiguous and rp.ir_r.flags.c_contiguous
    rp = P.plan_render(_ir_params(ir, space_ir_max_samps=20000, space_ir_tap_cap=12345, space_ir_stereo=np.bool_(True)))
    assert np.array_equal(rp.ir, ir[:12345, 0]) and np.array_equal(rp.ir_r, ir[:12345, 1])
    rp = P.plan_render(_ir_params(ir.astype(np.float32), space_ir_stereo=True))            # default cap: 8192 rows
    assert rp.ir.dtype == np.float64 and rp.ir.size == rp.ir_r.size == 8192
    assert np.array_equal(rp.ir_r, ir.astype(np.float32)[:8192, 1].astype(np.float64))
    rp = P.plan_render(_ir_params(ir[:4], space_ir_stereo=True))                            # "< 8 values": 8 values pass
    assert rp.ir.size == rp.ir_r.size == 4
    rp = P.plan_render(_ir_params(ir[:3], space_ir_stereo=True))                            # 6 values
    assert rp.ir is None and rp.ir_r is None
    a, b = P.ir_pair(ir, 30000, None, True), P.ir_pair(ir, 30000, None, True)
    assert a[0] is b[0] and a[1] is b[1]                                                    # cached per IR object
    assert P.plan_render(_ir_params(ir, space_ir_stereo=True, space_ir_on=False)).ir_r is None


@pytest.mark.parametrize("value", [1, 0, "yes", None, 1.0, [True]])
def test_non_bool_raises(value):
    p = _ir_params(_stereo_ir(0.2, 48000, 3), space_ir_stereo=value)
    for call in (P.plan_render, P._slim_params) + ((lambda q: hostplan.plan_chunk([q])),) * (hostplan.lib() is not None):
        with pytest.raises(ValueError, match="space_ir_stereo"):
            call(p)


@pytest.mark.parametrize("shape", [(5000, 3), (5000, 4), (5000, 1, 2), (5000, 2, 1)])
def test_more_than_two_channels_raises(shape):
    ir = np.random.default_rng(1).standard_normal(shape) * 0.1
    p = _ir_params(ir, space_ir_stereo=True)
    with pytest.raises(ValueError, match="space_ir_stereo"):
        P.plan_render(p)
    with pytest.raises(ValueError, match="space_ir_stereo"):
        P._slim_params(p)
    if len(shape) == 2:
        P.plan_render(dict(p, space_ir_stereo=False))            # the mono mix of any channel count, as before


def test_over_limit_per_channel_raises():
    ir = np.zeros((P.IR_TAP_LIMIT + 1, 2))
    ir[::1000] = 0.1
    p = _ir_params(ir, space_ir_max_samps=P.IR_TAP_LIMIT + 10, space_ir_tap_cap=None, space_ir_stereo=True)
    with pytest.raises(ValueError, match="outside the accelerated path"):
        P.plan_render(p)
    rp = P.plan_render(dict(p, space_ir_tap_cap=P.IR_TAP_LIMIT))
    assert rp.ir.size == rp.ir_r.size == P.IR_TAP_LIMIT


def _layout_checks(t, rps):
    """FIR rows and post records of each render as the layout table of INTEGRATION.md states them."""
    plane = sum(rp.out_n for rp in rps)
    fi = 0
    for r, rp in enumerate(rps):
        n, po = rp.out_n, t.post[r]
        if rp.ir is None and rp.er_offs is None:
            continue
        f = t.fir[fi]
        fi += 1
        if rp.ir_r is None:
            continue
        g = t.fir[fi]
        fi += 1
        for k in ("x", "x_begin", "x_end", "tap_begin", "tap_end", "out_n", "h_len", "ir_len", "h"):
            assert f[k] == g[k], k
        assert np.array_equal(t.irs[g["ir"]:g["ir"] + g["ir_len"]], rp.ir_r)
        y_r = int(g["y"])
        assert y_r >= 2 * plane and int(po["y"]) == int(f["y"])
        if not rp.stereo_on:
            assert (po["stereo_mode"], po["rbuf"], po["dl"]) == (2, y_r, 0)
        elif n % 2 == 0:
            assert (po["stereo_mode"], po["rbuf"]) == (3, y_r + n)
            assert np.array_equal(po["coef"], T.bessel_coeffs(rp.stereo_theta))
        else:
            assert (po["stereo_mode"], po["rbuf"]) == (2, y_r + 2 * n)
            assert any(tuple(o) == (y_r, y_r + n, n, rp.stereo_dr) for o in t.odd.tolist())


def test_tables_layout():
    st = _stereo_ir(0.3, 48000, 6)
    ps = [_ir_params(st, space_ir_stereo=True, out_dur_s=d, stereo_on=s, er_cloud_on=e, seed=3 + i, env_a=0.1, env_d=0.0, env_r=0.0)
          for i, (d, s, e) in enumerate([(0.25, True, True), (0.2500208, True, False), (0.25, False, True), (0.001, True, True)])]
    rps = [P.plan_render(p) for p in ps]
    assert rps[1].out_n % 2 == 1 and rps[3].out_n < 64 and not rps[3].stereo_on
    t = T.pack_chunk(rps)
    _layout_checks(t, rps)
    assert len(t.fir) == 8
    mono = T.pack_chunk([P.plan_render(dict(p, space_ir_stereo=False)) for p in ps])
    assert t.alg["fir_taps"] == 2 * mono.alg["fir_taps"] and t.alg["fir_in"] == 2 * mono.alg["fir_in"]
    assert len(t.irs) == 2 * 8192                               # one pair in the pool for the four renders


def _stereo_regions(t):
    """(start, length, (render, kind)) of every mono region of every render, stereo-IR extra regions included; checks
    that they do not overlap."""
    rows = {}
    for f in t.fir:
        rows.setdefault(int(f["x"]), []).append(f)
    regs = []
    for r, (o, p) in enumerate(zip(t.ola_r, t.post)):
        n, mode, at = int(p["n"]), int(p["stereo_mode"]), int(o["out"])
        regs.append((at, n, (r, "ola")))
        if int(p["y"]) != at:
            regs.append((int(p["y"]), n, (r, "fir")))
        fr = rows.get(at, [])
        if len(fr) == 2:                                       # [yR | right] / [yR | rolled | right] / [yR]
            regs.append((int(fr[1]["y"]), {3: 2 * n, 2: int(p["rbuf"]) - int(fr[1]["y"]) + n}[mode], (r, "extra")))
        elif mode:
            regs.append((int(p["rbuf"]) - (n if mode == 2 else 0), mode * n, (r, "extra")))
    regs.sort()
    for (a, n, _), (b, _, _) in zip(regs, regs[1:]):
        assert a + n <= b, "mono regions overlap"
    assert regs[-1][0] + regs[-1][1] <= t.mono_n
    return regs


def _canon(t, offsets):
    regs = _stereo_regions(t)
    starts = np.array([a for a, _, _ in regs])
    out = []
    for v in np.asarray(offsets).tolist():
        i = int(np.searchsorted(starts, v, side="right")) - 1
        a, n, key = regs[i]
        assert 0 <= v - a < n
        out.append((key, v - a))
    return out


def test_merged_chunks_match_one_chunk():
    """Stereo-IR renders (even / odd n, stereo on / off, with a mono render between) packed as three chunks and merged
    describe the same batch as one chunk: every mono offset (FIR rows, post records, odd rolls, rotations) points at the
    same place of the same render, every FIR row at the same taps."""
    st, mono = _stereo_ir(0.2, 48000, 12), configs.synth_ir(0.1, 48000, 13)
    ps = [_ir_params(ir, space_ir_stereo=True, out_dur_s=d, stereo_on=so, seed=40 + i, env_a=0.1, env_d=0.0, env_r=0.0)
          for i, (ir, d, so) in enumerate([(st, 0.25, True), (st, 0.2500208, True), (mono, 0.25, True), (st, 0.25, False),
                                           (st, 0.2500208, True), (st, 0.001, True), (st, 0.25, True)])]
    rps = [P.plan_render(p) for p in ps]
    whole = T.pack_chunk(rps)
    merged = T.merge_chunks([T.pack_chunk(rps[:2]), T.pack_chunk(rps[2:5]), T.pack_chunk(rps[5:])])
    for a, b in ((whole.fir, merged.fir), (whole.post, merged.post), (whole.odd, merged.odd)):
        assert len(a) == len(b)
    for table, cols in (("fir", ("x", "y")), ("post", ("y", "rbuf")), ("odd", ("y_at", "scratch")), ("rot", ("src", "dst"))):
        for c in cols:
            a, b = getattr(whole, table)[c], getattr(merged, table)[c]
            if table == "post" and c == "rbuf":
                keep = whole.post["stereo_mode"] != 0
                a, b = a[keep], b[keep]
            assert _canon(whole, a) == _canon(merged, b), (table, c)
    for k in ("ir_len", "h_len", "out_n", "x_begin", "x_end", "tap_begin", "tap_end"):
        assert np.array_equal(whole.fir[k], merged.fir[k]), k
    for f, g in zip(whole.fir, merged.fir):
        assert np.array_equal(whole.irs[f["ir"]:f["ir"] + f["ir_len"]], merged.irs[g["ir"]:g["ir"] + g["ir_len"]])
    for k in ("n", "stereo_mode", "dl", "dr", "coef", "drive", "peak"):
        assert np.array_equal(whole.post[k], merged.post[k]), k
    assert whole.mono_n == merged.mono_n and whole.alg == merged.alg


def test_pooled_digest_matches_in_process():
    st = _stereo_ir(0.7, 48000, 8)
    for kw in (dict(), dict(space_ir_tap_cap=None, space_ir_max_samps=30000), dict(space_ir_tap_cap=10000)):
        p = _ir_params(st, space_ir_stereo=True, **kw)
        q = P._slim_params(p)
        assert q["_ir_audio"] is None and q["_ir_digest"]["taps_r"] is not None
        _same_tables(T.pack_chunk([P.plan_render(p)]), T.pack_chunk([P.plan_render(q)]))
    q = P._slim_params(_ir_params(st))
    assert q["_ir_digest"]["taps_r"] is None


def _mixed_batch():
    st, mono = _stereo_ir(1.0, 48000, 9), configs.synth_ir(0.5, 48000, 10)
    rows = [(st, True, None, 0.25, True, True), (st, True, 8192, 0.2500208, True, True), (mono, True, None, 0.25, True, True),
            (st, False, None, 0.25, True, True), (st, True, 30000, 0.25, False, True), (st, True, 8192, 0.001, True, True),
            (st, True, 8192, 0.25, True, False), (None, True, 8192, 0.25, True, True), (st, True, None, 0.3, False, False),
            (st, True, 8192, 0.25, True, True)]
    return [_ir_params(ir, seed=21 + i, space_ir_stereo=s, space_ir_tap_cap=cap, space_ir_max_samps=48000, out_dur_s=d,
                       stereo_on=so, er_cloud_on=er, env_a=0.1, env_d=0.0, env_r=0.0)
            for i, (ir, s, cap, d, so, er) in enumerate(rows)]


def test_native_planner_matches_python():
    subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "audio_suite_b200", "csrc"), "libms_hostplan.so"])
    hostplan._lib = None
    assert hostplan.lib() is not None
    ps = _mixed_batch()
    rps = [P.plan_render(p) for p in ps]
    want = T.pack_chunk(rps)
    _layout_checks(want, rps)
    for got in (hostplan.plan_chunk(ps), hostplan.plan_chunk(ps, threads=3), hostplan.plan_chunk([P._slim_params(p) for p in ps])):
        for name in want.__dataclass_fields__:
            a, b = getattr(want, name), getattr(got, name)
            if isinstance(a, np.ndarray) and a.dtype.names:
                for f in a.dtype.names:
                    if not f.startswith("_pad"):
                        assert np.array_equal(a[f], b[f]), (name, f)
            elif isinstance(a, np.ndarray):
                assert np.array_equal(a, b), name
            else:
                assert a == b, name


# ---- front end ------------------------------------------------------------------------------------------------------------
def _write_pcm16(path, a, sr=48000):
    a = np.asarray(a)
    ch = 1 if a.ndim == 1 else a.shape[1]
    data = np.round(a * 32767).astype("<i2").tobytes()
    fmt = struct.pack("<HHIIHH", 1, ch, sr, sr * ch * 2, ch * 2, 16)
    body = b"WAVE" + b"fmt " + struct.pack("<I", len(fmt)) + fmt + b"data" + struct.pack("<I", len(data)) + data
    path.write_bytes(b"RIFF" + struct.pack("<I", len(body)) + body)


def test_load_ir_wav_stereo(tmp_path):
    rng = np.random.default_rng(2)
    a = rng.uniform(-0.5, 0.5, (3000, 2))
    a[:, 1] *= 0.25
    a[100, 0] = 0.6
    for i, write in enumerate((lambda p: _write_pcm16(p, a), lambda p: frontend.write_wav_float32(p, a, 48000))):
        path = tmp_path / ("st%d.wav" % i)
        write(path)
        raw, _ = frontend.read_wav(str(path))
        got = frontend.load_ir_wav(str(path), stereo=True)
        assert got.dtype == np.float64 and got.shape == (3000, 2)
        assert np.max(np.abs(got)) == pytest.approx(0.9, abs=1e-15)
        assert np.array_equal(got, raw * (0.9 / np.max(np.abs(raw))))             # one gain for both channels
        assert np.array_equal(frontend.load_ir_wav(str(path)), frontend.load_ir_wav(str(path), stereo=False))
    path = tmp_path / "mono.wav"
    _write_pcm16(path, a[:, 0])
    assert np.array_equal(frontend.load_ir_wav(str(path), stereo=True), frontend.load_ir_wav(str(path)))
    path = tmp_path / "silent.wav"
    _write_pcm16(path, np.zeros((50, 2)))
    assert np.array_equal(frontend.load_ir_wav(str(path), stereo=True), np.zeros((50, 2)))


def test_preset_and_cache_keys(tmp_path):
    path = tmp_path / "hall.json"
    path.write_text(json.dumps({"space_ir_on": True, "space_ir_stereo": True}))
    assert frontend.load_preset(str(path))["space_ir_stereo"] is True
    assert "space_ir_stereo" not in frontend.load_preset({}) and "space_ir_stereo" not in configs.FACTORY_DEFAULTS
    ir = _stereo_ir(0.3, 48000, 10)
    keys = {engine._cache_key(_ir_params(ir, **kw), None, "f64") for kw in ({}, dict(space_ir_stereo=False),
                                                                             dict(space_ir_stereo=True))}
    assert len(keys) == 3
    sweep = frontend.batch_params(frontend.load_preset({"space_ir_stereo": True, "space_ir_tap_cap": None}), [1, 2], [1.0], [1.0])
    assert all(p["space_ir_stereo"] is True and p["space_ir_tap_cap"] is None for p in sweep)


# ---- stage: FIR pair units, post mode 3 ----------------------------------------------------------------------------------
def pair_cases(big=False, long_part=None):
    """fir_case dicts with an "ir_r": a second row equal on the input side whose output goes to a range of its own."""
    rng = np.random.default_rng(41 if big else 4)
    s = 3 if big else 1

    def with_r(cs, ir_r=None):
        ir_r = rng.standard_normal(len(cs["ir"])) * np.exp(-np.arange(len(cs["ir"])) / max(1.0, len(cs["ir"]) / 3.0)) if ir_r is None else ir_r
        return dict(cs, ir_r=ir_r)
    if long_part:
        k = 8192 // long_part + 1
        return [with_r(S.fir_case("long-pair-taps", rng, 20000 * s, k * long_part + 5, 30, 700, 0, x_begin=50, x_end=18000 * s)),
                with_r(S.fir_case("long-pair-no-taps", rng, 15000 * s, 9000, 0, 0, 0, x_begin=3, x_end=14000 * s)),
                S.fir_case("long-lone", rng, 12000, 8500, 10, 300, 0)]
    c = [with_r(S.fir_case("pair-taps-odd-blocks", rng, 150000 * s, 6000, 320, 2160, 65536, x_begin=300, x_end=140000 * s, dup=12)),
         with_r(S.fir_case("pair-no-taps", rng, 100000 * s, 8192, 0, 0, 65536, x_begin=5, x_end=99000 * s)),
         with_r(S.fir_case("pair-residue-0", rng, 140000, 4000, 64, 46 * 256, 65536, residue=0, x_begin=1000, x_end=120000)),
         S.fir_case("lone-B65536", rng, 130000, 6000, 100, 2160, 65536, x_begin=40, x_end=125000),
         with_r(S.fir_case("pair-B8192", rng, 20000 * s, 1000, 40, 2000, 8192, x_begin=300, x_end=15000 * s, dup=3)),
         with_r(S.fir_case("pair-live-end-in-block-a", rng, 230000, 6000, 160, 2160, 65536, x_begin=70000, x_end=100000, dup=3))]
    c[2]["ir_r"] = c[2]["ir"].copy()                             # equal channels at two pool offsets
    return c


def fir_pair_run(dev, precision, cases, runs=1):
    """All rows as one ms_fir_create: a case's right row directly after its left row, same x, its own output range.
    Returns (outputs per run, the row cases -- right rows as cases with ir = ir_r --, their output starts, launch log)."""
    import ctypes as C
    from audio_suite_b200 import _abi
    api, real = _abi.Api(dev.lib, precision), S._real(precision)
    recs, irs, offs, gains, rows, starts = [], [], [], [], [], []
    ir_n, t_n, at = 0, 0, S.GAP
    x_parts = []
    for cs in cases:
        x_at = at
        at += len(cs["x"]) + S.GAP
        x_parts.append((x_at, cs["x"]))
        for side in ("ir", "ir_r"):
            if side not in cs:
                continue
            ir = cs[side]
            r = _abi.FirRender()
            r.ir, r.ir_len = ir_n, len(ir)
            r.h_len = len(ir) + (int(np.max(cs["offs"])) if len(cs["offs"]) else 0)
            r.tap_begin, r.tap_end = t_n, t_n + len(cs["offs"])
            y_at = x_at
            if side == "ir_r":
                y_at = at
                at += len(cs["x"]) + S.GAP
            r.x, r.y, r.out_n, r.x_begin, r.x_end = x_at, y_at, len(cs["x"]), cs["x_begin"], cs["x_end"]
            recs.append(r)
            irs.append(ir)
            ir_n += len(ir)
            rows.append(dict(cs, ir=ir, name=cs["name"] + ("-R" if side == "ir_r" else "")))
            starts.append(y_at)
        offs.append(cs["offs"])
        gains.append(cs["gains"])
        t_n += len(cs["offs"])
    x = np.full(at, S.X_SENTINEL)
    for s, v in x_parts:
        x[s:s + len(v)] = v
    arr = (_abi.FirRender * len(recs))(*recs)
    need = api.ms_fir_workspace_bytes(C.addressof(arr), len(recs))
    assert need > 0, dev.lib.ms_last_error()
    ws = dev.empty(need, np.uint8)
    d_ir = dev.upload(np.concatenate(irs).astype(real))
    d_off = dev.upload(np.concatenate(offs).astype(np.int32) if t_n else np.zeros(1, np.int32))
    d_gain = dev.upload((np.concatenate(gains) if t_n else np.zeros(1)).astype(real))
    d_x = dev.upload(x.astype(real))
    d_y = dev.upload(np.full(at, np.nan, real))
    h = C.c_void_p()
    outs = []
    with S.LaunchLog(dev) as log:
        rc = api.ms_fir_create(C.addressof(arr), len(recs), dev.ptr(d_ir), dev.ptr(d_off), dev.ptr(d_gain), dev.ptr(d_x),
                               dev.ptr(d_y), dev.ptr(ws), need, dev.stream_ptr(), C.byref(h))
        assert rc == 0, dev.lib.ms_last_error()
        try:
            for _ in range(runs):
                assert api.ms_fir_run(h, dev.stream_ptr()) == 0, dev.lib.ms_last_error()
                outs.append(S._fetch(dev, d_y, real, at).astype(np.float64))
        finally:
            api.ms_fir_destroy(h)
    return outs, rows, starts, log


def check_pairs(dev, precision, cases, fft=False):
    """The batch against float64 convolution per channel, two runs bitwise equal, every row bitwise equal to the same row
    run alone; the pair kernel ran exactly when the block class calls for it.  Returns {"errors", "kernels"}."""
    outs, rows, starts, log = fir_pair_run(dev, precision, cases, runs=2)
    assert np.array_equal(outs[0], outs[1], equal_nan=True), "second ms_fir_run on one handle differs"
    ref = S.fir_reference_fft if fft else S.fir_reference
    refs = [ref(S._as_ref(cs["ir"], precision), cs["offs"], S._as_ref(cs["gains"], precision), S._as_ref(cs["x"], precision),
                cs["x_begin"], cs["x_end"]) for cs in rows]
    errors = S.check_fir_outputs(precision, rows, outs[0], starts, refs=refs, label="pairs")
    alone, a_starts, _ = S.fir_run(dev, precision, [dict(cs, share=None) for cs in rows])
    for cs, s, sa in zip(rows, starts, a_starts):
        n = len(cs["x"])
        assert np.array_equal(outs[0][s:s + n], alone[0][sa:sa + n]), (precision, cs["name"], "differs from the lone row")
    fused_pair = any("ir_r" in cs and cs["B"] == 65536 for cs in cases)
    assert ("FirP2PairK" in log.base()) == fused_pair, sorted(log.base())
    return {"errors": errors, "kernels": sorted(set(log.names))}


@pytest.mark.parametrize("precision", ["f64", "f32"])
def test_fir_pairs_emulated(emul, precision):
    res = check_pairs(emul, precision, pair_cases())
    print("FIR pairs %s: worst %.2e" % (precision, max(res["errors"].values())))


def _workspace(dev, precision, cases):
    """ms_fir_workspace_bytes of the rows fir_pair_run would build for `cases`."""
    import ctypes as C
    from audio_suite_b200 import _abi
    recs = []
    for cs in cases:
        for side in ("ir", "ir_r"):
            if side in cs:
                r = _abi.FirRender()
                r.ir, r.ir_len = 0, len(cs[side])
                r.h_len = len(cs[side]) + (int(np.max(cs["offs"])) if len(cs["offs"]) else 0)
                r.tap_begin, r.tap_end = 0, len(cs["offs"])
                r.x, r.y, r.out_n, r.x_begin, r.x_end = 0, 0 if side == "ir" else len(cs["x"]), len(cs["x"]), cs["x_begin"], cs["x_end"]
                recs.append(r)
    arr = (_abi.FirRender * len(recs))(*recs)
    return _abi.Api(dev.lib, precision).ms_fir_workspace_bytes(C.addressof(arr), len(recs))


@pytest.mark.parametrize("precision", ["f64", "f32"])
def test_fir_long_pairs_emulated(emul, precision, monkeypatch):
    """Long-route pairs share the reflection pass and the input spectra Z: each channel bitwise equal to its lone row,
    and the pair's workspace is one Z and one reflection buffer smaller than two lone rows' (the right channel's own
    inverse work area is as large as a Z)."""
    monkeypatch.setenv("MS_FIR_PART", "64")
    cases = pair_cases(long_part=64)
    res = check_pairs(emul, precision, cases)
    assert "FirLongMacK" in {k.split("<")[0] for k in res["kernels"]}
    cpx = 2 * np.dtype(S._real(precision)).itemsize
    for cs in cases[:2]:
        n = len(cs["x"])
        J = -(-n // 64); Jh = (J + 1) // 2; K = -(-min(len(cs["ir"]), n - cs["x_begin"]) // 64); head = min(K - 1, Jh)
        ent = (Jh + head) * 128 * cpx                               # one row's Z (and its Y, and a right channel's W)
        left = {k: v for k, v in cs.items() if k != "ir_r"}
        pair = _workspace(emul, precision, [cs])
        two = _workspace(emul, precision, [left]) + _workspace(emul, precision, [dict(left, ir=cs["ir_r"])])
        assert pair < two, (cs["name"], pair, two)
        refl = n * np.dtype(S._real(precision)).itemsize if len(cs["offs"]) else 0
        assert two - pair >= refl - 4096 and pair - _workspace(emul, precision, [left]) >= 2 * ent, cs["name"]


def test_fir_pairs_thread_schedule():
    """Pairs under MS_EMUL_SHUFFLE (fibres of a block in a fresh order between barriers): bitwise equal results."""
    code = ("import sys, hashlib; sys.path[:0] = [%r, %r, %r]\n"
            "from emul_device import EmulDevice; import test_stereo_ir as M\n"
            "dev = EmulDevice(); h = hashlib.sha256()\n"
            "for prec in ('f64', 'f32'):\n"
            "    outs, _, _, log = M.fir_pair_run(dev, prec, M.pair_cases()[:3]); h.update(outs[0].tobytes())\n"
            "    assert 'FirP2PairK' in log.base()\n"
            "print(h.hexdigest())\n") % (ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "tests", "host_emul"))
    digests = []
    for seed in (None, "1", "7"):
        env = dict(os.environ)
        env.pop("MS_EMUL_SHUFFLE", None)
        if seed:
            env["MS_EMUL_SHUFFLE"] = seed
        p = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, cwd=ROOT)
        assert p.returncode == 0, p.stderr[-4000:]
        digests.append(p.stdout.strip().splitlines()[-1])
    assert len(set(digests)) == 1, digests


def check_post_mode3(dev, precision, big=False):
    """ms_post mode 3 records (right channel = Bessel FIR of the n samples before rbuf) beside modes 1 and 2, with
    sentinels: the right channel left at rbuf against both float64 forms, the output against the post chain."""
    import ctypes as C
    from audio_suite_b200 import _abi
    api, real = _abi.Api(dev.lib, precision), S._real(precision)
    rng = np.random.default_rng(17)
    s = 40 if big else 1
    cases = [(64, 3, 5, 9, 0.63, 1.0, 1.0), (66, 3, 65, 63, 0.9, 2.0, 3.0), (3000, 3, 2999, 2998, 0.9, 1.3, 0.8),
             (50000 * s, 3, 36, 50, 0.81, 1.0, 179.0), (4000, 3, 17, 21, 0.27, 0.0, 2.5), (2048, 1, 7, 9, 0.5, 1.0, 1.0),
             (1025, 2, 0, 0, 0.0, 1.0, 1.0)]
    recs, layout, mono_n, frames = [], [], S.GAP, S.GAP
    for n, mode, dl, dr, theta, drive, scale in cases:
        y_at = mono_n
        mono_n += n + S.GAP
        src_at = mono_n                                          # mode 3: [yR | right]; mode 2: [right]
        mono_n += (2 * n if mode == 3 else n) + S.GAP
        rbuf = src_at + n if mode == 3 else src_at
        coef = T.bessel_coeffs(theta) if mode in (1, 3) else np.zeros(2 * _abi.POST_K + 1)
        r = np.zeros(1, np.dtype(_abi.PostRender))
        r[0] = (y_at, frames, rbuf, n, mode, dl, dr, drive, 1.0 / np.tanh(drive) if drive > 0 else 1.0, 0.98, coef)
        recs.append(r[0])
        layout.append((y_at, src_at, rbuf, frames, rng.standard_normal(n) * scale, rng.standard_normal(n) * scale * 0.6))
        frames += n + S.GAP
    mono = np.full(mono_n, S.X_SENTINEL)
    for y_at, src_at, _, _, y, y2 in layout:
        mono[y_at:y_at + len(y)] = y
        mono[src_at:src_at + len(y2)] = y2
    d_rec = dev.upload(np.array(recs, dtype=np.dtype(_abi.PostRender)))
    d_mono = dev.upload(mono.astype(real))
    maxbits = dev.zeros(len(recs), np.uint64)
    out = dev.upload(np.full(2 * frames, np.nan, np.float32))
    with S.LaunchLog(dev):
        assert api.ms_post(dev.ptr(d_rec), len(recs), max(c[0] for c in cases), dev.ptr(d_mono), dev.ptr(maxbits), dev.ptr(out),
                           dev.stream_ptr()) == 0, dev.lib.ms_last_error()
    o = S._fetch(dev, out, np.float32, 2 * frames).reshape(-1, 2)
    m = S._fetch(dev, d_mono, real, mono_n).astype(np.float64)
    mono_q = S._as_ref(mono, precision)
    errors, gaps = {}, np.ones(len(o), bool)
    for (n, mode, dl, dr, theta, drive, scale), (y_at, src_at, rbuf, fr, _, _) in zip(cases, layout):
        gaps[fr:fr + n] = False
        yq, y2q = mono_q[y_at:y_at + n], mono_q[src_at:src_at + n]
        tag = "n=%d mode=%d" % (n, mode)
        got = o[fr:fr + n].astype(np.float64)
        src = {1: yq, 2: None, 3: y2q}[mode]
        if mode == 2:
            right = y2q
        else:
            r_dev = m[rbuf:rbuf + n]
            r_fft = S.rotate_right(src, dr, theta)
            e_r = max(float(np.max(np.abs(r_dev - r_fft))), float(np.max(np.abs(r_dev - S.bessel_right(src, dr, T.bessel_coeffs(theta)))))) \
                / float(np.max(np.abs(src)))
            errors[tag + " right"] = e_r
            assert e_r < S.POST_R_TOL[precision], (tag, e_r)
            right = r_fft
        if mode == 3:                                            # the input of the right channel is left as it was
            assert np.array_equal(m[src_at:src_at + n], mono_q[src_at:src_at + n]), tag
        want = O.peak_normalize(O.soft_saturate(np.column_stack([np.roll(yq, dl), right]), drive), 0.98)
        e = float(np.max(np.abs(got - want)))
        errors[tag] = e
        mx = float(max(np.max(np.abs(yq)), np.max(np.abs(right))))
        slope = 0.98 * (drive / np.tanh(drive * mx) if drive > 0 else 1.0 / mx)
        tol = S.POST_OUT_TOL[precision] + (S.POST_R_TOL[precision] * mx * slope if mode != 2 else 0.0)
        assert e < tol, (tag, precision, e, tol)
    assert np.all(np.isnan(o[gaps])), "write outside every render's frames"
    return errors


@pytest.mark.parametrize("precision", ["f64", "f32"])
def test_post_mode3_emulated(emul, precision):
    errs = check_post_mode3(emul, precision)
    print("post mode 3 %s: worst right %.2e" % (precision, max(v for k, v in errs.items() if "right" in k)))


# ---- end to end -----------------------------------------------------------------------------------------------------------
def stereo_reference(p):
    """The float64 render of a space_ir_stereo render from the oracle's stages: its mono mix after the reflection cloud,
    each channel of the IR (slice, cut) convolved with it, the stereo diffusion with the right channel taken from yR."""
    taps = {}
    O.render(dict(p, space_ir_on=False), taps=taps)
    u = taps["after_er"]
    n = len(u)
    h = np.asarray(p["_ir_audio"])[:int(p["space_ir_max_samps"])]
    cap = p.get("space_ir_tap_cap", P.IR_TAP_CAP)
    h = (h if cap is None else h[:cap]).astype(np.float64)
    y_l, y_r = np.convolve(u, h[:, 0])[:n], np.convolve(u, h[:, 1])[:n]
    if p["stereo_on"] and n >= 64:
        dl, dr, w = O.stereo_shifts(int(p["base_sr"]), float(p["stereo_width"]))
        st = np.column_stack([np.roll(y_l, dl), S.rotate_right(y_r, dr, w * 0.9)])
    else:
        st = np.column_stack([y_l, y_r])
    return O.peak_normalize(O.soft_saturate(st, float(p["sat_drive"])), float(p["peak"]))


def test_render_stereo_emulated(emul):
    st = _stereo_ir(0.15, 48000, 13)
    for kw in (dict(), dict(out_dur_s=0.2500208), dict(stereo_on=False), dict(er_cloud_on=False)):
        p = _ir_params(st, space_ir_stereo=True, **kw)
        out, _ = engine.render(p, device=emul, precision="f64")
        err = float(np.max(np.abs(out - stereo_reference(p))))
        assert err < 1e-5, (kw, err)
    h = st[:, 0]
    p = _ir_params(np.column_stack([h, h]), space_ir_stereo=True)
    a, _ = engine.render(p, device=emul, precision="f64")
    b, _ = engine.render(_ir_params(h), device=emul, precision="f64")
    assert np.array_equal(a, b)


# ---- GPU ------------------------------------------------------------------------------------------------------------------
def _stereo_c5(i, **kw):
    p = configs.c5_params(i)
    return dict(p, _ir_audio=_c5_ir(), space_ir_stereo=True, **kw)


@functools.lru_cache(maxsize=None)
def _c5_ir():
    return _stereo_ir(1.0, 48000, 77)


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["f64", "f32"])
def test_identical_channels_equal_mono_gpu(cuda_dev, precision):
    """column_stack([h, h]) under space_ir_stereo renders exactly what h renders in mono."""
    for p in (configs.canonical("C3"), dict(configs.c5_params(7), out_dur_s=1.5)):
        ir = np.asarray(p["_ir_audio"])
        h = ir.astype(np.float64).mean(axis=1) if ir.ndim > 1 else ir.astype(np.float64)
        a, _ = engine.render(dict(p, _ir_audio=np.column_stack([h, h]), space_ir_stereo=True), device=cuda_dev, precision=precision, cache=False)
        b, _ = engine.render(dict(p, _ir_audio=h), device=cuda_dev, precision=precision, cache=False)
        assert np.array_equal(a, b), p.get("seed")


def check_in_situ_stereo(dev, params_list, precision="f64", sample=None):
    """FIR rows of each render (left and right) against float64 convolution of the device's own plane A, and the output
    against the post chain of the device's own FIR outputs.  `sample`: compare the FIR at that many seeded positions
    (direct sums) instead of whole convolutions."""
    from scipy.signal import oaconvolve
    br = engine.BatchRenderer(params_list, device=dev, precision=precision)
    t = br.tables
    snap = {}

    def mark(name):
        if name == "overlap_add":
            snap["A"] = S._fetch(dev, br.mono, br.real, t.mono_n).astype(np.float64)
        elif name == "fir_overlap_save":
            snap["B"] = S._fetch(dev, br.mono, br.real, t.mono_n).astype(np.float64)
    errs = []
    try:
        br.run(mark=mark)
        dev.synchronize()
        rows = {}
        for f in t.fir:
            rows.setdefault(int(f["x"]), []).append(f)
        for r, p in enumerate(params_list):
            rp = P.plan_render(p)
            at, n = int(t.ola_r[r]["out"]), int(t.ola_r[r]["out_n"])
            u = snap["A"][at:at + n]
            if p["er_cloud_on"]:
                u = O.reflection_cloud(u, int(p["base_sr"]), int(p["er_taps"]), float(p["er_max_ms"]), int(p["seed"]))
            fr = rows[at]
            assert len(fr) == (2 if rp.ir_r is not None else 1), r
            ys = []
            for f, h in zip(fr, (rp.ir, rp.ir_r)):
                y = snap["B"][int(f["y"]):int(f["y"]) + n]
                hq = S._as_ref(h, precision)
                if sample:
                    rng = np.random.default_rng(r)
                    pos = np.unique(np.concatenate([rng.integers(0, n, sample), [n - 1]]))
                    want = np.array([float(np.dot(hq[:i - max(0, i - hq.size + 1) + 1], u[max(0, i - hq.size + 1):i + 1][::-1]))
                                     for i in pos.tolist()])
                    e = float(np.max(np.abs(y[pos] - want))) / max(1e-300, float(np.max(np.abs(y))))
                else:
                    e = S._rel(y, oaconvolve(u, hq)[:n])
                assert e < S.FIR_TOL[precision], (r, "FIR", e)
                ys.append(y)
            y_l = ys[0]
            y_r = ys[1] if len(ys) > 1 else y_l
            if rp.stereo_on:
                st = np.column_stack([np.roll(y_l, rp.stereo_dl), S.rotate_right(y_r, rp.stereo_dr, rp.stereo_theta)])
            else:
                st = np.column_stack([y_l, y_r])
            want = O.peak_normalize(O.soft_saturate(st, float(p["sat_drive"])), float(p["peak"]))
            e_post = float(np.max(np.abs(br.output(r).astype(np.float64) - want)))
            mx = float(np.max(np.abs(st)))
            slope = float(p["peak"]) * (float(p["sat_drive"]) / np.tanh(float(p["sat_drive"]) * mx) if p["sat_drive"] > 0 else 1.0 / mx)
            tol = S.POST_OUT_TOL[precision] + S.POST_R_TOL[precision] * mx * slope
            assert e_post < tol, (r, "post", e_post, tol)
            errs.append(dict(n=n, post=e_post))
        return errs
    finally:
        br.close()


@pytest.mark.gpu
def test_in_situ_stereo_gpu(cuda_dev):
    c3 = dict(configs.canonical("C3"), space_ir_stereo=True)
    c5 = [_stereo_c5(i, out_dur_s=2.0 + 0.0000208 * (i % 2)) for i in range(6)]
    check_in_situ_stereo(cuda_dev, [c3] + c5, "f64")
    check_in_situ_stereo(cuda_dev, c5[:3], "f32")
    c4 = dict(configs.canonical("C4"), space_ir_stereo=True)
    check_in_situ_stereo(cuda_dev, [c4], "f64", sample=48)
    check_in_situ_stereo(cuda_dev, [dict(c4, space_ir_tap_cap=None)], "f64", sample=48)


@pytest.mark.gpu
def test_mixed_batch_gpu(cuda_dev):
    mono = [configs.c5_params(i) for i in range(8)]
    mixed = [_stereo_c5(i) if i % 2 else p for i, p in enumerate(mono)]
    a = [np.array(x) for x in engine.render_batch(mixed, device=cuda_dev)]
    b = [np.array(x) for x in engine.render_batch(mono[0::2], device=cuda_dev)]
    for x, y in zip(a[0::2], b):
        assert np.array_equal(x, y)
    c = [np.array(x) for x in engine.render_batch(mixed[1::2], device=cuda_dev)]
    for x, y in zip(a[1::2], c):
        assert np.array_equal(x, y)
    for i in (1, 3):                                             # render_batch (native planner, streamed) == render()
        d, _ = engine.render(mixed[i], device=cuda_dev, cache=False)
        assert np.array_equal(a[i], d.astype(a[i].dtype)) or np.array_equal(a[i].astype(np.float64), d), i


@pytest.mark.gpu
def test_fir_pairs_gpu(cuda_dev):
    for precision in ("f64", "f32"):
        r = check_pairs(cuda_dev, precision, pair_cases(big=True), fft=True)
        print("FIR pairs %s: worst %.2e" % (precision, max(r["errors"].values())))


@pytest.mark.gpu
def test_post_mode3_gpu(cuda_dev):
    for precision in ("f64", "f32"):
        check_post_mode3(cuda_dev, precision, big=True)


@pytest.mark.gpu
def test_graph_replay_stereo(cuda_dev):
    engine.clear_render_cache()
    p = _stereo_c5(5)
    a, _ = engine.render(p)                                     # eager
    b, _ = engine.render(p)                                     # captured and replayed
    c, _ = engine.render(p)                                     # replayed
    engine.clear_render_cache()
    assert np.array_equal(a, b) and np.array_equal(a, c)
    d, _ = engine.render(dict(p, space_ir_stereo=False), cache=False)
    assert not np.array_equal(a, d)
