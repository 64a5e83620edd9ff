"""Export sample rate (EXTENSION; the reference delivers every render at base_sr): the optional key `export_sr` through both
planners, the tables, the post stage's resampling pass (ms_post_export) and the engine, against scipy.signal.resample_poly.

A render with export_sr runs exactly as without it; each channel of its clipped and normalised signal x (before the
float32 rounding) is then resample_poly(x, up, down) with up / down = export_sr / base_sr in lowest terms.

The CPU tests run the stage on the block emulator; the GPU tests repeat them on real renders."""
import hashlib
import math
import os
import subprocess
import sys

import numpy as np
import pytest
import scipy.signal as ss

import stage_checks as S
from audio_suite_b200 import _abi, configs, decimate, engine, frontend, hostplan, plan as P, tables as T
from oracle import microsound_np as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RATIOS = ((1, 2), (2, 1), (147, 160), (160, 147), (147, 320), (640, 147), (1, 6))


def _ratio(base, ex):
    g = math.gcd(base, ex)
    return ex // g, base // g


def _short(**kw):
    base = dict(gen_mode="Resonant strike", micro_ms=3.0, time_unfold=20.0, out_dur_s=0.06, event_process="Poisson",
                grains_per_sec=60.0, bp_density="", stereo_on=True, er_cloud_on=True, er_taps=20, sat_drive=1.5)
    base.update(kw)
    return configs.with_defaults(base)


def _same_tables(a, b):
    for name in a.__dataclass_fields__:
        x, y = getattr(a, name), getattr(b, name)
        if isinstance(x, np.ndarray):
            assert x.dtype == y.dtype and x.shape == y.shape, name
            for f in (x.dtype.names or (None,)):
                if f is None or not f.startswith("_pad"):
                    assert np.array_equal(T.column(x, f), T.column(y, f)), (name, f)
        else:
            assert x == y, name


# ---- validation, identity, the filter ------------------------------------------------------------------------------------
@pytest.mark.parametrize("value", [True, False, np.bool_(True), 0, -44100, 44100.0, "44100", np.float64(44100.0)])
def test_invalid_values_raise(value, emul):
    p = _short(export_sr=value)
    with pytest.raises(ValueError, match="export_sr"):
        P.plan_render(p)
    with pytest.raises(ValueError, match="export_sr"):
        engine.render(p, device=emul, cache=False)
    with pytest.raises(ValueError, match="export_sr"):
        hostplan.plan_chunk([p])


@pytest.mark.parametrize("base,ex", [(32000, 11025), (96000, 11025), (192000, 11025), (192000, 22050), (48000, 47999)])
def test_over_limit_ratios_raise(base, ex):
    with pytest.raises(ValueError, match="at most 640"):
        P.plan_render(_short(base_sr=base, export_sr=ex))


def test_standard_rates_within_limit():
    rates = (8000, 11025, 16000, 22050, 32000, 44100, 48000, 88200, 96000, 176400, 192000)
    over = {(b, e) for b in rates for e in rates if max(_ratio(b, e)) > P.EXPORT_RATIO_LIMIT}
    assert {frozenset(x) for x in over} == {frozenset(x) for x in ((11025, 32000), (11025, 96000), (11025, 192000), (22050, 192000))}
    assert max(2 * 10 * max(_ratio(b, e)) + 1 for b in rates for e in rates if (b, e) not in over) == 12801
    assert P.export_ratio(_short(export_sr=np.int64(44100))) == (147, 160)


def test_identity_tables_and_output(emul):
    """Absent, None and export_sr == base_sr (int or numpy int): identical tables from both planners, bitwise output."""
    ps = [_short(), _short(export_sr=None), _short(export_sr=48000), _short(export_sr=np.int32(48000))]
    want = T.pack_chunk([P.plan_render(ps[0])])
    assert len(want.export) == 0 and want.bank.size == 0
    for p in ps:
        _same_tables(T.pack_chunk([P.plan_render(p)]), want)
        _same_tables(hostplan.plan_chunk([p]), hostplan.plan_chunk([ps[0]]))
    outs = [engine.render(p, device=emul, precision="f64", cache=False) for p in ps]
    for a, m in outs:
        assert np.array_equal(a, outs[0][0]) and m["out_sr"] == 48000


def test_design_matches_scipy():
    for up, down in RATIOS + ((1, 3), (3, 1)):
        q = max(up, down)
        want = up * ss.firwin(2 * 10 * q + 1, 1.0 / q, window=("kaiser", 5.0))
        assert np.max(np.abs(decimate.resample_taps(up, down) - want)) <= 1e-15, (up, down)
    for q in (2, 3, 7):                                 # the decimator's design is the up = 1 case, value for value
        half = 10 * q
        m = np.arange(-half, half + 1, dtype=np.float64)
        h = (1.0 / q) * np.sinc(m / q) * np.kaiser(2 * half + 1, 5.0)
        assert np.array_equal(decimate.design_taps(q), h / np.sum(h))


def _poly_reference(x, up, down):
    """The formula of include/microsound_b200.h in a plain loop over the polyphase bank."""
    half, taps, bank = decimate.polyphase_bank(up, down)
    a, n = half // up, len(x)
    out = np.zeros(-(-n * up // down))
    for m in range(out.size):
        q, p = divmod(m * down, up)
        for s in range(-a, taps - a):
            if 0 <= q + s < n:
                out[m] += x[q + s] * bank[p, s + a]
    return out


def test_formula_matches_resample_poly():
    rng = np.random.default_rng(3)
    for up, down in RATIOS + ((1, 3),):
        x = rng.standard_normal(157)
        want = ss.resample_poly(x, up, down)
        got = _poly_reference(x, up, down)
        assert got.shape == want.shape
        assert np.max(np.abs(got - want)) / np.max(np.abs(want)) <= 1e-15, (up, down)


# ---- planners -------------------------------------------------------------------------------------------------------------
def _sweep(k, seed):
    rng = np.random.default_rng(seed)
    rates = (None, 44100, 16000, 96000, 22050, 8000, 48000, np.int64(32000))
    ps = []
    for i in range(k):
        p = dict(configs.c5_params(int(rng.integers(0, 4096))), out_dur_s=float(rng.uniform(0.05, 0.3)))
        p["export_sr"] = rates[int(rng.integers(0, len(rates)))]
        p["stereo_on"] = bool(rng.integers(0, 2))
        ps.append(p)
    return ps


def _check_layout(t, rps, one_chunk=True):
    at = 0
    for r, rp in enumerate(rps):
        n_x = P.export_frames(rp.out_n, rp.export)
        assert t.out_at[r] == at and t.out_n[r] == n_x and t.post[r]["out"] == at and t.post[r]["n"] == rp.out_n
        at += n_x
    assert t.frames == at
    assert t.export_of.tolist() == [r for r, rp in enumerate(rps) if rp.export is not None]
    for e, r in zip(t.export, t.export_of.tolist()):
        up, down = rps[r].export
        half, taps, bank = decimate.polyphase_bank(up, down)
        assert e["out"] == t.out_at[r] and e["out_end"] - e["out"] == t.out_n[r]
        assert e["rate"].tolist() == [up, down, half, taps]
        assert np.array_equal(t.bank[e["bank"]:e["bank_end"]], bank.reshape(-1))
    if one_chunk:                                       # one bank per ratio (merged chunks keep one per ratio and chunk)
        assert len({(int(e["bank"]), int(e["bank_end"])) for e in t.export}) == len({rps[r].export for r in t.export_of.tolist()})


@pytest.mark.parametrize("seed", [1, 2])
def test_native_planner_matches_python(seed):
    subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "audio_suite_b200", "csrc"), "libms_hostplan.so"])
    hostplan._lib = None
    assert hostplan.lib() is not None
    ps = _sweep(40, seed)
    rps = [P.plan_render(p) for p in ps]
    want = T.pack_chunk(rps)
    _check_layout(want, rps)
    plain = T.pack_chunk([P.plan_render(dict(p, export_sr=None)) for p in ps])
    for name in ("mono_n", "pool_n", "sy1", "ola_r", "fir", "odd", "rot", "y_at", "srs"):      # only the output side moves
        a, b = getattr(want, name), getattr(plain, name)
        assert (np.array_equal(a, b) if isinstance(a, np.ndarray) else a == b), name
    keep = [f for f in want.post.dtype.names if f != "out"]
    assert np.array_equal(want.post[keep], plain.post[keep])
    for got in (hostplan.plan_chunk(ps), hostplan.plan_chunk(ps, threads=3), hostplan.plan_chunk([P._slim_params(p) for p in ps])):
        _same_tables(got, want)


def test_merged_chunks_match_one_chunk():
    ps = _sweep(30, 5)
    rps = [P.plan_render(p) for p in ps]
    whole = T.pack_chunk(rps)
    parts = [T.pack_chunk(rps[a:b]) for a, b in ((0, 7), (7, 8), (8, 30))]
    merged = T.merge_chunks(parts)
    _check_layout(merged, rps, one_chunk=False)
    for name in ("out_at", "out_n", "export_of"):
        assert np.array_equal(getattr(merged, name), getattr(whole, name)), name
    frames = ["out", "n", "stereo_mode", "dl", "dr"]            # (y and rbuf: the mono planes are laid out per chunk)
    assert np.array_equal(merged.post[frames], whole.post[frames])
    keep = ["out", "out_end", "rate"]
    assert np.array_equal(merged.export[keep], whole.export[keep]) and merged.frames == whole.frames


# ---- the stage on the block emulator ---------------------------------------------------------------------------------------
def export_cases():
    """(n, stereo mode, dl, dr, theta, drive, scale, (up, down)): modes 0-3, drive 0 and > 0, n = 1, 63, 64, odd, and n not a
    multiple of the tile, every ratio at least once."""
    rs = RATIOS
    return [(1, 0, 0, 0, 0.0, 1.0, 1.0, rs[5]), (63, 0, 0, 0, 0.0, 0.0, 2.0, rs[0]), (64, 1, 5, 9, 0.63, 1.0, 1.0, rs[1]),
            (1001, 2, 17, 0, 0.0, 1.3, 0.8, rs[2]), (3000, 1, 29, 41, 0.9, 2.0, 3.0, rs[3]), (2500, 3, 7, 11, 0.45, 0.0, 1.7, rs[4]),
            (4097, 2, 0, 0, 0.0, 0.0, 1.0, rs[6]), (2050, 3, 2049, 2048, 0.81, 1.0, 5.0, rs[5]), (999, 0, 0, 0, 0.0, 2.5, 0.3, rs[2]),
            (6144, 1, 3, 3, 0.2, 0.7, 1.0, rs[6])]


def export_run(dev, precision, cases):
    """ms_post_export on hand-built records with sentinels around every range.  Returns (outputs, device mono, layout, log)."""
    api, real = _abi.Api(dev.lib, precision), S._real(precision)
    rng = np.random.default_rng(11)
    recs, exps, layout, banks, bank_of = [], [], [], [], {}
    mono_n, frames, n_bank = S.GAP, S.GAP, S.GAP
    for n, mode, dl, dr, theta, drive, scale, (up, down) in cases:
        y_at = mono_n
        mono_n += n + S.GAP
        src_at = mono_n                                           # mode 3: [yR | right]; modes 1, 2: [right]
        mono_n += (2 * n if mode == 3 else n) + S.GAP
        rbuf = src_at + n if mode == 3 else src_at
        coef = T.bessel_coeffs(theta) if mode in (1, 3) else np.zeros(2 * _abi.POST_K + 1)
        r = np.zeros(1, np.dtype(_abi.PostRender))
        r[0] = (y_at, frames, rbuf if mode else 0, n, mode, dl, dr, drive, 1.0 / np.tanh(drive) if drive > 0 else 1.0, 0.98, coef)
        recs.append(r[0])
        half, taps, bk = decimate.polyphase_bank(up, down)
        if (up, down) not in bank_of:
            bank_of[up, down] = n_bank
            banks.append((n_bank, bk.reshape(-1)))
            n_bank += bk.size + S.GAP
        n_x = -(-n * up // down)
        e = np.zeros(1, np.dtype(_abi.ExportRender))
        e[0] = (frames, frames + n_x, bank_of[up, down], bank_of[up, down] + bk.size, (up, down, half, taps))
        exps.append(e[0])
        layout.append((y_at, src_at, rbuf, frames, n_x, rng.standard_normal(n) * scale, rng.standard_normal(n) * scale * 0.6))
        frames += n_x + S.GAP
    mono = np.full(mono_n, S.X_SENTINEL)
    for y_at, src_at, _, _, _, y, y2 in layout:
        mono[y_at:y_at + len(y)] = y
        mono[src_at:src_at + len(y2)] = y2
    bank = np.full(n_bank, 1e3)
    for at, bk in banks:
        bank[at:at + bk.size] = bk
    d_rec, d_exp = dev.upload(np.array(recs, np.dtype(_abi.PostRender))), dev.upload(np.array(exps, np.dtype(_abi.ExportRender)))
    d_mono, d_bank = dev.upload(mono.astype(real)), dev.upload(bank.astype(real))
    maxbits = dev.zeros(len(recs), np.uint64)
    out = dev.upload(np.full(2 * frames, np.nan, np.float32))
    with S.LaunchLog(dev) as log:
        rc = api.ms_post_export(dev.ptr(d_rec), dev.ptr(d_exp), len(recs), max(c[0] for c in cases), max(l[4] for l in layout),
                                dev.ptr(d_mono), dev.ptr(maxbits), dev.ptr(d_bank), dev.ptr(out), dev.stream_ptr())
        assert rc == 0, dev.lib.ms_last_error()
    o = S._fetch(dev, out, np.float32, 2 * frames).reshape(-1, 2)
    m = S._fetch(dev, d_mono, real, mono_n).astype(np.float64)
    return o, m, mono, layout, log


def check_export(dev, precision, cases):
    o, m, mono, layout, log = export_run(dev, precision, cases)
    assert log.base() >= {"PostMaxK", "PostExportK"} and "PostWriteK" not in log.base(), log.names
    mono_q = S._as_ref(mono, precision)
    gaps, worst = np.ones(len(o), bool), 0.0
    for (n, mode, dl, dr, theta, drive, scale, (up, down)), (y_at, src_at, rbuf, fr, n_x, _, _) in zip(cases, layout):
        gaps[fr:fr + n_x] = False
        yq = mono_q[y_at:y_at + n]
        # the right channel as the max pass left it (checked against float64 in the ms_post tests), else the input
        right = {0: yq, 2: mono_q[src_at:src_at + n]}.get(mode)
        if right is None:
            right = m[rbuf:rbuf + n]
            assert np.max(np.abs(right - S.rotate_right(yq if mode == 1 else mono_q[src_at:src_at + n], dr, theta))) \
                <= S.POST_R_TOL[precision] * max(1.0, scale)
        st = np.column_stack([np.roll(yq, dl) if mode else yq, right])
        x = O.peak_normalize(O.soft_saturate(st, drive), 0.98)
        want = np.column_stack([ss.resample_poly(x[:, k], up, down) for k in range(2)])
        got = o[fr:fr + n_x].astype(np.float64)
        assert got.shape == want.shape
        e = float(np.max(np.abs(got - want)))
        worst = max(worst, e)
        tol = 4 * 2.0 ** -24 if precision == "f64" else 2e-6 * 0.98
        assert e < tol, (n, mode, up, down, precision, e, tol)
    assert np.all(np.isnan(o[gaps])), "write outside every render's frames"
    return worst, o


@pytest.mark.parametrize("precision", ["f64", "f32"])
def test_stage_emulated(emul, precision):
    worst, _ = check_export(emul, precision, export_cases())
    print("ms_post_export %s: worst %.2e" % (precision, worst))


def test_stage_thread_schedule():
    """The same batch under MS_EMUL_SHUFFLE (fibres of a block in a fresh order between barriers): bitwise equal outputs."""
    code = ("import sys, hashlib; sys.path[:0] = [%r, %r, %r]\n"
            "from emul_device import EmulDevice; import test_export_sr as M\n"
            "dev = EmulDevice(); h = hashlib.sha256()\n"
            "for prec in ('f64', 'f32'):\n"
            "    o = M.export_run(dev, prec, M.export_cases())[0]; h.update(o.tobytes())\n"
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


# ---- end to end ----------------------------------------------------------------------------------------------------------
def _against_plain(out, meta, plain, p, tol):
    up, down = P.export_ratio(p)
    want = np.column_stack([ss.resample_poly(np.asarray(plain[:, k], np.float64), up, down) for k in range(2)])
    assert out.shape == want.shape and meta["out_sr"] == int(p["export_sr"])
    e = float(np.max(np.abs(out - want)))
    assert e < tol, (p.get("seed"), p["export_sr"], e)
    return e


def test_render_emulated(emul):
    """A short render with export_sr against resample_poly of the same render without it (whose float32 rounding the
    reference carries: a few 1e-7)."""
    for kw in (dict(), dict(stereo_on=False), dict(out_dur_s=0.0600208), dict(sat_drive=0.0), dict(base_sr=44100)):
        p = _short(**kw)
        plain, m0 = engine.render(p, device=emul, precision="f64", cache=False)
        for ex in (44100, 16000, 96000, 11025):
            if ex == int(p["base_sr"]):
                continue
            out, meta = engine.render(dict(p, export_sr=ex), device=emul, precision="f64", cache=False)
            _against_plain(out, meta, plain, dict(p, export_sr=ex), 5e-7)
            assert meta["design_sr_base"] == m0["design_sr_base"] and np.array_equal(meta["grain_last"], m0["grain_last"])


def test_render_batch_and_frontend_emulated(emul, tmp_path, monkeypatch):
    ps = [_short(seed=3 + i, export_sr=(None, 16000, 44100)[i % 3]) for i in range(5)]
    outs = engine.render_batch(ps, device=emul, precision="f64", workers=1)
    for p, o in zip(ps, outs):
        a, _ = engine.render(p, device=emul, precision="f64", cache=False)
        assert np.array_equal(o, a.astype(np.float32))
    monkeypatch.setattr(engine, "render_batch", lambda plist, device=None, precision="auto": engine._render_batch(
        plist, emul, "f64", None, 384, 3, 1, 32, True))
    base = _short(export_sr=22050)
    written = frontend.batch_render(base, [1], [20.0], [1.0, 2.0], str(tmp_path))
    for name, path in written:
        assert name.endswith("_22050Hzpwav")
        a, sr = frontend.read_wav(path)
        assert sr == 22050 and a.shape == (-(-int(round(0.06 * 48000)) * 147 // 320), 2)


# ---- GPU ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["f64", "f32"])
def test_stage_gpu(cuda_dev, precision):
    # modes 1 and 3 (the Bessel-tap right channel) are defined for even n only; modes 0 and 2 take odd n here
    cases = export_cases() + [(200000 + 2 * i + (i % 2 == 0), i % 4, 31, 77, 0.7, 1.0, 2.0, r) for i, r in enumerate(RATIOS)]
    worst, _ = check_export(cuda_dev, precision, cases)
    print("ms_post_export %s on the GPU: worst %.2e" % (precision, worst))


def _sweep_c5(k, ex):
    return [dict(configs.c5_params(i), export_sr=ex) for i in range(k)]


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["f64", "f32"])
def test_c3_c5_gpu(cuda_dev, precision):
    c3 = configs.canonical("C3")
    plain = [np.array(x) for x in engine.render_batch([c3] + _sweep_c5(64, None), device=cuda_dev, precision=precision)]
    worst = 0.0
    for ex in (44100, 16000):
        ps = [dict(c3, export_sr=ex)] + _sweep_c5(64, ex)
        outs = engine.render_batch(ps, device=cuda_dev, precision=precision)
        for p, o, a in zip(ps, outs, plain):
            up, down = P.export_ratio(p)
            want = np.column_stack([ss.resample_poly(a[:, k].astype(np.float64), up, down) for k in range(2)])
            e = float(np.max(np.abs(np.asarray(o, np.float64) - want)))
            worst = max(worst, e)
            assert e < (5e-7 if precision == "f64" else 3e-6), (ex, p["seed"], e)
    print("C3 + C5 %s: worst %.2e" % (precision, worst))


@pytest.mark.gpu
def test_c4_gpu(cuda_dev):
    c4 = configs.canonical("C4")
    plain, _ = engine.render(c4, device=cuda_dev, cache=False)
    for ex in (48000, 44100):
        out, meta = engine.render(dict(c4, export_sr=ex), device=cuda_dev, cache=False)
        print("C4 at %d: %.2e" % (ex, _against_plain(out, meta, plain, dict(c4, export_sr=ex), 5e-7)))


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["f64", "f32"])
def test_mixed_batch_gpu(cuda_dev, precision):
    """Plain renders of a mixed batch are bitwise those of a batch without exports; streamed pieces equal render()."""
    plain = [configs.c5_params(i) for i in range(12)]
    mixed = [dict(p, export_sr=(44100, 16000, 96000)[i % 3]) if i % 2 else p for i, p in enumerate(plain)]
    a = [np.array(x) for x in engine.render_batch(mixed, device=cuda_dev, precision=precision, chunk=4, ramp=False)]
    b = [np.array(x) for x in engine.render_batch(plain[0::2], device=cuda_dev, precision=precision)]
    for x, y in zip(a[0::2], b):
        assert np.array_equal(x, y)
    for i in (1, 3, 5, 6):
        d, m = engine.render(mixed[i], device=cuda_dev, precision=precision, cache=False)
        assert np.array_equal(a[i].astype(np.float64), d), i
        assert m["out_sr"] == int(mixed[i].get("export_sr", mixed[i]["base_sr"]))


@pytest.mark.gpu
def test_graph_replay_gpu(cuda_dev):
    engine.clear_render_cache()
    p = dict(configs.c5_params(9), export_sr=44100)
    a, _ = engine.render(p)                                     # eager
    b, _ = engine.render(p)                                     # captured and replayed
    c, _ = engine.render(p)                                     # replayed
    engine.clear_render_cache()
    assert np.array_equal(a, b) and np.array_equal(a, c) and a.shape == (88200, 2)
