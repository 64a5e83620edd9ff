"""Integer PCM export (EXTENSION; the reference returns float samples): the optional keys `export_format` ("pcm16" / "pcm24")
and `export_dither` through both planners, the tables' slot layout, the post stage's PCM write passes (ms_post_pcm) and the
engine and front end.

A PCM render runs exactly as a float render; the value its float path would round to float32 (x, widened to float64) is
quantised per channel as q = clamp(rint(x S + d), -S, S - 1), S = 2^(bits - 1), with d the TPDF dither of the output frame
drawn from Philox4x32-10 keyed by the seed (0 without dither).

The CPU tests run the stage on the block emulator; the GPU tests repeat them on the device and on real renders."""
import ctypes
import hashlib
import os
import subprocess
import sys

import numpy as np
import pytest

import stage_checks as S
from audio_suite_b200 import _abi, configs, decimate, engine, frontend, hostplan, plan as P, tables as T
from conftest import ROOT
from oracle import microsound_np as O


# ---- Philox4x32-10 and the quantiser, restated in numpy ---------------------------------------------------------------------
def philox4x32_10(ctr, key):
    """Philox4x32-10 (Random123) on arrays of counters: ctr = 4 arrays of uint32 words, key = 2 ints.  Returns 4 arrays."""
    m32 = np.uint64(0xFFFFFFFF)
    c = [np.asarray(w, np.uint64) & m32 for w in ctr]
    k0, k1 = int(key[0]) & 0xFFFFFFFF, int(key[1]) & 0xFFFFFFFF
    for r in range(10):
        if r:
            k0, k1 = (k0 + 0x9E3779B9) & 0xFFFFFFFF, (k1 + 0xBB67AE85) & 0xFFFFFFFF
        p0, p1 = np.uint64(0xD2511F53) * c[0], np.uint64(0xCD9E8D57) * c[2]
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ np.uint64(k0), p1 & m32, (p0 >> np.uint64(32)) ^ c[3] ^ np.uint64(k1), p0 & m32]
    return c


def seed_key(seed):
    s = int(seed) % (1 << 64)
    return s & 0xFFFFFFFF, s >> 32


def tpdf(n, seed):
    """float64 [n, 2]: the dither of output frames 0 .. n - 1 (d_L = (w0 - w1) 2^-32, d_R = (w2 - w3) 2^-32)."""
    i = np.arange(n, dtype=np.uint64)
    w = philox4x32_10((i & np.uint64(0xFFFFFFFF), i >> np.uint64(32), np.full(n, 0x64697468, np.uint64), np.zeros(n, np.uint64)),
                      seed_key(seed))
    w = [x.astype(np.float64) for x in w]
    return np.column_stack([(w[0] - w[1]) * 2.0 ** -32, (w[2] - w[3]) * 2.0 ** -32])


def quantise(x, bits, d):
    """The reference quantiser: float64 values in LSB before rounding, and the integers."""
    s = float(1 << (bits - 1))
    v = np.asarray(x, np.float64) * s + d
    return v, np.clip(np.rint(v), -s, s - 1).astype(np.int64)


def decode(q, bits):
    """int16 [n, 2] / uint8 [n, 6] -> int64 [n, 2]."""
    if bits == 16:
        return np.asarray(q, np.int64).reshape(-1, 2)
    b = np.asarray(q, np.uint8).reshape(-1, 2, 3).astype(np.int64)
    v = b[..., 0] | (b[..., 1] << 8) | (b[..., 2] << 16)
    return np.where(v >= 1 << 23, v - (1 << 24), v)


def test_philox_known_answers():
    kat = [((0, 0, 0, 0), (0, 0), "6627e8d5 e169c58d bc57ac4c 9b00dbd8"),
           ((0xFFFFFFFF,) * 4, (0xFFFFFFFF,) * 2, "408f276d 41c83b0e a20bc7c6 6d5451fd"),
           ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0), "d16cfe09 94fdcceb 5001e420 24126ea1")]
    for ctr, key, want in kat:
        got = philox4x32_10([np.array([w]) for w in ctr], key)
        assert " ".join("%08x" % int(w[0]) for w in got) == want


def test_dither_is_triangular():
    d = tpdf(1 << 16, 12345)
    assert np.all(np.abs(d) < 1.0) and abs(float(d.mean())) < 0.01
    assert abs(float(d.var()) - 1.0 / 6.0) < 0.01                  # TPDF on (-1, 1): variance 1/6
    assert not np.array_equal(tpdf(64, 1), tpdf(64, 2)) and np.array_equal(tpdf(64, 1 + (1 << 64)), tpdf(64, 1))


# ---- validation, identity -------------------------------------------------------------------------------------------------
def _short(**kw):
    base = dict(gen_mode="Resonant strike", micro_ms=3.0, time_unfold=20.0, out_dur_s=0.06, event_process="Poisson",
                grains_per_sec=60.0, bp_density="", stereo_on=True, er_cloud_on=True, er_taps=20, sat_drive=1.5)
    base.update(kw)
    return configs.with_defaults(base)


@pytest.mark.parametrize("kw,key", [(dict(export_format="pcm32"), "export_format"), (dict(export_format="PCM16"), "export_format"),
                                    (dict(export_format=16), "export_format"), (dict(export_format=b"pcm16"), "export_format"),
                                    (dict(export_format=["pcm16"]), "export_format"), (dict(export_format=True), "export_format"),
                                    (dict(export_format="pcm16", export_dither=1), "export_dither"),
                                    (dict(export_format="pcm24", export_dither="yes"), "export_dither"),
                                    (dict(export_format="pcm24", export_dither=None), "export_dither")])
def test_invalid_values_raise(kw, key, emul):
    p = _short(**kw)
    with pytest.raises(ValueError, match=key):
        P.plan_render(p)
    with pytest.raises(ValueError, match=key):
        engine.render(p, device=emul, cache=False)
    with pytest.raises(ValueError, match=key):
        hostplan.plan_chunk([p])


def test_dither_ignored_for_float_and_numpy_bool_taken():
    assert P.pcm_format(_short(export_format="float32", export_dither="anything")) is None
    assert P.pcm_format(_short(export_dither=3)) is None
    assert P.pcm_format(_short(export_format="pcm16", export_dither=np.bool_(False))) == (16, 0)
    assert P.pcm_format(_short(export_format="pcm24")) == (24, 1)


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


def test_identity_tables_and_output(emul):
    """Absent, None and "float32" (with any export_dither): identical tables from both planners, bitwise output."""
    ps = [_short(), _short(export_format=None), _short(export_format="float32"), _short(export_format="float32", export_dither=False)]
    want = T.pack_chunk([P.plan_render(ps[0])])
    assert len(want.pcm) == 0 and len(want.pcm_of) == 0
    for p in ps:
        _same_tables(T.pack_chunk([P.plan_render(p)]), want)
        _same_tables(hostplan.plan_chunk([p]), hostplan.plan_chunk([ps[0]]))
    outs = [engine.render(p, device=emul, precision="f64", cache=False)[0] for p in ps]
    for a in outs:
        assert a.dtype == np.float64 and np.array_equal(a, outs[0])


# ---- planners and the slot layout ------------------------------------------------------------------------------------------
def _sweep(k, seed):
    rng = np.random.default_rng(seed)
    fmts = (None, "float32", "pcm16", "pcm24", "pcm16", "pcm24")
    ps = []
    for i in range(k):
        p = dict(configs.c5_params(int(rng.integers(0, 4096))), out_dur_s=float(rng.uniform(0.05, 0.3)) + int(rng.integers(0, 4)) / 48000)
        p["export_format"] = fmts[int(rng.integers(0, len(fmts)))]
        if rng.integers(0, 2):
            p["export_dither"] = bool(rng.integers(0, 2))
        p["export_sr"] = (None, 44100, 16000)[int(rng.integers(0, 3))]
        p["stereo_on"] = bool(rng.integers(0, 2))
        p["seed"] = int(rng.integers(0, 1 << 40))
        ps.append(p)
    return ps


def _check_layout(t, rps):
    at = 0
    for r, rp in enumerate(rps):
        n_x = P.export_frames(rp.out_n, rp.export)
        bits = None if rp.pcm is None else rp.pcm[0]
        assert t.out_at[r] == at and t.out_n[r] == n_x and t.post[r]["out"] == at
        at += {None: n_x, 16: -(-n_x // 2), 24: -(-3 * n_x // 4)}[bits]
    assert t.frames == at
    assert t.pcm_of.tolist() == [r for r, rp in enumerate(rps) if rp.pcm is not None]
    for q, r in zip(t.pcm, t.pcm_of.tolist()):
        bits, dither, seed = rps[r].pcm
        assert q["fmt"].tolist() == [bits, dither] and q["key"].tolist() == list(seed_key(seed))
    for e, r in zip(t.export, t.export_of.tolist()):
        assert e["out"] == t.out_at[r] and e["out_end"] - e["out"] == t.out_n[r]


def test_slot_counts():
    for n in range(1, 40):
        assert P.output_slots(n) == n and P.output_slots(n, 16) == -(-n // 2) and P.output_slots(n, 24) == -(-3 * n // 4)
        assert 8 * P.output_slots(n, 16) >= 4 * n and 8 * P.output_slots(n, 24) >= 6 * n
        assert 8 * (P.output_slots(n, 24) - 1) < 6 * n and 8 * (P.output_slots(n, 16) - 1) < 4 * n


@pytest.mark.parametrize("seed", [1, 2])
def test_native_planner_matches_python(seed):
    subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "audio_suite_b200", "csrc"), "libms_hostplan.so"])
    hostplan._lib = None
    assert hostplan.lib() is not None
    ps = _sweep(40, seed)
    rps = [P.plan_render(p) for p in ps]
    want = T.pack_chunk(rps)
    _check_layout(want, rps)
    plain = T.pack_chunk([P.plan_render(dict(p, export_format=None)) for p in ps])
    for name in ("mono_n", "pool_n", "sy1", "ola_r", "fir", "odd", "rot", "y_at", "srs", "out_n", "export_of", "bank"):
        a, b = getattr(want, name), getattr(plain, name)
        assert (np.array_equal(a, b) if isinstance(a, np.ndarray) else a == b), name      # only the output slots move
    keep = [f for f in want.post.dtype.names if f != "out"]
    assert np.array_equal(want.post[keep], plain.post[keep])
    for got in (hostplan.plan_chunk(ps), hostplan.plan_chunk(ps, threads=3), hostplan.plan_chunk([P._slim_params(p) for p in ps])):
        _same_tables(got, want)
    for c5 in (["C4"], ["C3", "C2", "C1b"]):          # canonical configs, every render in one format
        for fmt in ("pcm16", "pcm24"):
            cs = [dict(configs.canonical(c), export_format=fmt) for c in c5]
            _same_tables(hostplan.plan_chunk(cs), T.pack_chunk([P.plan_render(p) for p in cs]))


def test_merged_chunks_match_one_chunk():
    ps = _sweep(30, 5)
    rps = [P.plan_render(p) for p in ps]
    whole = T.pack_chunk(rps)
    merged = T.merge_chunks([T.pack_chunk(rps[a:b]) for a, b in ((0, 7), (7, 8), (8, 30))])
    _check_layout(merged, rps)
    for name in ("out_at", "out_n", "pcm", "pcm_of", "export_of"):
        assert np.array_equal(getattr(merged, name), getattr(whole, name)), name
    assert merged.frames == whole.frames


def test_struct_size_matches_the_header():
    src = '#include "%s"\n#include <stdio.h>\n#include <stddef.h>\nint main(){printf("%%zu %%zu %%zu\\n", sizeof(ms_pcm_render),' \
          'offsetof(ms_pcm_render, key), offsetof(ms_pcm_render, fmt));}' \
          % os.path.join(ROOT, "include", "microsound_b200.h")
    import tempfile
    with tempfile.TemporaryDirectory() as d:
        open(os.path.join(d, "s.c"), "w").write(src)
        subprocess.check_call(["gcc", "-o", os.path.join(d, "s"), os.path.join(d, "s.c")])
        got = [int(x) for x in subprocess.check_output([os.path.join(d, "s")], text=True).split()]
    R = _abi.PcmRender
    assert got == [ctypes.sizeof(R), R.key.offset, R.fmt.offset] == [16, 0, 8]


# ---- the stage ------------------------------------------------------------------------------------------------------------
def stage_cases():
    """(n, stereo mode, dl, dr, theta, drive, scale, peak): modes 0-3, drive 0 and > 0, n = 1, 63, 64, odd, not a multiple
    of the tile, and a peak above full scale (the clamp)."""
    return [(1, 0, 0, 0, 0.0, 1.0, 1.0, 0.98), (63, 0, 0, 0, 0.0, 0.0, 2.0, 0.98), (64, 1, 5, 9, 0.63, 1.0, 1.0, 0.98),
            (1001, 2, 17, 0, 0.0, 1.3, 0.8, 0.98), (3000, 1, 29, 41, 0.9, 2.0, 3.0, 0.98), (2500, 3, 7, 11, 0.45, 0.0, 1.7, 0.98),
            (4097, 2, 0, 0, 0.0, 0.0, 1.0, 1.25), (2050, 3, 2049, 2048, 0.81, 1.0, 5.0, 0.98), (999, 0, 0, 0, 0.0, 2.5, 0.3, 1.1),
            (1027, 1, 3, 3, 0.2, 0.0, 1.0, 0.98)]


SENTINEL_BYTE = 0xA5


def stage_run(dev, precision, cases, ratio, bits, dither):
    """ms_post / ms_post_export (float) and ms_post_pcm on the same hand-built inputs, sentinels around every range.
    Returns per case (float32 output [n_x, 2], PCM output as int64 [n_x, 2], x reference inputs) and the launch log."""
    api, real = _abi.Api(dev.lib, precision), S._real(precision)
    rng = np.random.default_rng(17)
    recs, layout = [], []
    mono_n = S.GAP
    for n, mode, dl, dr, theta, drive, scale, peak in cases:
        y_at = mono_n
        mono_n += n + S.GAP
        src_at = mono_n
        mono_n += (2 * n if mode == 3 else n) + S.GAP
        rbuf = src_at + n if mode == 3 else src_at
        coef = T.bessel_coeffs(theta) if mode in (1, 3) else np.zeros(2 * _abi.POST_K + 1)
        r = np.zeros(1, np.dtype(_abi.PostRender))
        r[0] = (y_at, 0, rbuf if mode else 0, n, mode, dl, dr, drive, 1.0 / np.tanh(drive) if drive > 0 else 1.0, peak, coef)
        recs.append(r[0])
        n_x = n if ratio is None else -(-n * ratio[0] // ratio[1])
        layout.append(dict(y_at=y_at, src_at=src_at, rbuf=rbuf, n_x=n_x, y=rng.standard_normal(n) * scale,
                           y2=rng.standard_normal(n) * scale * 0.6, seed=0x123456789ABC + 977 * len(layout)))
    mono = np.full(mono_n, S.X_SENTINEL)
    for L in layout:
        mono[L["y_at"]:L["y_at"] + len(L["y"])] = L["y"]
        mono[L["src_at"]:L["src_at"] + len(L["y2"])] = L["y2"]
    # float layout: frames with GAP between renders; PCM layout: slots with GAP between renders
    fr, sl = S.GAP, S.GAP
    for L in layout:
        L["fr"], L["sl"], L["slots"] = fr, sl, P.output_slots(L["n_x"], bits)
        fr += L["n_x"] + S.GAP
        sl += L["slots"] + S.GAP
    bank = exps_f = exps_p = None
    if ratio is not None:
        half, taps, bk = decimate.polyphase_bank(*ratio)
        bank = dev.upload(bk.reshape(-1).astype(real))
        mk = lambda key: np.array([(L[key], L[key] + L["n_x"], 0, bk.size, ratio + (half, taps)) for L in layout], np.dtype(_abi.ExportRender))
        exps_f, exps_p = dev.upload(mk("fr")), dev.upload(mk("sl"))
    rec_f, rec_p = np.array(recs, np.dtype(_abi.PostRender)), np.array(recs, np.dtype(_abi.PostRender))
    rec_f["out"] = [L["fr"] for L in layout]
    rec_p["out"] = [L["sl"] for L in layout]
    pcm = np.array([(seed_key(L["seed"]), (bits, dither)) for L in layout], np.dtype(_abi.PcmRender))
    max_n, max_x = max(c[0] for c in cases), max(L["n_x"] for L in layout)
    d_rec_f, d_rec_p, d_pcm = dev.upload(rec_f), dev.upload(rec_p), dev.upload(pcm)         # (kept alive across the calls)
    # float run
    d_mono, mb = dev.upload(mono.astype(real)), dev.zeros(len(recs), np.uint64)
    out_f = dev.upload(np.full(2 * fr, np.nan, np.float32))
    if ratio is None:
        rc = api.ms_post(dev.ptr(d_rec_f), len(recs), max_n, dev.ptr(d_mono), dev.ptr(mb), dev.ptr(out_f), dev.stream_ptr())
    else:
        rc = api.ms_post_export(dev.ptr(d_rec_f), dev.ptr(exps_f), len(recs), max_n, max_x, dev.ptr(d_mono), dev.ptr(mb),
                                dev.ptr(bank), dev.ptr(out_f), dev.stream_ptr())
    assert rc == 0, dev.lib.ms_last_error()
    # PCM run
    d_mono2, mb2 = dev.upload(mono.astype(real)), dev.zeros(len(recs), np.uint64)
    out_p = dev.upload(np.full(8 * sl, SENTINEL_BYTE, np.uint8))
    with S.LaunchLog(dev) as log:
        rc = api.ms_post_pcm(dev.ptr(d_rec_p), dev.ptr(d_pcm), dev.ptr(exps_p) if ratio else None, len(recs), max_n,
                             max_x if ratio else 0, bits, dither, dev.ptr(d_mono2), dev.ptr(mb2), dev.ptr(bank) if ratio else None,
                             dev.ptr(out_p), dev.stream_ptr())
        assert rc == 0, dev.lib.ms_last_error()
    of = S._fetch(dev, out_f, np.float32, 2 * fr).reshape(-1, 2)
    op = S._fetch(dev, out_p, np.uint8, 8 * sl)
    m = S._fetch(dev, d_mono, real, mono_n).astype(np.float64)
    gaps = np.ones(op.size, bool)
    res = []
    for c, L in zip(cases, layout):
        a, nb = 8 * L["sl"], 8 * L["slots"]
        gaps[a:a + nb] = False
        raw = op[a:a + nb]
        used = (4 if bits == 16 else 6) * L["n_x"]
        assert np.all(raw[used:] == 0), "bytes past the last frame of a render's slots must be zero"
        q = engine.pcm_frames(raw.copy(), L["n_x"], bits)
        assert q.dtype == (np.int16 if bits == 16 else np.uint8)
        res.append((of[L["fr"]:L["fr"] + L["n_x"]].astype(np.float64), decode(q, bits), L, m))
    assert np.all(op[gaps] == SENTINEL_BYTE), "write outside every render's slots"
    return res, mono, log


def _lsb_check(got, v, x_err, bits):
    """Within 1 LSB everywhere; exact wherever v lies farther than x_err (in LSB) from a half-integer.  Returns mismatches."""
    s = float(1 << (bits - 1))
    want = np.clip(np.rint(v), -s, s - 1)
    diff = np.abs(got - want)
    assert np.all(diff <= 1)
    far = np.abs(np.abs(v - np.floor(v)) - 0.5) > x_err
    assert np.all(diff[far] == 0), (int(np.count_nonzero(diff[far])), int(far.sum()))
    return int(np.count_nonzero(diff))


def check_stage(dev, precision, cases, ratio, bits, dither):
    res, mono, log = stage_run(dev, precision, cases, ratio, bits, dither)
    assert "PostMaxK" in log.base() and ("PostWritePcmK" if ratio is None else "PostExportPcmK") in log.base(), log.names
    assert len(log.names) == 2, log.names
    mono_q = S._as_ref(mono, precision)
    s = float(1 << (bits - 1))
    mism = 0
    for (xf, got, L, m), (n, mode, dl, dr, theta, drive, scale, peak) in zip(res, cases):
        d = tpdf(L["n_x"], L["seed"]) if dither else np.zeros((L["n_x"], 2))
        v, _ = quantise(xf, bits, d)
        if precision == "f32":
            # the quantiser's input is exactly the float32 value the float path stores: every sample is exact
            assert np.array_equal(got, np.clip(np.rint(v), -s, s - 1)), (n, mode, ratio, bits, dither)
        else:
            # the float path rounds x to float32: at most half an ulp of |x| away
            mism += _lsb_check(got, v, s * np.abs(xf) * 2.0 ** -24 + 1e-9, bits)
            if drive == 0 and (ratio is None or n <= EXACT_EXPORT_MAX):
                # the quantiser of float64 x = v * (peak / max|L, R|) (resampled in the kernel's order), restated: exact
                yq = mono_q[L["y_at"]:L["y_at"] + n]
                right = {0: yq, 2: mono_q[L["src_at"]:L["src_at"] + n]}.get(mode)
                if right is None:
                    right = m[L["rbuf"]:L["rbuf"] + n]
                st = np.column_stack([np.roll(yq, dl) if mode else yq, right])
                x = O.peak_normalize(st, peak)
                if ratio is not None:
                    x = np.column_stack([resample_in_order(x[:, k], ratio, fused=hasattr(dev, "torch")) for k in range(2)])
                assert np.array_equal(got, quantise(x, bits, d)[1]), (n, mode, ratio, bits, dither)
    return mism


# renders up to this length get the exact float64 check under export_sr too (the fused reference runs in exact rationals)
EXACT_EXPORT_MAX = 5000


def resample_in_order(x, ratio, fused):
    """float64 x through the polyphase bank exactly as the export pass sums it: per output m, acc += h * x[q + s] in
    ascending s from acc = 0.  `fused`: each step is one correctly rounded fused multiply-add, as nvcc compiles the loop;
    otherwise a rounded product, then a rounded sum (the block emulator's g++ build).  Terms with q + s outside [0, n)
    multiply a zero and leave the sum as it is."""
    from fractions import Fraction
    up, down = ratio
    half, taps, bank = decimate.polyphase_bank(up, down)
    a, n = half // up, len(x)
    q, p = np.divmod(np.arange(-(-n * up // down), dtype=np.int64) * down, up)
    acc = np.zeros(len(q))
    for j in range(taps):
        idx = q + j - a
        ok = (idx >= 0) & (idx < n)
        h, w = bank[p[ok], j], x[idx[ok]]
        if fused:
            acc[ok] = [float(Fraction(hh) * Fraction(ww) + Fraction(cc)) for hh, ww, cc in zip(h.tolist(), w.tolist(), acc[ok].tolist())]
        else:
            acc[ok] = acc[ok] + h * w
    return acc


STAGE_CONFIGS = [(r, b, d) for r in (None, (147, 160), (2, 1)) for b in (16, 24) for d in (0, 1)]


@pytest.mark.parametrize("precision", ["f64", "f32"])
@pytest.mark.parametrize("ratio,bits,dither", STAGE_CONFIGS)
def test_stage_emulated(emul, precision, ratio, bits, dither):
    mism = check_stage(emul, precision, stage_cases(), ratio, bits, dither)
    print("ms_post_pcm %s ratio %s pcm%d dither %d: %d samples 1 LSB off the float32 path" % (precision, ratio, bits, dither, mism))


def test_stage_rejects_other_formats(emul):
    api = _abi.Api(emul.lib, "f64")
    for bits, dither in ((8, 0), (32, 1), (16, 2)):
        assert api.ms_post_pcm(None, None, None, 0, 0, 0, bits, dither, None, None, None, None, None) != 0
        assert b"unsupported format" in emul.lib.ms_last_error()


def test_stage_thread_schedule():
    """A pcm24 batch with dither, plain and exporting, under MS_EMUL_SHUFFLE: bitwise equal outputs."""
    code = ("import sys, hashlib; sys.path[:0] = [%r, %r, %r]\n"
            "from emul_device import EmulDevice; import test_pcm_export as M\n"
            "dev = EmulDevice(); h = hashlib.sha256()\n"
            "for prec in ('f64', 'f32'):\n"
            "    for ratio in (None, (147, 160)):\n"
            "        for q in M.stage_run(dev, prec, M.stage_cases()[:6], ratio, 24, 1)[0]: h.update(q[1].tobytes())\n"
            "print(h.hexdigest())\n") % (ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "tests", "host_emul"))
    digests = []
    for seed in (None, "3"):
        env = dict(os.environ)
        env.pop("MS_EMUL_SHUFFLE", None)
        if seed:
            env["MS_EMUL_SHUFFLE"] = seed
        p = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, cwd=ROOT)
        assert p.returncode == 0, p.stderr[-4000:]
        digests.append(p.stdout.strip().splitlines()[-1])
    assert len(set(digests)) == 1, digests


# ---- end to end ------------------------------------------------------------------------------------------------------------
def _against_float(q, f, bits, tol_lsb=1):
    """PCM without dither against rint(float render * S): within tol_lsb, and only where f S is near a half-integer."""
    s = float(1 << (bits - 1))
    v = f * s
    got = decode(q, bits)
    return _lsb_check(got, v, s * np.abs(f) * 2.0 ** -23 + 1e-9, bits)


def test_render_emulated(emul):
    """render() with pcm16 / pcm24, dither off and on, plain and exported, against the float render of the same params."""
    p = _short()
    for ex in (None, 44100):
        f, m0 = engine.render(dict(p, export_sr=ex), device=emul, precision="f64", cache=False)
        for fmt, bits in (("pcm16", 16), ("pcm24", 24)):
            q, m = engine.render(dict(p, export_sr=ex, export_format=fmt, export_dither=False), device=emul, precision="f64", cache=False)
            assert q.dtype == (np.int16 if bits == 16 else np.uint8) and q.shape == ((len(f), 2) if bits == 16 else (len(f), 6))
            assert m["out_sr"] == m0["out_sr"] and np.array_equal(m["grain_last"], m0["grain_last"])
            _against_float(q, f, bits)
            qd, _ = engine.render(dict(p, export_sr=ex, export_format=fmt), device=emul, precision="f64", cache=False)
            v, want = quantise(f, bits, tpdf(len(f), p["seed"]))
            _lsb_check(decode(qd, bits), v, float(1 << (bits - 1)) * np.abs(f) * 2.0 ** -23 + 1e-9, bits)


def test_render_batch_and_frontend_emulated(emul, tmp_path, monkeypatch):
    ps = [_short(seed=3 + i, export_sr=(None, 16000, 44100)[i % 3], export_format=(None, "pcm16", "pcm24", "pcm16")[i % 4],
                 out_dur_s=0.06 + i / 48000) for i in range(7)]
    outs = engine.render_batch(ps, device=emul, precision="f64", workers=1)
    for p, o in zip(ps, outs):
        a, _ = engine.render(p, device=emul, precision="f64", cache=False)
        assert o.dtype == {None: np.float32, "pcm16": np.int16, "pcm24": np.uint8}[p["export_format"]]
        assert np.array_equal(o, a.astype(o.dtype))
    monkeypatch.setattr(engine, "render_batch", lambda plist, device=None, precision="auto": engine._render_batch(
        plist, emul, "f64", None, 384, 3, 1, 32, True))
    for fmt, bits in (("pcm16", 16), ("pcm24", 24)):
        base = _short(export_format=fmt, export_sr=44100)
        written = frontend.batch_render(base, [1], [20.0], [1.0, 2.0], str(tmp_path / fmt))
        for (name, path), p in zip(written, frontend.batch_params(base, [1], [20.0], [1.0, 2.0])):
            _check_wav(path, bits, 44100, engine.render(p, device=emul, precision="f64", cache=False)[0])


def _check_wav(path, bits, rate, q):
    import struct
    raw = open(path, "rb").read()
    kind, ch, sr, byte_rate, align, b = struct.unpack("<HHIIHH", raw[20:36])
    assert (kind, ch, sr, byte_rate, align, b) == (1, 2, rate, rate * 2 * bits // 8, 2 * bits // 8, bits)
    a, sr2 = frontend.read_wav(path)
    assert sr2 == rate and np.array_equal(a * float(1 << (bits - 1)), decode(q, bits).astype(np.float64))


def test_write_wav_pcm_rejects_other_arrays(tmp_path):
    for bad in (np.zeros((4, 2), np.float32), np.zeros((4, 3), np.uint8), np.zeros(8, np.int16)):
        with pytest.raises(ValueError):
            frontend.write_wav_pcm(str(tmp_path / "x.wav"), bad, 48000)


# ---- GPU ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["f64", "f32"])
@pytest.mark.parametrize("ratio,bits,dither", STAGE_CONFIGS)
def test_stage_gpu(cuda_dev, precision, ratio, bits, dither):
    # modes 1 and 3 (the Bessel-tap right channel) are defined for even n only
    cases = stage_cases() + [(200000 + 2 * i + (i % 2 == 0), i % 4, 31, 77, 0.7, (1.0, 0.0)[i % 2], 2.0, 0.98) for i in range(4)]
    mism = check_stage(cuda_dev, precision, cases, ratio, bits, dither)
    print("ms_post_pcm %s ratio %s pcm%d dither %d on the GPU: %d samples 1 LSB off the float32 path" % (precision, ratio, bits, dither, mism))


@pytest.mark.gpu
@pytest.mark.parametrize("name,ex", [("C1", None), ("C1b", None), ("C2", None), ("C3", 44100)])
def test_whole_renders_gpu(cuda_dev, name, ex):
    p = dict(configs.canonical(name), export_sr=ex)
    f, _ = engine.render(p, device=cuda_dev, cache=False)
    q, _ = engine.render(dict(p, export_format="pcm16", export_dither=False), device=cuda_dev, cache=False)
    print("%s pcm16: %d samples 1 LSB off rint(float * 32768)" % (name, _against_float(q, f, 16)))


def _mixed():
    base = [configs.c5_params(i) for i in range(12)]
    kinds = [(None, None), ("pcm16", None), ("pcm24", None), (None, 44100), ("pcm16", 44100), ("pcm24", 16000),
             ("pcm16", None), (None, None), ("pcm24", 44100), ("float32", 44100), ("pcm16", 16000), ("pcm24", None)]
    out = []
    for i, (p, (fmt, ex)) in enumerate(zip(base, kinds)):
        q = dict(p, export_format=fmt, export_sr=ex)
        if i % 3 == 1:
            q["export_dither"] = False
        out.append(q)
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["f64", "f32"])
def test_mixed_batch_gpu(cuda_dev, precision):
    """A mixed batch: the float renders equal a batch without the PCM ones; each PCM render is the quantiser of the same
    render in an all-float batch of the same params (exactly in f32, where its input is that float32 value); in f64 every
    render equals its lone render().  (In f32 a lone render can differ from the batch's in the last bits: grains of equal
    length share a transform with a different partner.)"""
    ps = _mixed()
    a = [np.array(x) for x in engine.render_batch(ps, device=cuda_dev, precision=precision, chunk=5, ramp=False)]
    fmts = [P.pcm_format(p) for p in ps]
    b = [np.array(x) for x in engine.render_batch([p for p, f in zip(ps, fmts) if f is None], device=cuda_dev, precision=precision)]
    assert [np.array_equal(x, y) for x, y in zip([x for x, f in zip(a, fmts) if f is None], b)] == [True] * len(b)
    c = [np.array(x) for x in engine.render_batch([dict(p, export_format=None) for p in ps], device=cuda_dev, precision=precision,
                                                  chunk=5, ramp=False)]
    for i, (p, f) in enumerate(zip(ps, fmts)):
        if f is None:
            assert np.array_equal(a[i], c[i]), i
            continue
        bits, dither = f
        v, want = quantise(c[i].astype(np.float64), bits, tpdf(len(c[i]), p["seed"]) if dither else 0.0)
        if precision == "f32":
            assert np.array_equal(decode(a[i], bits), want), i
        else:
            _lsb_check(decode(a[i], bits), v, float(1 << (bits - 1)) * np.abs(c[i]) * 2.0 ** -24 + 1e-9, bits)
    if precision == "f64":
        for i, p in enumerate(ps):
            d, m = engine.render(p, device=cuda_dev, precision=precision, cache=False)
            assert d.dtype == (np.float64 if fmts[i] is None else a[i].dtype)
            assert np.array_equal(a[i].astype(d.dtype), d), i
            assert m["out_sr"] == int(p["export_sr"] or p["base_sr"])


@pytest.mark.gpu
def test_repeatable_and_graph_replay_gpu(cuda_dev):
    ps = _mixed()
    h = [hashlib.sha256(b"".join(np.ascontiguousarray(x).tobytes() for x in engine.render_batch(ps, device=cuda_dev))).hexdigest()
         for _ in range(2)]
    assert h[0] == h[1]
    engine.clear_render_cache()
    for fmt in ("pcm16", "pcm24"):
        p = dict(configs.c5_params(9), export_sr=44100, export_format=fmt)
        a, _ = engine.render(p)                                     # eager
        b, _ = engine.render(p)                                     # captured and replayed
        c, _ = engine.render(p)                                     # replayed
        assert np.array_equal(a, b) and np.array_equal(a, c) and len(a) == 88200
    engine.clear_render_cache()


@pytest.mark.gpu
def test_frontend_gpu(cuda_dev, tmp_path, monkeypatch):
    monkeypatch.setattr(engine, "render_batch", lambda plist, device=None, precision="auto": engine._render_batch(
        plist, cuda_dev, "auto", None, 384, 3, None, 32, True))
    for fmt, bits in (("pcm16", 16), ("pcm24", 24)):
        base = dict(configs.c5_params(0), export_format=fmt)
        written = frontend.batch_render(base, [1, 2], [1.0], [1.0], str(tmp_path / fmt))
        for (name, path), p in zip(written, frontend.batch_params(base, [1, 2], [1.0], [1.0])):
            _check_wav(path, bits, int(p["base_sr"]), engine.render(p, device=cuda_dev, cache=False)[0])
