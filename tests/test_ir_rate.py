"""IR sample rate (EXTENSION; the reference plays an impulse response at base_sr whatever its file rate): the optional key
`space_ir_sr` resamples every column of `_ir_audio` to base_sr on the device (ms_resample_poly, resample_poly's filter)
before the planners cut and mix it; the IR fragment generator keeps reading `_ir_audio` as given.

The CPU tests run the resampler and short renders on the block emulator; the GPU tests repeat the kernel checks at full
size and render through every FIR route."""
import ctypes as C
import hashlib
import os
import subprocess
import sys

import numpy as np
import pytest
import scipy.signal as ss

from audio_suite_b200 import _abi, configs, decimate, engine, frontend, hostplan, plan as P, tables as T
from oracle import microsound_np as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RATIOS = ((2, 1), (4, 1), (160, 147), (147, 160), (320, 147), (640, 147), (1, 4))


def _short(ir, **kw):
    base = dict(gen_mode="Resonant strike", micro_ms=3.0, time_unfold=20.0, out_dur_s=0.06, event_process="Poisson",
                grains_per_sec=60.0, bp_density="", stereo_on=True, er_cloud_on=True, er_taps=20, sat_drive=1.5,
                space_ir_on=True, space_ir_max_samps=12000, _ir_audio=ir)
    base.update(kw)
    return configs.with_defaults(base)


def _same_tables(a, b):
    for name in a.__dataclass_fields__:
        x, y = getattr(a, name), getattr(b, name)
        if isinstance(x, np.ndarray):
            assert x.dtype == y.dtype and x.shape == y.shape, name
            for f in (x.dtype.names or (None,)):
                if f is None or not (f.startswith("_pad") or f == "h"):     # (ms_fir_render.h is unused)
                    assert np.array_equal(T.column(x, f), T.column(y, f)), (name, f)
        else:
            assert x == y, name


class _NoDevice:
    """A device on which every use fails: validation must raise before any device work."""
    def __getattr__(self, name):
        raise AssertionError(f"device touched ({name})")


# ---- the kernel against scipy -------------------------------------------------------------------------------------------
def kernel_cases(big):
    """(up, down, n): shorter than one phase's taps, odd, 2880 (the shortest shipped IR), and about 1e5 (on the emulator only
    for the cheaper ratios)."""
    out = []
    for up, down in RATIOS:
        taps = decimate.polyphase_bank(up, down)[1]
        for n in (max(1, taps // 3), 1001, 2880, 100003):
            if n == 100003 and not big and up * 1.0 / down > 2.5:
                continue
            out.append((up, down, n))
    return out


def _strided_run(dev, precision, up, down, x, n_out=None, pad=37):
    """ms_resample_poly on len(x) signals of n samples placed at strided offsets of one buffer (stride n + pad, first signal
    at pad), outputs likewise between sentinels.  Returns [signals, n_out] and checks that no sentinel moved."""
    api = _abi.Api(dev.lib, precision)
    real = np.float32 if precision == "f32" else np.float64
    s, n = x.shape
    full = -(-n * up // down)
    n_out = full if n_out is None else n_out
    xs, ys = n + pad, n_out + pad
    xb = np.full(pad + s * xs, 7.0, real)
    for k in range(s):
        xb[pad + k * xs:pad + k * xs + n] = x[k]
    half, taps, bank = decimate.polyphase_bank(up, down)
    dx, db = dev.upload(xb), dev.upload(bank.astype(real))
    dy = dev.upload(np.full(pad + s * ys, -3.0, real))
    esz = np.dtype(real).itemsize
    px = C.c_void_p(dev.ptr(dx).value + pad * esz)
    py = C.c_void_p(dev.ptr(dy).value + pad * esz)
    assert api.ms_resample_poly(px, xs, n, s, dev.ptr(db), up, down, half, taps, py, ys, n_out, dev.stream_ptr()) == 0
    dev.synchronize()
    yb = np.asarray(dev.download(dy, 0, (pad + s * ys) * esz)).view(real)
    y = np.stack([yb[pad + k * ys:pad + k * ys + n_out] for k in range(s)])
    gaps = np.concatenate([yb[:pad]] + [yb[pad + k * ys + n_out:pad + (k + 1) * ys] for k in range(s)])
    assert np.all(gaps == -3.0)
    return y


def check_kernel(dev, precision, big):
    tol = 1e-12 if precision == "f64" else 2e-6
    rng = np.random.default_rng(2026)
    worst = 0.0
    for up, down, n in kernel_cases(big):
        for s in (1, 2):
            x = rng.standard_normal((s, n))
            want = np.stack([ss.resample_poly(x[k], up, down) for k in range(s)])
            got = _strided_run(dev, precision, up, down, x)
            assert got.shape == want.shape
            e = float(np.max(np.abs(got - want)) / np.max(np.abs(want)))
            worst = max(worst, e)
            assert e < tol, (up, down, n, s, e)
        # the wrapper, along axis 0 like scipy; n_out: bitwise the first rows of the full call
        col = np.ascontiguousarray(x.T)
        full = decimate.resample_poly(col, up, down, dev, precision)
        assert full.shape == (want.shape[1], s) and np.array_equal(full, got.T)
        for k in (0, 1, want.shape[1] // 3 + 1, want.shape[1] - 1):
            part = decimate.resample_poly(col, up, down, dev, precision, n_out=k)
            assert part.shape == (k, s) and np.array_equal(part, full[:k]), (up, down, n, k)
        assert np.array_equal(_strided_run(dev, precision, up, down, x, n_out=want.shape[1] // 2), got[:, :want.shape[1] // 2])
    return worst


@pytest.mark.parametrize("precision", ["f64", "f32"])
def test_kernel_against_scipy_emulated(emul, precision):
    print("ms_resample_poly %s on the emulator: worst %.2e of the peak" % (precision, check_kernel(emul, precision, False)))


def test_kernel_refuses_bad_arguments(emul):
    api = _abi.Api(emul.lib, "f64")
    half, taps, bank = decimate.polyphase_bank(2, 1)
    x, y, b = emul.upload(np.zeros(64)), emul.zeros(256, np.float64), emul.upload(bank)
    p = emul.ptr
    for args in ((0, 1, half, taps, 64, 1, 128), (2, 0, half, taps, 64, 1, 128), (2, 1, half, taps + 1, 64, 1, 128),
                 (2, 1, half, taps, -1, 1, 128), (2, 1, half, taps, 64, 2, 128)):
        up, down, h, t, n, s, n_out = args
        assert api.ms_resample_poly(p(x), 64 if s == 1 else 32, n, s, p(b), up, down, h, t, p(y), n_out, n_out, None) == -1
        assert b"ms_resample_poly" in emul.lib.ms_last_error()
    assert np.all(y == 0)


def kernel_digest(dev):
    h = hashlib.sha256()
    rng = np.random.default_rng(5)
    for prec in ("f64", "f32"):
        for up, down in RATIOS:
            h.update(_strided_run(dev, prec, up, down, rng.standard_normal((2, 3001))).tobytes())
    return h.hexdigest()


def test_kernel_thread_schedule():
    """The kernel under MS_EMUL_SHUFFLE (fibres of a block in a fresh order between barriers): bitwise equal outputs."""
    code = ("import sys; sys.path[:0] = [%r, %r, %r]\n"
            "from emul_device import EmulDevice; import test_ir_rate as M\n"
            "print(M.kernel_digest(EmulDevice()))\n") % (ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "tests", "host_emul"))
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


# ---- validation and identity ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("value", [True, np.bool_(False), 0, -1, 44100.0, "44100", np.float64(44100.0)])
@pytest.mark.parametrize("ir_on", [True, False])
def test_invalid_values_raise(value, ir_on):
    p = _short(configs.synth_ir(0.05, 48000, 3), space_ir_sr=value, space_ir_on=ir_on)
    with pytest.raises(ValueError, match="space_ir_sr"):
        engine.render(p, device=_NoDevice(), cache=False)
    with pytest.raises(ValueError, match="space_ir_sr"):
        engine.resolve_ir_rate([_short(None), p], _NoDevice())
    with pytest.raises(ValueError, match="space_ir_sr"):
        P.plan_render(p)
    with pytest.raises(ValueError, match="space_ir_sr"):
        hostplan.plan_chunk([p])


@pytest.mark.parametrize("base,sr", [(192000, 22050), (96000, 11025), (48000, 47999)])
def test_over_limit_ratios_raise(base, sr):
    p = _short(configs.synth_ir(0.05, 48000, 3), base_sr=base, space_ir_sr=sr)
    with pytest.raises(ValueError, match="at most 640"):
        engine.render(p, device=_NoDevice(), cache=False)
    with pytest.raises(ValueError, match="at most 640"):
        P.plan_render(p)


def test_ratios():
    assert P.ir_rate(_short(None, space_ir_sr=np.int64(44100))) == (160, 147)
    assert P.ir_rate(_short(None, base_sr=96000, space_ir_sr=48000)) == (2, 1)
    assert P.ir_rate(_short(None, base_sr=44100, space_ir_sr=48000)) == (147, 160)
    for base in (48000, 96000, 192000):
        assert max(P.ir_rate(_short(None, base_sr=base, space_ir_sr=44100))) <= P.EXPORT_RATIO_LIMIT
    for base in (44100, 96000):
        assert max(P.ir_rate(_short(None, base_sr=base, space_ir_sr=48000))) <= P.EXPORT_RATIO_LIMIT
    assert P.ir_rate(_short(None, space_ir_sr=48000)) is None and P.ir_rate(_short(None)) is None


def test_planners_refuse_an_unresolved_ir():
    p = _short(configs.synth_ir(0.05, 44100, 3), space_ir_sr=44100)
    with pytest.raises(ValueError, match="not been resampled"):
        P.plan_render(p)
    with pytest.raises(ValueError, match="not been resampled"):
        hostplan.plan_chunk([p])


def test_identity_tables_and_output(emul):
    """Absent, None and space_ir_sr == base_sr (int or numpy int): identical tables from both planners and bitwise renders;
    with the IR off or absent, the key changes nothing either."""
    ir = configs.synth_ir(0.05, 48000, 3)
    ps = [_short(ir), _short(ir, space_ir_sr=None), _short(ir, space_ir_sr=48000), _short(ir, space_ir_sr=np.int32(48000))]
    want = T.pack_chunk([P.plan_render(ps[0])])
    for p in ps:
        q = engine.resolve_ir_rate([p], _NoDevice())[0]
        assert q is p
        _same_tables(T.pack_chunk([P.plan_render(q)]), want)
        _same_tables(hostplan.plan_chunk([q]), hostplan.plan_chunk([ps[0]]))
    for precision in ("f64", "f32"):
        a, _ = engine.render(ps[0], device=emul, precision=precision, cache=False)
        for p in ps[1:]:
            assert np.array_equal(engine.render(p, device=emul, precision=precision, cache=False)[0], a)
    for off in (_short(ir, space_ir_on=False), _short(None)):
        q = dict(off, space_ir_sr=44100)
        assert engine.resolve_ir_rate([q], _NoDevice())[0] is q
        _same_tables(T.pack_chunk([P.plan_render(q)]), T.pack_chunk([P.plan_render(off)]))


def test_resolution_copies_and_caches(emul):
    ir = configs.synth_ir(0.2, 44100, 4)
    p = _short(ir, space_ir_sr=44100, space_ir_tap_cap=None, space_ir_max_samps=5000)
    before = dict(p)
    ps = engine.resolve_ir_rate([p, dict(p, seed=9), _short(ir)], emul)
    assert p == before and P.IR_RESAMPLED not in p                       # the caller's dict is untouched
    h = ps[0][P.IR_RESAMPLED]
    assert ps[1][P.IR_RESAMPLED] is h and P.IR_RESAMPLED not in ps[2] and ps[0]["_ir_audio"] is ir
    assert h.shape == (5000, 2) and h.dtype == np.float64
    full = decimate.resample_poly(ir, 160, 147, emul, "f64")
    assert np.array_equal(h, full[:5000])
    assert engine.resolve_ir_rate([p], emul)[0][P.IR_RESAMPLED] is h   # cached per (IR, rates, kept rows)
    assert P.ir_rate_rows(dict(p, space_ir_tap_cap=3)) == 8 and P.ir_rate_rows(dict(p, space_ir_tap_cap=100)) == 100
    assert P.ir_rate_rows(dict(p, space_ir_tap_cap=None)) == 5000 and P.ir_rate_rows(p | {"space_ir_max_samps": -1}) is None


def test_semantics_resample_first(emul):
    """The planners' taps are the slice / "< 8 values" test / cut / mono mix (or pair) of resample_poly of the WHOLE IR."""
    ir = configs.synth_ir(0.1, 44100, 6)
    full = ss.resample_poly(ir, 160, 147)
    for kw, want in ((dict(), full[:8192].mean(axis=1)), (dict(space_ir_tap_cap=None, space_ir_max_samps=3000), full[:3000].mean(axis=1)),
                     (dict(space_ir_tap_cap=3), full[:3].mean(axis=1)), (dict(space_ir_max_samps=3), None)):
        p = engine.resolve_ir_rate([_short(ir, space_ir_sr=44100, **kw)], emul)[0]
        got = P.plan_render(p).ir
        if want is None:
            assert got is None
        else:
            assert got.shape == want.shape and np.max(np.abs(got - want)) < 1e-12
    p = engine.resolve_ir_rate([_short(ir, space_ir_sr=44100, space_ir_stereo=True)], emul)[0]
    rp = P.plan_render(p)
    assert np.max(np.abs(rp.ir - full[:8192, 0])) < 1e-12 and np.max(np.abs(rp.ir_r - full[:8192, 1])) < 1e-12


def _random_sweep(k, seed, emul):
    rng = np.random.default_rng(seed)
    irs = [configs.synth_ir(0.3, 44100, 11), configs.synth_ir(0.2, 96000, 12, channels=1), configs.synth_ir(0.25, 48000, 13)]
    ps = []
    for i in range(k):
        ir_i = int(rng.integers(0, 3))
        base = int(rng.choice([44100, 48000, 96000]))
        ps.append(_short(irs[ir_i], seed=int(rng.integers(0, 10 ** 6)), base_sr=base, time_unfold=float(rng.integers(10, 40)),
                         gen_mode=str(rng.choice(configs.BASIC_MODES)), stereo_on=bool(rng.integers(0, 2)),
                         space_ir_sr=[None, 44100, 48000, 96000, 22050][int(rng.integers(0, 5))],
                         space_ir_tap_cap=[8192, None, 2000, 5][int(rng.integers(0, 4))],
                         space_ir_max_samps=int(rng.choice([12000, 3000, 40000])), space_ir_stereo=bool(rng.integers(0, 2)),
                         space_ir_on=bool(rng.integers(0, 8))))
    return engine.resolve_ir_rate(ps, emul)


@pytest.mark.parametrize("seed", [1, 2])
def test_planner_parity(emul, seed, monkeypatch):
    """Native planner, Python planner and the pooled digests: identical tables for 64 randomised renders, mono and stereo."""
    subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "audio_suite_b200", "csrc"), "libms_hostplan.so"])
    hostplan._lib = None
    assert hostplan.lib() is not None
    # (the planners' tap caches start empty, so that 64 renders never overflow them: a cache cleared in the middle of a
    #  call hands out new arrays for an IR already pooled, and the two planners would pool them at different places)
    P._TAPS_CACHE.clear()
    P._PAIR_CACHE.clear()
    ps = _random_sweep(64, seed, emul)
    assert sum(P.IR_RESAMPLED in p for p in ps) >= 16
    want = T.pack_chunk([P.plan_render(p) for p in ps])
    for got in (hostplan.plan_chunk(ps), hostplan.plan_chunk(ps, threads=3), hostplan.plan_chunk([P._slim_params(p) for p in ps]),
                T.pack_chunk([P.plan_render(P._slim_params(p)) for p in ps])):
        _same_tables(got, want)
    monkeypatch.setenv("MS_PLAN_PYTHON", "1")
    [tb] = T.plan_stream(ps, 64, workers=1)
    _same_tables(tb, want)
    for p in ps:
        q = P._slim_params(p)
        assert P.IR_RESAMPLED not in q and (q is p or q["_ir_audio"] is None)


# ---- end to end on the emulator --------------------------------------------------------------------------------------------
def test_render_emulated(emul):
    """render() with the key equals render() of the resampled array without it, bitwise; render_batch equals render()."""
    ir = configs.synth_ir(0.06, 44100, 21)
    for kw in (dict(), dict(space_ir_stereo=True), dict(space_ir_tap_cap=None, space_ir_max_samps=2000)):
        p = _short(ir, space_ir_sr=44100, **kw)
        h = decimate.resample_poly(ir, 160, 147, emul, "f64", n_out=P.ir_rate_rows(p))
        for precision in ("f64", "f32"):
            a, ma = engine.render(p, device=emul, precision=precision, cache=False)
            b, mb = engine.render(dict(p, _ir_audio=h, space_ir_sr=None), device=emul, precision=precision, cache=False)
            assert np.array_equal(a, b) and a.shape == b.shape, (kw, precision)
            assert np.array_equal(ma["grain_last"], mb["grain_last"])
    ps = [_short(ir, seed=3 + i, space_ir_sr=(None, 44100, 96000)[i % 3]) for i in range(4)]
    outs = engine.render_batch(ps, device=emul, precision="f64", workers=1)
    for p, o in zip(ps, outs):
        a, _ = engine.render(p, device=emul, precision="f64", cache=False)
        assert np.array_equal(o, a.astype(np.float32))


def test_ir_fragment_generator_reads_the_file_rate_ir(emul):
    ir = configs.synth_ir(0.06, 44100, 22)
    p = _short(ir, gen_mode="IR fragment")
    a, ma = engine.render(p, device=emul, precision="f64", cache=False)
    b, mb = engine.render(dict(p, space_ir_sr=44100), device=emul, precision="f64", cache=False)
    assert np.array_equal(ma["micro_last"], mb["micro_last"]) and not np.array_equal(a, b)


def test_load_ir_wav_with_rate(tmp_path):
    x = np.random.default_rng(3).uniform(-0.5, 0.5, (300, 2))
    frontend.write_wav_float32(str(tmp_path / "ir.wav"), x, 44100)
    ir, sr = frontend.load_ir_wav(str(tmp_path / "ir.wav"), with_rate=True)
    assert sr == 44100 and np.array_equal(ir, frontend.load_ir_wav(str(tmp_path / "ir.wav")))
    st, sr = frontend.load_ir_wav(str(tmp_path / "ir.wav"), stereo=True, with_rate=True)
    assert sr == 44100 and st.shape == (300, 2)


# ---- GPU -------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["f64", "f32"])
def test_kernel_against_scipy_gpu(cuda_dev, precision):
    print("ms_resample_poly %s on the GPU: worst %.2e of the peak" % (precision, check_kernel(cuda_dev, precision, True)))


def _shipped_ir(tmp_path):
    import kernel_checks as K
    (tmp_path / "irs").mkdir(exist_ok=True)
    irs = K.shipped_irs(tmp_path / "irs")
    path = next(p for p in irs if p.endswith("ir_tiny_room_250ms.wav"))
    return frontend.load_ir_wav(path, with_rate=True)


def _with_key_equals_explicit(dev, p):
    up, down = P.ir_rate(p)
    h = decimate.resample_poly(p["_ir_audio"], up, down, dev, "f64", n_out=P.ir_rate_rows(p))
    a, _ = engine.render(p, device=dev, precision="f64", cache=False)
    b, _ = engine.render(dict(p, _ir_audio=h, space_ir_sr=None), device=dev, precision="f64", cache=False)
    assert a.shape == b.shape and np.array_equal(a, b)
    return a


@pytest.mark.gpu
def test_render_mono_route_gpu(cuda_dev):
    """The 8192-tap mono route at base_sr 48000 with a 44.1 kHz IR: bitwise the render of the device-resampled array, and
    within the parity bar of the oracle's render with scipy's resample_poly of the IR."""
    c3 = configs.canonical("C3")
    ir = configs.synth_ir(1.0, 44100, 31)
    p = dict(c3, _ir_audio=ir, space_ir_sr=44100)
    a = _with_key_equals_explicit(cuda_dev, p)
    ref, _ = O.render(dict(c3, _ir_audio=ss.resample_poly(ir, 160, 147)))
    e = float(np.max(np.abs(a - ref)))
    print("C3 with a 44.1 kHz IR against the oracle: %.2e" % e)
    assert e < 1e-5


@pytest.mark.gpu
def test_render_stereo_gpu(cuda_dev):
    c3 = configs.canonical("C3")
    _with_key_equals_explicit(cuda_dev, dict(c3, _ir_audio=configs.synth_ir(1.0, 44100, 32), space_ir_sr=44100, space_ir_stereo=True))


@pytest.mark.gpu
def test_render_long_route_gpu(cuda_dev, tmp_path):
    """A shipped 48 kHz IR at base_sr 96000, uncapped (24000 rows after resampling: the long FIR route)."""
    ir, sr = _shipped_ir(tmp_path)
    assert sr == 48000
    p = dict(configs.canonical("C3"), base_sr=96000, out_dur_s=2.0, _ir_audio=ir, space_ir_sr=sr, space_ir_tap_cap=None)
    _with_key_equals_explicit(cuda_dev, p)
    assert engine.resolve_ir_rate([p], cuda_dev)[0][P.IR_RESAMPLED].shape == (2 * ir.shape[0],)


@pytest.mark.gpu
def test_mixed_batch_gpu(cuda_dev):
    """A render_batch where only some renders set the key: each render equal to its lone render()."""
    ir = configs.synth_ir(0.5, 44100, 33)
    ps = [dict(configs.c5_params(i), _ir_audio=ir) for i in range(12)]
    ps = [dict(p, space_ir_sr=44100) if i % 3 else p for i, p in enumerate(ps)]
    outs = [np.array(x) for x in engine.render_batch(ps, device=cuda_dev, precision="f64", chunk=4, ramp=False)]
    for i, (p, o) in enumerate(zip(ps, outs)):
        a, _ = engine.render(p, device=cuda_dev, precision="f64", cache=False)
        assert np.array_equal(o.astype(np.float64), a), i


@pytest.mark.gpu
def test_batch_render_gpu(cuda_dev, tmp_path):
    ir, sr = _shipped_ir(tmp_path)
    base = dict(configs.canonical("C3"), base_sr=96000, out_dur_s=0.5, _ir_audio=ir, space_ir_sr=sr)
    written = frontend.batch_render(base, [1, 2], [20.0], [1.0], str(tmp_path / "out"), device=cuda_dev, precision="f64")
    assert len(written) == 2
    for name, path in written:
        a, rate = frontend.read_wav(path)
        assert rate == 96000 and a.shape == (48000, 2) and np.all(np.isfinite(a)) and np.max(np.abs(a)) > 0.1
