"""Stage-level checks of the time-domain kernels -- the FIR (reflection cloud + impulse response by overlap-save),
overlap-add + ADSR and the stereo / clip / normalise tail -- against plain float64 restatements of the same operations.

Every check drives the C ABI directly with hand-built records, on whichever device it is given (the block emulator in
the CPU suite, the B200 in the GPU suite).  In float32 every input is rounded to float32 before the reference sees it,
so reference and kernel start from the same data.  Buffers carry sentinels around each render's range: reads outside
the range show up as wrong values, writes outside it as overwritten sentinels."""
import ctypes as C
import re

import numpy as np

from audio_suite_b200 import _abi, engine, tables
from oracle import microsound_np as O

# Tolerances, set from measurement.  Worst cases measured on the block emulator and on an NVIDIA B200 (1000 W power
# limit), which agree to within a factor of two:
#   FIR, relative to max|ref|:                f64 2.3e-15 (B200) / 1.6e-15 (emulator), f32 7.4e-7 / 7.3e-7
#   overlap-add + ADSR, relative to max|ref|: f64 4.3e-16 / 1.7e-16, f32 4.7e-7 / 4.7e-7
#   ms_post right channel, relative to max|y|: f64 8.7e-15 / 8.7e-15, f32 1.9e-7 / 1.9e-7
#   float32 stereo output, absolute:          f64 1.3e-7 = 2.2 units of 2^-24, f32 1.6e-7 = 2.7 units (clip and scale
#                                             are then float32 operations), beyond what the right channel carries in
# i.e. margins of 40x and more (f64), 4x and more (f32) on the stage errors; the float32 output is held to 4 (f64) and
# 8 (f32) units of 2^-24: its own rounding plus tanhf of a float32 argument.
FIR_TOL = {"f64": 1e-13, "f32": 3e-6}
OLA_TOL = {"f64": 1e-13, "f32": 3e-6}
POST_R_TOL = {"f64": 1e-13, "f32": 3e-6}
POST_OUT_TOL = {"f64": 4 * 2.0 ** -24, "f32": 8 * 2.0 ** -24}

GAP = 64                         # sentinel samples between two renders' ranges
X_SENTINEL = 1.0e3               # in input gaps: a read outside a render's input changes its output visibly


def _real(precision):
    return np.float32 if precision == "f32" else np.float64


def _as_ref(a, precision):
    """What the kernel sees of `a`, widened to float64 for the reference."""
    return np.asarray(a, np.float64).astype(_real(precision)).astype(np.float64)


def _fetch(dev, buf, dtype, count):
    """`count` elements of `dtype` from the start of a device buffer (uploaded buffers are bytes)."""
    dev.synchronize()
    raw = np.asarray(dev.download(buf, 0, count if _elem_bytes(buf) != 1 else count * np.dtype(dtype).itemsize))
    return raw.view(dtype)[:count].copy() if raw.dtype != dtype else raw[:count].copy()


def _elem_bytes(buf):
    return buf.element_size() if hasattr(buf, "element_size") else buf.dtype.itemsize


def _rel(got, want):
    return float(np.max(np.abs(got - want)) / max(1e-300, float(np.max(np.abs(want))))) if want.size else 0.0


# ---- launch log: which kernels a call ran (ms_set_launch_hook; the emulator passes __PRETTY_FUNCTION__ as well) ----------
_KNAME = re.compile(r"K = (?:\w+::)*(\w+(?:<[^;\]]*>)?)")


class LaunchLog:
    """Records kernel names while active.  With a hook set, ms_spectral_run leaves out its side streams, so only the
    direct stage checks use this; the in-situ checks run the production schedule without it."""

    def __init__(self, dev):
        self.dev, self.names = dev, []

    def __enter__(self):
        def hook(name, stream):
            m = _KNAME.search(name.decode())
            self.names.append(m.group(1) if m else name.decode())
        self._hook = _abi.LAUNCH_HOOK(hook)
        self.dev.lib.ms_set_launch_hook(C.cast(self._hook, C.c_void_p))
        return self

    def __exit__(self, *exc):
        self.dev.lib.ms_set_launch_hook(None)
        return False

    def base(self):
        return {n.split("<")[0] for n in self.names}


# ---- 1. FIR: reflection cloud + impulse response, overlap-save (ms_fir_*) ------------------------------------------------
def fir_reference(ir, offs, gains, x, x_begin, x_end):
    """M:409-421 then M:438-445, as written: x_er = x + sum_t g_t shift(x, off_t) (taps sharing a delay add up), then the
    direct convolution np.convolve(x_er, ir)[:n] -- restricted to where x_er can be non-zero."""
    n = len(x)
    hi = min(n, x_end + (int(np.max(offs)) if len(offs) else 0))
    xer = np.zeros(hi - x_begin)
    xer[:x_end - x_begin] = x[x_begin:x_end]
    for off, g in zip(np.asarray(offs).tolist(), np.asarray(gains).tolist()):
        if 0 < off < hi - x_begin:
            xer[off:] += g * x[x_begin:x_begin + hi - x_begin - off]
    y = np.zeros(n)
    seg = np.convolve(xer, ir)[:n - x_begin]
    y[x_begin:x_begin + len(seg)] = seg
    return y


def fir_reference_fft(ir, offs, gains, x, x_begin, x_end):
    """Same filter, for the many-unit batches: h = ir * (delta + cloud) by direct convolution, then a float64 FFT
    convolution (its own rounding, ~1e-15 of the peak, is 100x below the f64 tolerance)."""
    from scipy.signal import fftconvolve
    e = np.zeros(int(np.max(offs)) + 1 if len(offs) else 1)
    e[0] = 1.0
    np.add.at(e, np.asarray(offs), np.asarray(gains))
    h = np.convolve(ir, e)
    y = np.zeros(len(x))
    seg = fftconvolve(x[x_begin:x_end], h)[:len(x) - x_begin]
    y[x_begin:x_begin + len(seg)] = seg
    return y


def fir_case(name, rng, n, ir_len, ntaps, max_off, B, x_begin=None, x_end=None, residue=None, dup=0, share=None):
    """One render: a decaying random IR, `ntaps` reflection taps with off = 1 and off = max_off among them (`residue`:
    every delay = residue mod 256; `dup`: that many taps repeat an earlier delay), input support [x_begin, x_end) with
    non-zero samples at both ends.  `B`: the overlap-save block length the planner must choose."""
    ir = rng.standard_normal(ir_len) * np.exp(-np.arange(ir_len) / max(1.0, ir_len / 4.0))
    ir[-1] = 0.5 if ir_len > 1 else 1.0              # the last tap reaches the last output of the live range
    if ntaps:
        offs = rng.integers(1, max_off + 1, ntaps)
        if residue is not None:
            assert max_off % 256 == residue
            offs = (offs // 256) * 256 + residue
            offs[offs < 1] += 256
            offs[offs > max_off] -= 256
            offs[1] = 256 if residue == 0 else residue
        else:
            offs[1] = 1
        offs[0] = max_off
        for k in range(dup):                         # delays shared by several taps (some three or more times)
            offs[-1 - k] = offs[2 + (k % max(1, min(dup // 3 + 1, ntaps - 3)))]
        gains = rng.uniform(-1.0, 1.0, ntaps) * 0.3
        gains[0] = 0.7                               # the longest delay carries weight
    else:
        offs, gains = np.zeros(0, np.int64), np.zeros(0)
    x_begin = 0 if x_begin is None else x_begin
    x_end = n if x_end is None else x_end
    x = np.zeros(n)
    x[x_begin:x_end] = rng.standard_normal(x_end - x_begin)
    x[x_begin], x[x_end - 1] = 1.5, -1.25
    return dict(name=name, ir=ir, offs=np.asarray(offs, np.int64), gains=np.asarray(gains), x=x, x_begin=x_begin,
                x_end=x_end, B=B, share=share)


def fir_cases(big):
    """Every branch of ols_block_len / fir_layout and the tap sets that reach the special rows of the fused kernel."""
    rng = np.random.default_rng(2026 if big else 7)
    s = 3 if big else 1                              # longer outputs on the GPU; filter lengths are what pick the path
    c = [
        fir_case("B8192", rng, 20000 * s, 1000, 40, 2000, 8192, x_begin=300, x_end=15000 * s, dup=6),
        fir_case("B32768-one-pair", rng, 30000, 4000, 100, 2000, 32768, x_begin=17, x_end=29000, dup=10),
        # h_len 8160 -> hop 57377: 3 (7 on the GPU) blocks, so the last unit has no partner block
        fir_case("B65536-taps-odd-blocks", rng, 400000 if big else 150000, 6000, 320, 2160, 65536, x_begin=300,
                 x_end=390000 if big else 140000, dup=12),
        fir_case("B65536-no-taps", rng, 100000 * s, 8192, 0, 0, 65536, x_begin=5, x_end=99000 * s),
        fir_case("B65536-residue-0", rng, 140000, 4000, 64, 46 * 256, 65536, residue=0, x_begin=1000, x_end=120000),
        fir_case("B65536-residue-128", rng, 140000, 4000, 64, 46 * 256 + 128, 65536, residue=128, x_end=139000),
        fir_case("B65536-4096-taps", rng, 120000 * s, 2000, 4096, 6000, 65536, x_begin=64, x_end=110000 * s, dup=300),
        fir_case("B131072", rng, 200000 * s, 8192, 200, 10000, 131072, x_begin=3, x_end=190000 * s, dup=8),
        fir_case("B262144", rng, 300000 * s, 8192, 100, 30000, 262144, x_begin=2, x_end=260000 * s, dup=4),
        fir_case("delta-IR-taps", rng, 70000, 1, 300, 2500, 8192, x_begin=11, x_end=69000, dup=20),
        # five blocks, three units: the live range ends in block 1, the first block of unit 1 (the cases above end
        # their live range in a partner block or at out_n)
        fir_case("B65536-live-end-in-block-a", rng, 230000, 6000, 160, 2160, 65536, x_begin=70000, x_end=100000, dup=3),
    ]
    # one IR spectrum shared by two renders, and equal IR content at a second pool offset
    c.append(dict(fir_case("B65536-shared-IR", rng, 130000, 6000, 320, 2160, 65536, x_begin=40, x_end=125000, dup=5),
                  ir=c[2]["ir"], share="B65536-taps-odd-blocks"))
    c.append(dict(fir_case("B65536-equal-IR-copy", rng, 130000, 6000, 100, 2160, 65536, x_begin=0, x_end=130000),
                  ir=c[2]["ir"].copy()))
    return c


def fir_many_units_batch(n_renders=100):
    """300 fused units (three per render) sharing one IR spectrum, with and without taps: one launch per phase covers
    every unit, each with its own scratch block."""
    rng = np.random.default_rng(404)
    hop = 65536 - 8160 + 1
    base = fir_case("cluster-0", rng, 5 * hop + 1000, 6000, 320, 2160, 65536, dup=12)
    out = []
    for i in range(n_renders):
        ntaps = 0 if i % 4 == 3 else 320 - i % 7
        cse = fir_case("cluster-%d" % i, rng, 5 * hop + 1000 + 37 * i, 6000, ntaps, 2160 if ntaps else 0, 65536,
                       x_begin=i, x_end=5 * hop + 900 + 37 * i, dup=i % 9)
        cse["ir"] = base["ir"]
        cse["share"] = "cluster-0"
        if ntaps == 0:                                # same h_len for every render: pad the IR instead of the taps
            cse["ir"] = np.concatenate([base["ir"], np.zeros(2160)])
            cse["ir"][-1] = 0.25
            cse["share"] = "cluster-padded"
        out.append(cse)
    return out


def fir_run(dev, precision, cases, runs=1):
    """All `cases` as ONE ms_fir_create (renders interleaved as given) and `runs` ms_fir_run calls on that handle.
    Returns (list of outputs per run, each the full output buffer; per-case offsets; kernel base names)."""
    api, real = _abi.Api(dev.lib, precision), _real(precision)
    recs, irs, offs, gains = [], [], [], []
    pool_at, ir_n, t_n, at = {}, 0, 0, GAP
    xbuf = []
    starts = []
    for cs in cases:
        key = cs.get("share") or cs["name"]
        if key not in pool_at:
            pool_at[key] = ir_n
            irs.append(cs["ir"])
            ir_n += len(cs["ir"])
        r = _abi.FirRender()
        r.ir, r.ir_len = pool_at[key], len(cs["ir"])
        r.h_len = len(cs["ir"]) + (int(np.max(cs["offs"])) if len(cs["offs"]) else 0)
        r.tap_begin, r.tap_end = t_n, t_n + len(cs["offs"])
        r.x, r.y, r.out_n, r.x_begin, r.x_end = at, at, len(cs["x"]), cs["x_begin"], cs["x_end"]
        recs.append(r)
        offs.append(cs["offs"])
        gains.append(cs["gains"])
        xbuf.append(cs["x"])
        starts.append(at)
        t_n += len(cs["offs"])
        at += len(cs["x"]) + GAP
    total = at
    x = np.full(total, X_SENTINEL)
    for s, v in zip(starts, xbuf):
        x[s:s + len(v)] = v
    arr = (_abi.FirRender * len(recs))(*recs)
    need = api.ms_fir_workspace_bytes(C.addressof(arr), len(recs))
    assert need > 0, dev.lib.ms_last_error()
    ws = dev.empty(need, np.uint8)
    d_ir = dev.upload(np.concatenate(irs).astype(real))
    d_off = dev.upload(np.concatenate(offs).astype(np.int32) if t_n else np.zeros(1, np.int32))
    d_gain = dev.upload((np.concatenate(gains) if t_n else np.zeros(1)).astype(real))
    d_x = dev.upload(x.astype(real))
    d_y = dev.upload(np.full(total, np.nan, real))
    h = C.c_void_p()
    outs = []
    with LaunchLog(dev) as log:
        rc = api.ms_fir_create(C.addressof(arr), len(recs), dev.ptr(d_ir), dev.ptr(d_off), dev.ptr(d_gain), dev.ptr(d_x),
                               dev.ptr(d_y), dev.ptr(ws), need, dev.stream_ptr(), C.byref(h))
        assert rc == 0, dev.lib.ms_last_error()
        try:
            for _ in range(runs):
                assert api.ms_fir_run(h, dev.stream_ptr()) == 0, dev.lib.ms_last_error()
                outs.append(_fetch(dev, d_y, real, total).astype(np.float64))
        finally:
            api.ms_fir_destroy(h)
    return outs, starts, log


def fir_expected_route(cases):
    """Kernel base names each case must have launched: fused 65536-point units (one launch per phase), or the spectral
    engine's rows / columns behind the dense tap scatter."""
    fused = [cs["B"] == 65536 for cs in cases]
    want, absent = set(), set()
    if any(fused):
        want |= {"FirP1K", "FirP2K", "FirP3K"}
        if any(f and len(cs["offs"]) for f, cs in zip(fused, cases)):
            want.add("FirSortK")
    else:
        absent |= {"FirP1K", "FirP2K", "FirP3K", "FirSortK"}
    legacy = [not f for f in fused]
    if any(legacy):
        want.add("RowsK")
        if any(lg and len(cs["offs"]) for lg, cs in zip(legacy, cases)):
            want.add("ErScatterK")
    else:
        absent.add("ErScatterK")
    return want, absent


def check_fir_outputs(precision, cases, out, starts, ref=fir_reference, refs=None, label=""):
    """Per case: exact zeros outside [x_begin, x_end + h_len - 1), reference inside, sentinel gaps untouched."""
    errs = {}
    gaps = np.ones(len(out), bool)
    for k, (cs, s) in enumerate(zip(cases, starts)):
        n = len(cs["x"])
        gaps[s:s + n] = False
        got = out[s:s + n]
        assert not np.any(np.isnan(got)), (label, cs["name"], "output not written", int(np.argmax(np.isnan(got))))
        h_len = len(cs["ir"]) + (int(np.max(cs["offs"])) if len(cs["offs"]) else 0)
        live_hi = min(n, cs["x_end"] + h_len - 1)
        assert np.all(got[:cs["x_begin"]] == 0.0) and np.all(got[live_hi:] == 0.0), (label, cs["name"], "non-zero outside the support")
        want = refs[k] if refs is not None else ref(_as_ref(cs["ir"], precision), cs["offs"], _as_ref(cs["gains"], precision),
                                                    _as_ref(cs["x"], precision), cs["x_begin"], cs["x_end"])
        errs[cs["name"]] = _rel(got, want)
        assert errs[cs["name"]] < FIR_TOL[precision], (label, precision, cs["name"], errs[cs["name"]], int(np.argmax(np.abs(got - want))))
    assert np.all(np.isnan(out[gaps])), (label, "write outside every render's range")
    return errs


def check_fir(dev, precision, big=False, many=False):
    """Each case alone (its route asserted), then all of them as one batch run twice (bitwise-identical repeats), and
    optionally the many-unit batch.  Returns {"errors": ..., "kernels": ...}."""
    cases = fir_cases(big)
    refs = [fir_reference(_as_ref(cs["ir"], precision), cs["offs"], _as_ref(cs["gains"], precision), _as_ref(cs["x"], precision),
                          cs["x_begin"], cs["x_end"]) for cs in cases]
    errors, kernels = {}, set()
    for cs, r in zip(cases, refs):
        (out,), starts, log = fir_run(dev, precision, [cs])
        want, absent = fir_expected_route([cs])
        assert want <= log.base() and not (absent & log.base()), (cs["name"], sorted(log.base()))
        errors.update(check_fir_outputs(precision, [cs], out, starts, refs=[r], label="alone"))
        kernels |= set(log.names)
    # one batch: the classes interleaved (stable sort by class, per-render offsets), IRs shared and duplicated
    order = [0, 2, 7, 3, 1, 11, 4, 9, 12, 5, 10, 8, 6]
    assert sorted(order) == list(range(len(cases)))
    batch = [cases[i] for i in order]
    outs, starts, log = fir_run(dev, precision, batch, runs=2)
    assert np.array_equal(outs[0], outs[1], equal_nan=True), "second ms_fir_run on one handle differs"
    berr = check_fir_outputs(precision, batch, outs[0], starts, refs=[refs[i] for i in order], label="batch")
    errors.update({"batch:" + k: v for k, v in berr.items()})
    if many:
        mb = fir_many_units_batch()
        outs, starts, log = fir_run(dev, precision, mb, runs=2)
        assert np.array_equal(outs[0], outs[1], equal_nan=True), "second ms_fir_run on the many-unit batch differs"
        want, absent = fir_expected_route(mb)
        assert want <= log.base() and not (absent & log.base()), sorted(log.base())
        merr = check_fir_outputs(precision, mb, outs[0], starts, ref=fir_reference_fft, label="many-unit batch")
        errors["many-unit-batch-worst"] = max(merr.values())
        kernels |= set(log.names)
    return {"errors": errors, "kernels": sorted(kernels)}


# ---- 2. overlap-add + ADSR (ms_adsr_tables, ms_overlap_add) ---------------------------------------------------------------
def ola_record(out_at, n, events, adsr):
    """ms_ola_render of one render: events (start-sorted) at ev_begin..ev_end; adsr = (A, D, R samples, S, curve) turned
    into the closed-form description exactly as the planner does (tables.pack_chunk)."""
    a, d, rel, S, curve = adsr
    d_end = min(n, a + d) if d > 0 else a
    sus_end = max(d_end, n - rel)
    r = np.zeros(1, np.dtype(_abi.OlaRender))
    r[0] = (out_at, n, events[0], events[1], events[2], a, d_end, sus_end, 1 if (rel > 0 and n > sus_end) else 0,
            1.0 / a if a > 0 else 0.0, 1.0 / (d_end - a) if d_end > a else 0.0,
            1.0 / (n - sus_end - 1) if n - sus_end > 1 else 0.0, S, curve, -1)
    return r[0]


def ola_cases(big):
    """(out_n, adsr, events) per render; events are (start, len) pairs, grains drawn later.  Covers: events spanning
    several 1024-sample tiles, more overlapping events than a tile has threads, start = 0, an event ending exactly at
    out_n, a render with no events, ADSR with A = 0, no release, a one-sample release, curve != 1, an attack that fills
    the whole render, a decay cut short by out_n, and release lengths where k * (1 / k) != 1 in float64."""
    s = 8 if big else 1
    rng = np.random.default_rng(11)
    cases = []
    n = 9000 * s
    ev = [(0, 2600), (1500, 3000), (n - 777, 777), (n - 3000, 3000)]
    ev += [(3000 + int(v), 700) for v in rng.integers(0, 300, 300)]            # 300 events over one tile
    cases.append((n, (0, 500, 1000, 0.6, 1.0), ev))                             # A = 0
    n = 7001 * s
    ev = [(int(a), int(rng.integers(1, 2500))) for a in rng.integers(0, n - 1, 60)]
    ev = [(a, min(ln, n - a)) for a, ln in ev] + [(n - 1, 1)]
    cases.append((n, (300, 200, 0, 0.5, 2.3), ev))                              # no release, curve 2.3
    n = 4097
    cases.append((n, (100, 300, 1, 0.7, 0.5), [(0, n), (5, 1024), (1023, 1025)]))  # out_n - sus_end == 1, curve 0.5
    n = 3000
    cases.append((n, (3000, 0, 0, 1.0, 1.7), [(0, 3000), (2047, 953)]))         # the attack fills the render
    n = 5000
    cases.append((n, (0, 0, 0, 1.0, 1.0), []))                                  # no events
    n = 6000 * s
    cases.append((n, (4000 * s, 5000 * s, 0, 0.3, 1.0), [(1, n - 1), (1024, 2048)]))   # decay cut short by out_n
    n = 2500
    cases.append((n, (10, 20, 49 + 1, 0.8, 3.0), [(int(a), 200) for a in range(0, 2300, 97)] + [(n - 60, 60)]))   # 49 * (1 / 49) != 1
    return cases


def ola_reference(n, adsr, events, grains, amps):
    mix = np.zeros(n)
    for (st, ln), g, amp in zip(events, grains, amps):       # event order, as M:755
        mix[st:st + ln] += amp * g[:ln]
    a, d, rel, S, curve = adsr
    return mix * O.adsr_envelope(n, 1000.0, float(a), float(d), float(S), float(rel), float(curve))


def check_ola(dev, precision, big=False):
    """Closed-form envelope (env < 0) and tabulated envelope (ms_adsr_tables) against the reference and each other."""
    api, real = _abi.Api(dev.lib, precision), _real(precision)
    rng = np.random.default_rng(12)
    cases = ola_cases(big)
    recs, evts, pool, grains, amps_all = [], [], [], [], []
    pool_n, out_at = 0, GAP
    for n, adsr, ev in cases:
        ev = sorted(ev, key=lambda e: e[0])                   # stable: equal starts keep their order
        b0 = len(evts)
        gs, am = [], []
        for st, ln in ev:
            off = int(rng.integers(0, 40))                    # the event starts `off` samples into its grain
            g = rng.standard_normal(off + ln + 3)
            amp = float(rng.uniform(0.2, 1.7))
            pool.append(g)
            evts.append((pool_n + off, st, ln, amp))
            gs.append(_as_ref(g[off:off + ln], precision))
            am.append(float(real(amp)))
            pool_n += len(g)
        max_len = max([ln for _, ln in ev], default=0)
        recs.append(ola_record(out_at, n, (b0, len(evts), max_len), adsr))
        grains.append((ev, gs, am))
        out_at += n + GAP
    total = out_at
    rec = np.array(recs, dtype=np.dtype(_abi.OlaRender))
    ev_arr = np.zeros(max(1, len(evts)), np.dtype(_abi.OlaEvt))
    for i, e in enumerate(evts):
        ev_arr[i] = e
    d_pool = dev.upload(np.concatenate(pool).astype(real))
    d_ev = dev.upload(ev_arr)
    max_n = max(n for n, _, _ in cases)
    results = {}
    with LaunchLog(dev) as log:
        for form in ("closed", "table"):
            r = rec.copy()
            env_n = 0
            if form == "table":
                for i, (n, _, _) in enumerate(cases):
                    r["env"][i] = env_n
                    env_n += n
            d_r = dev.upload(r)
            d_env = dev.upload(np.full(max(1, env_n), np.nan, real))
            mono = dev.upload(np.full(total, np.nan, real))
            if form == "table":
                assert api.ms_adsr_tables(dev.ptr(d_r), len(r), max_n, dev.ptr(d_env), dev.stream_ptr()) == 0, dev.lib.ms_last_error()
            assert api.ms_overlap_add(dev.ptr(d_r), len(r), max_n, dev.ptr(d_ev), dev.ptr(d_pool), dev.ptr(d_env), dev.ptr(mono),
                                      dev.stream_ptr()) == 0, dev.lib.ms_last_error()
            results[form] = _fetch(dev, mono, real, total).astype(np.float64)
    assert {"AdsrTableK", "OlaK"} <= log.base(), sorted(log.base())
    errors = {}
    for form, out in results.items():
        gaps = np.ones(total, bool)
        for (n, adsr, _), rr, (ev, gs, am) in zip(cases, recs, grains):
            at = int(rr["out"])
            gaps[at:at + n] = False
            got = out[at:at + n]
            want = ola_reference(n, adsr, ev, gs, am)
            e = _rel(got, want) if np.any(want) else float(np.max(np.abs(got)))
            errors["%s n=%d adsr=%s" % (form, n, adsr)] = e
            assert e < OLA_TOL[precision], (form, precision, n, adsr, e, int(np.argmax(np.abs(got - want))))
            if rr["has_release"] and n - int(rr["sus_end"]) > 1:
                assert got[-1] == 0.0, (form, n, adsr, "the release must close at exactly 0", got[-1])
        assert np.all(np.isnan(out[gaps])), (form, "write outside every render's range")
    d = float(np.max(np.abs(results["closed"] - results["table"]), initial=0.0, where=~np.isnan(results["closed"])))
    errors["closed vs table"] = d
    assert d <= 4 * np.finfo(real).eps * max(float(np.nanmax(np.abs(results["closed"]))), 1e-300), d
    return errors


# ---- 3. stereo diffusion + soft clip + normalise (ms_post) -----------------------------------------------------------------
def rotate_right(y, dr, theta):
    """Right channel of M:423-436 for the shifts given: irfft(rfft(roll(y, -dr)) * exp(i theta sin(2 pi k / kmax)))."""
    spec = np.fft.rfft(np.roll(y, -dr))
    k = np.arange(spec.size, dtype=np.float64)
    return np.fft.irfft(spec * np.exp(1j * theta * np.sin(2 * np.pi * k / max(1.0, k[-1]))), n=len(y))


def bessel_right(y, dr, coef):
    """The same channel for even n as the direct 25-tap sum R[i] = sum_m J_m(theta) y[(i + dr + 2m) mod n]."""
    K = (len(coef) - 1) // 2
    n = len(y)
    i = np.arange(n)
    return sum(coef[K + m] * y[(i + dr + 2 * m) % n] for m in range(-K, K + 1))


def post_reference(y, mode, dl, dr, theta, drive, peak, rbuf=None):
    if mode == 0:
        st = np.column_stack([y, y])
    else:
        right = rotate_right(y, dr, theta) if mode == 1 else rbuf
        st = np.column_stack([np.roll(y, dl), right])
    return O.peak_normalize(O.soft_saturate(st, drive), peak)


def post_cases(big):
    """(n, mode, dl, dr, theta, drive, scale of y).  Even n of 64 and 66 (the window wraps twice), 1026, a non-multiple
    of the 1024-sample tile, a large n, shifts near n, drive 0, an all-zero render, precomputed right channels."""
    s = 40 if big else 1
    return [
        (64, 1, 5, 9, 0.63, 1.0, 1.0),
        (66, 1, 65, 63, 0.9, 2.0, 3.0),
        (1026, 1, 24, 34, 0.45, 1.0, 1.0),
        (3000, 1, 2999, 2998, 0.9, 1.3, 0.8),
        (50000 * s, 1, 36, 50, 0.81, 1.0, 179.0),
        (4000, 1, 17, 21, 0.27, 0.0, 2.5),                 # drive 0: no clip
        (3002, 1, 7, 9, 0.5, 1.0, 0.0),                    # all zeros
        (2048, 0, 0, 0, 0.0, 1.05, 1.2),
        (1025, 2, 1024, 0, 0.0, 1.0, 1.0),                 # odd n: right channel supplied in rbuf
        (4096, 2, 4000, 0, 0.0, 0.7, 0.5),
    ]


def check_post(dev, precision, big=False):
    api, real = _abi.Api(dev.lib, precision), _real(precision)
    rng = np.random.default_rng(13)
    cases = post_cases(big)
    recs, ys, rbufs, frames, at = [], [], [], GAP, GAP
    mono_parts, mono_n = [], GAP
    layout = []
    for n, mode, dl, dr, theta, drive, scale in cases:
        y = rng.standard_normal(n) * scale
        rb = rng.standard_normal(n) * scale if mode == 2 else None
        y_at = mono_n
        mono_n += n + GAP
        rb_at = 0
        if mode:
            rb_at = mono_n
            mono_n += n + GAP
        r = np.zeros(1, np.dtype(_abi.PostRender))
        coef = tables.bessel_coeffs(theta) if mode == 1 else np.zeros(2 * _abi.POST_K + 1)
        r[0] = (y_at, frames, rb_at, n, mode, dl, dr, drive, 1.0 / np.tanh(drive) if drive > 0 else 1.0, 0.98, coef)
        recs.append(r[0])
        layout.append((y_at, rb_at, frames))
        ys.append(y)
        rbufs.append(rb)
        frames += n + GAP
    mono = np.full(mono_n, X_SENTINEL)
    for (y_at, rb_at, _), y, rb in zip(layout, ys, rbufs):
        mono[y_at:y_at + len(y)] = y
        if rb is not None:
            mono[rb_at:rb_at + len(rb)] = rb
    rec = np.array(recs, dtype=np.dtype(_abi.PostRender))
    d_rec = dev.upload(rec)
    d_mono = dev.upload(mono.astype(real))
    maxbits = dev.zeros(len(rec), np.uint64)
    out = dev.upload(np.full(2 * frames, np.nan, np.float32))
    max_n = max(c[0] for c in cases)
    with LaunchLog(dev) as log:
        assert api.ms_post(dev.ptr(d_rec), len(rec), max_n, dev.ptr(d_mono), dev.ptr(maxbits), dev.ptr(out), dev.stream_ptr()) == 0, \
            dev.lib.ms_last_error()
    assert {"PostMaxK", "PostWriteK"} <= log.base(), sorted(log.base())
    o = _fetch(dev, out, np.float32, 2 * frames).reshape(-1, 2)
    m = _fetch(dev, d_mono, real, mono_n).astype(np.float64)
    errors = {}
    gaps = np.ones(len(o), bool)
    for (n, mode, dl, dr, theta, drive, scale), (y_at, rb_at, fr), y, rb in zip(cases, layout, ys, rbufs):
        gaps[fr:fr + n] = False
        yq = _as_ref(y, precision)
        got = o[fr:fr + n].astype(np.float64)
        tag = "n=%d mode=%d dl=%d dr=%d drive=%g" % (n, mode, dl, dr, drive)
        assert not np.any(np.isnan(got)), tag
        if scale == 0.0:
            assert np.all(got == 0.0), tag
            errors[tag] = 0.0
            continue
        if mode == 1:                                        # the right channel the max pass left at rbuf
            r_dev = m[rb_at:rb_at + n]
            r_fft = rotate_right(yq, dr, theta)
            r_bes = bessel_right(yq, dr, tables.bessel_coeffs(theta))
            sc = float(np.max(np.abs(yq)))
            e_r = max(float(np.max(np.abs(r_dev - r_fft))), float(np.max(np.abs(r_dev - r_bes)))) / sc
            errors[tag + " right"] = e_r
            assert e_r < POST_R_TOL[precision], (tag, "right channel", e_r)
        want = post_reference(yq, mode, dl, dr, theta, drive, 0.98, None if rb is None else _as_ref(rb, precision))
        e = float(np.max(np.abs(got - want)))
        errors[tag] = e
        # plus the right channel's own error (bounded above) times the largest slope of clip + normalise: at a zero
        # crossing tanh has unit slope, so a float32 right channel of a loud render moves the output by eps * peak
        mx = float(np.max(np.abs(yq)))
        slope = 0.98 * (drive / np.tanh(drive * mx) if drive > 0 else 1.0 / mx)
        tol = POST_OUT_TOL[precision] + (POST_R_TOL[precision] * mx * slope if mode == 1 else 0.0)
        assert e < tol, (tag, precision, e, tol, np.unravel_index(int(np.argmax(np.abs(got - want))), got.shape))
    assert np.all(np.isnan(o[gaps])), "write outside every render's frames"
    return errors


# ---- 4. in situ: each stage of real renders on the device's own input (BatchRenderer.run(mark=...)) ----------------------
def check_in_situ(dev, params_list, precision="f64"):
    """Runs the batch with the production schedule (no launch hook) and, at the stage marks, reads the device's mono
    planes: plane A after overlap_add against OLA + ADSR of the device's own grains, plane B after the FIR against
    reflection_cloud + short_ir_convolve of plane A, the float32 output against the post chain of plane B.  Every
    comparison starts from the device's own stage input, so none depends on how well the reference determines the
    grains.  Returns per-render errors."""
    br = engine.BatchRenderer(params_list, device=dev, precision=precision)
    t = br.tables
    real = br.real
    snap = {}

    def mark(name):
        if name == "overlap_add":
            snap["pool"] = _fetch(dev, br.pool, real, t.pool_n).astype(np.float64)
            snap["A"] = _fetch(dev, br.mono, real, t.mono_n).astype(np.float64)
        elif name == "fir_overlap_save":
            snap["B"] = _fetch(dev, br.mono, real, t.mono_n).astype(np.float64)
    try:
        br.run(mark=mark)
        dev.synchronize()
        fir_by_x = {int(f["x"]): f for f in t.fir}
        errs = []
        for r, p in enumerate(params_list):
            rr = t.ola_r[r]
            at, n = int(rr["out"]), int(rr["out_n"])
            mix = np.zeros(n)
            for e in t.ola_e[int(rr["ev_begin"]):int(rr["ev_end"])]:
                st, ln, g = int(e["start"]), int(e["len"]), int(e["grain"])
                mix[st:st + ln] += float(real(e["amp"])) * snap["pool"][g:g + ln]
            mix *= O.adsr_envelope(n, int(p["base_sr"]), float(p["env_a"]), float(p["env_d"]), float(p["env_s"]), float(p["env_r"]),
                                   float(p["env_curve"]))
            plane_a = snap["A"][at:at + n]
            e_ola = _rel(plane_a, mix)
            assert e_ola < OLA_TOL[precision], (r, "overlap-add", e_ola)
            y = plane_a
            e_fir = None
            ir = p.get("_ir_audio")
            wants_fir = bool(p["er_cloud_on"]) or (bool(p["space_ir_on"]) and ir is not None)
            assert wants_fir == (at in fir_by_x), (r, "FIR planned", wants_fir)
            if wants_fir:
                want = plane_a
                if p["er_cloud_on"]:
                    want = O.reflection_cloud(want, int(p["base_sr"]), int(p["er_taps"]), float(p["er_max_ms"]), int(p["seed"]))
                if p["space_ir_on"] and ir is not None:
                    want = O.short_ir_convolve(want, ir[:int(p["space_ir_max_samps"])])
                f = fir_by_x[at]
                y = snap["B"][int(f["y"]):int(f["y"]) + n]
                e_fir = _rel(y, want)
                assert e_fir < FIR_TOL[precision], (r, "FIR", e_fir)
            if p["stereo_on"]:
                st = O.stereo_diffuse(y, int(p["base_sr"]), float(p["stereo_width"]))
            else:
                st = np.column_stack([y, y])
            want = O.peak_normalize(O.soft_saturate(st, float(p["sat_drive"])), float(p["peak"]))
            e_post = float(np.max(np.abs(br.output(r).astype(np.float64) - want)))
            assert e_post < POST_OUT_TOL[precision], (r, "post", e_post)
            errs.append(dict(n=n, ola=e_ola, fir=e_fir, post=e_post, peak_pre_clip=float(np.max(np.abs(y)))))
        return errs
    finally:
        br.close()
