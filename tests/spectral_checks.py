"""Stage-level checks of the spectral engine (ms_spectral_*, ms_fft_pair_forward) against float64 references: every
transform route in both precisions, in both directions, with every spectral operator, at unaligned offsets between
sentinels, in mixed batches and through the split entry points.

Routes are read from the launch log (kernel names with their template arguments), never from a restatement of the
planner.  ROUTE_KERNELS lists the exact forward and inverse kernel sequence of each route.  The generic columns kernel
serves two routes with one instantiation: plain mixed-radix columns (smooth n, two passes) and generic in-tile Bluestein
columns (`B1 > 0`); a length that is not 2-3-5-smooth cannot be transformed by mixed-radix columns, so the observed
kernels plus the smoothness of n name the route.

The static in-tile Bluestein columns of 128 (`ColsK<..., 128>`, sb_id 1) are unreachable from the planner: they need
B1 = 128 (a co-factor F1 of 33..64) and 16 | F2.  Then F2 / 2 >= 16 is smooth too, and the co-factor 2 F1 with B1 = 256
costs 256 / (2 F1) per element against 1.4 * 128 / F1, with more rows per tile, so plan_mixed always takes it
(F2 = 16 alone would need n = 16 F1 <= 1024, below the mixed threshold).  The catalogue holds lengths of that shape
(3904 = 61 * 64, 4880 = 61 * 80) and asserts that no catalogued length takes the static 128 route.

Errors are relative to the larger reference peak of the pair, since the two signals of a job share one complex
transform: the smaller one carries eps times its partner's peak.  Worst cases measured (relative to that scale):
  block emulator: forward f64 1.5e-15, f32 5.8e-7;  inverse f64 2.4e-13 (power-warp cases, see WARP_TOL_PER_N; the
                  other operators stay near 1e-15), f32 1.1e-6;  batch against single-length results f64 1.0e-15,
                  f32 4.8e-7;  Z of the split entry points f64 1.1e-15, f32 5.1e-7
A grain paired with a +6 dB/oct tilt is reported separately ("grain/tilt pair"): relative to the grain's own peak its
error reaches 1.1e-3 in f32 (6.6e-12 in f64) on the emulator; relative to the tilt's peak it is at the level above.
Tolerances: f64 1e-13 (forward and inverse), f32 2e-6 forward, 6e-6 inverse."""
import ctypes as C

import numpy as np

from audio_suite_b200 import _abi, configs, plan
from oracle import microsound_np as O
from stage_checks import LaunchLog, _fetch, _real

FWD_TOL = {"f64": 1e-13, "f32": 2e-6}
INV_TOL = {"f64": 1e-13, "f32": 6e-6}
GAP = 37                          # sentinel samples between jobs; jobs start at odd offsets
SENTINEL = 1.0e3
# the power warp gathers at pos = (k / kmax) ** (1 / power) * kmax: one rounding of pow() moves pos by ~eps * kmax, so
# the warp cases hold their error to the tolerance plus 1e-16 * n (measured on the emulator: up to 1.4e-17 * n in f64)
WARP_TOL_PER_N = 1e-16


def inv_tol(precision, n, label):
    return INV_TOL[precision] + (WARP_TOL_PER_N * n if "warp" in label else 0.0)


SR = 48000 * 30                   # grain sample rate of the operator cases (df = SR / n)

# route -> (forward kernels of ms_fft_pair_forward, kernels of one ms_spectral_run with a hook set: forward, inverse)
_FWD2 = "RowsK<0, 0, 2>"
_INV2 = "RowsK<0, 0, 4>"
ROUTE_KERNELS = {
    "direct": (["RowsK<2, 0, 2>"], ["RowsK<4, 0, 4>"]),
    "two-pass": (["ColsK<2, 0, 1, 0>", _FWD2], ["SpecOpK", "ColsK<0, 0, 1, 0>", _INV2]),
    "warp-plain-256": (["ColsWarpPlainK<2, 0, 1>", _FWD2], ["SpecOpK", "ColsWarpPlainK<0, 0, 1>", _INV2]),
    "mixed-static-128": (["ColsK<2, 0, 1, 128>", _FWD2], ["SpecOpK", "ColsK<0, 0, 1, 128>", _INV2]),
    "mixed-warp-256": (["ColsWarpK<2, 0, 1>", _FWD2], ["SpecOpK", "ColsWarpK<0, 0, 1>", _INV2]),
    "mixed-warp-512": (["ColsWarp512K<2, 0, 1>", _FWD2], ["SpecOpK", "ColsWarp512K<0, 0, 1>", _INV2]),
    "mixed-static-1024": (["ColsK<2, 0, 1, 1024>", _FWD2], ["SpecOpK", "ColsK<0, 0, 1, 1024>", _INV2]),
    "bluestein": (["RowsK<3, 1, 3>"], ["RowsK<5, 1, 5>"]),
    "bluestein-2p": (["ColsK<3, 0, 1, 0>", "RowsK<0, 1, 0>", "ColsK<0, 3, 0, 0>"],
                     ["ColsK<5, 0, 1, 0>", "RowsK<0, 1, 0>", "ColsK<0, 5, 0, 0>"]),
}
# what a label means in the catalogue: "two-pass" split by smoothness (see the module docstring)
ROUTES = ["direct", "direct-2p", "mixed-generic", "warp-plain-256", "mixed-static-128", "mixed-warp-256", "mixed-warp-512",
          "mixed-static-1024", "bluestein", "bluestein-2p"]
REACHABLE = {
    "f32": {"direct", "direct-2p", "mixed-generic", "warp-plain-256", "bluestein", "bluestein-2p"},
    "f64": {"direct", "direct-2p", "mixed-generic", "warp-plain-256", "mixed-warp-256", "mixed-warp-512", "mixed-static-1024",
            "bluestein", "bluestein-2p"},
}


def smooth(n):
    for p in (2, 3, 5):
        while n % p == 0:
            n //= p
    return n == 1


# n -> (f32 route, f64 route).  MS_SMALL_MAX = MS_TILE_MAX = 8192 (f32) / 4096 (f64); mixed columns from n > SMALL_MAX / 2.
_CATALOGUE = {
    4096: ("direct", "direct"),                     # f64 SMALL_MAX; n / 256 = 16 but a power of two
    4320: ("direct", "direct-2p"),                  # the smooth length after 4096
    4608: ("direct", "warp-plain-256"),             # n / 256 = 18
    8192: ("direct", "direct-2p"),                  # f32 SMALL_MAX
    8640: ("direct-2p", "direct-2p"),               # the smooth length after 8192
    9216: ("warp-plain-256", "warp-plain-256"),     # n / 256 = 36
    16384: ("direct-2p", "direct-2p"),              # n / 256 = 64, a power of two: generic columns
    2047: ("bluestein", "bluestein"),               # non-smooth just below f64 SMALL_MAX / 2; f64 Bluestein M = 4096
    2049: ("bluestein", "bluestein-2p"),            # just above: f64 M = 8192, no smooth factor >= 16
    2050: ("bluestein", "mixed-generic"),           # 41 * 50, just above f64 SMALL_MAX / 2
    4093: ("bluestein", "bluestein-2p"),            # prime just below f32 SMALL_MAX / 2; f32 M = 8192
    4097: ("bluestein-2p", "bluestein-2p"),         # 17 * 241 just above: f32 M = 16384
    4100: ("mixed-generic", "mixed-generic"),       # 41 * 100, just above f32 SMALL_MAX / 2; 100 % 8 != 0 in f64
    4875: ("mixed-generic", "mixed-generic"),       # co-factor 13 * 3: B1 = 32 (f32)
    3250: ("bluestein", "mixed-generic"),           # B1 = 64 (f64)
    2115: ("bluestein", "mixed-generic"),           # 47 * 45: B1 = 128 with F2 odd
    4125: ("mixed-generic", "mixed-generic"),       # 33 * 125: B1 = 128 with F2 odd
    3904: ("bluestein", "mixed-warp-256"),          # 61 * 64: taken as 122 * 32 (B1 = 256), not static 128
    4880: ("mixed-generic", "mixed-warp-256"),      # 61 * 80: likewise
    4160: ("mixed-generic", "mixed-warp-256"),      # 65 * 64: co-factor 65, B1 = 256
    4128: ("mixed-generic", "mixed-warp-256"),      # 129 * 32: B1 = 256 (as 43 * 96)
    8128: ("mixed-generic", "mixed-warp-256"),      # 127 * 64: co-factor 127, B1 = 256
    2096: ("bluestein", "mixed-warp-512"),          # 131 * 16: co-factor 131, B1 = 512
    8032: ("mixed-generic", "mixed-warp-512"),      # 251 * 32: co-factor 251, B1 = 512
    2358: ("bluestein", "mixed-generic"),           # B1 = 512 with F2 % 4 != 0 (f64)
    4112: ("mixed-generic", "mixed-static-1024"),   # 257 * 16: co-factor 257, B1 = 1024
    4208: ("mixed-generic", "mixed-static-1024"),   # 263 * 16
    8144: ("mixed-generic", "mixed-static-1024"),   # 509 * 16: co-factor 509, B1 = 1024
    6425: ("mixed-generic", "mixed-generic"),       # B1 = 1024 with odd F2 (f64)
    8336: ("mixed-generic", "bluestein-2p"),        # 521 * 16: B1 = 2048 -- f32 only; f64 falls to Bluestein
    8208: ("mixed-generic", "mixed-warp-256"),      # 513 * 16 = 27 * 19 * 16: split at a co-factor of 19, not 513
    16385: ("bluestein-2p", "bluestein-2p"),        # M = 32768
}
# full size only (GPU): n / 256 at MS_TILE_MAX / 4 and beyond, the largest accepted Bluestein lengths (M = 2^22)
_CATALOGUE_BIG = {
    262144: ("direct-2p", "direct-2p"),             # n / 256 = 1024 = f64 TILE_MAX / 4, a power of two
    256000: ("warp-plain-256", "warp-plain-256"),   # n / 256 = 1000
    276480: ("warp-plain-256", "direct-2p"),        # n / 256 = 1080 > f64 TILE_MAX / 4
    518400: ("warp-plain-256", "direct-2p"),        # n / 256 = 2025 <= f32 TILE_MAX / 4 = 2048
    524288: ("direct-2p", "direct-2p"),             # n / 256 = 2048, a power of two
    83040: ("mixed-generic", "mixed-warp-512"),
    1048583: ("bluestein-2p", "bluestein-2p"),      # M = 2^22 (f64: F1 = 1024, F2 = 4096)
    2097143: ("bluestein-2p", "bluestein-2p"),      # the largest n with M = 2^22 and no smooth factor >= 16
}


def catalogue(big):
    """[(n, {precision: route})]: n = 1..64 exhaustively (direct if smooth, else one-kernel Bluestein), then the table."""
    out = [(n, {"f32": r, "f64": r}) for n in range(1, 65) for r in ["direct" if smooth(n) else "bluestein"]]
    tab = dict(_CATALOGUE)
    if big:
        tab.update(_CATALOGUE_BIG)
    out += [(n, {"f32": a, "f64": b}) for n, (a, b) in tab.items()]
    return out


def route_of(n, fwd, inv):
    """Route label of the observed kernel sequences (None when they match no route)."""
    for name, (f, i) in ROUTE_KERNELS.items():
        if fwd == f and inv == f + i:
            if name == "two-pass":
                return "direct-2p" if smooth(n) else "mixed-generic"
            return name
    return None


# ---- device helpers ------------------------------------------------------------------------------------------------------
def fft_pair(dev, precision, a, b):
    """ms_fft_pair_forward of (a, b); returns (Z, kernel names).  The workspace query prepares the plan first, so the
    log holds only the transform's own launches."""
    api, real = _abi.Api(dev.lib, precision), _real(precision)
    n = len(a)
    need = api.ms_fft_pair_workspace_bytes(n)
    assert need > 0, (n, dev.lib.ms_last_error())
    ws = dev.empty(need, np.uint8)
    da, db = dev.upload(np.asarray(a, real)), dev.upload(np.asarray(b, real))
    z = dev.empty(2 * n, real)
    with LaunchLog(dev) as log:
        rc = api.ms_fft_pair_forward(dev.ptr(da), dev.ptr(db), n, dev.ptr(z), dev.ptr(ws), need, dev.stream_ptr())
    assert rc == 0, dev.lib.ms_last_error()
    zz = _fetch(dev, z, real, 2 * n).astype(np.float64)
    return zz[0::2] + 1j * zz[1::2], log.names


def layout(specs, rng=None):
    """Jobs at odd offsets with GAP sentinel samples between them.  specs: [(n, op_a, op_b or None)] -> (records,
    [(in_a, in_b, out_a, out_b)], total length)."""
    recs, at, pos = [], [], 13
    for n, oa, ob in specs:
        j = _abi.SpecJob()
        j.n = n
        ia = pos
        pos += n + GAP
        ib = -1
        if ob is not None:
            ib = pos
            pos += n + GAP
        j.in_a, j.in_b, j.out_a, j.out_b = ia, ib, ia, ib
        j.op[0] = oa
        j.op[1] = ob if ob is not None else _abi.SpecOp()
        recs.append(j)
        at.append((ia, ib))
    return recs, at, pos


def spectral_apply(dev, precision, recs, src, log=True, runs=1):
    """One ms_spectral_apply over `recs`; dst starts as NaN.  Returns (list of dst per run, src after, kernel names)."""
    api, real = _abi.Api(dev.lib, precision), _real(precision)
    arr = (_abi.SpecJob * len(recs))(*recs)
    need = api.ms_spectral_workspace_bytes(C.addressof(arr), len(recs))
    assert need > 0, dev.lib.ms_last_error()
    ws = dev.empty(need, np.uint8)
    dsrc = dev.upload(np.asarray(src, real))
    outs, names = [], []
    for _ in range(runs):
        dst = dev.upload(np.full(len(src), np.nan, real))
        if log:
            with LaunchLog(dev) as lg:
                rc = api.ms_spectral_apply(C.addressof(arr), len(recs), dev.ptr(dsrc), dev.ptr(dst), dev.ptr(ws), need, dev.stream_ptr())
            names = lg.names
        else:
            rc = api.ms_spectral_apply(C.addressof(arr), len(recs), dev.ptr(dsrc), dev.ptr(dst), dev.ptr(ws), need, dev.stream_ptr())
        assert rc == 0, dev.lib.ms_last_error()
        outs.append(_fetch(dev, dst, real, len(src)).astype(np.float64))
    return outs, _fetch(dev, dsrc, real, len(src)).astype(np.float64), names


# ---- operators and their references --------------------------------------------------------------------------------------
def _params(**kw):
    p = configs.with_defaults()
    p.update(kw)
    return p


def grain_case(n, kind):
    """(params, stretch, op) of one OP_GRAIN variant; None when the planner would not build that operator at this n."""
    p, st = None, 1.0
    if kind == "lp-cos/stretch-up":
        p, st = _params(bandlimit_roll_hz=20000.0), 1.7
    elif kind == "lp-brick/stretch-down":
        p, st = _params(bandlimit_roll_hz=0.0), 0.5
    elif kind == "warp/on-kmax":                       # stretch on with factor 1: the gather of bin kmax lands on kmax
        p, st = _params(nl_warp_on=True, nl_warp_power=1.6, bandlimit_on=False), 1.0
    elif kind == "bands-zero-brick":                   # band 1 empty (u1 = 0), brick lower edges (roll 0)
        p, st = _params(bandlimit_on=False, unfold_mode="Multi-band unfold", mb_u1=0.0, mb_u2=30.0, mb_u3=20.0, mb_roll=0.0), 1.3
    elif kind == "bands-cos/lp":
        p, st = _params(unfold_mode="Multi-band unfold", mb_roll=4000.0), 0.77
    elif kind == "stretch-only":                       # no mask: bin kmax gathers a complex value (its imaginary part is dropped)
        p, st = _params(bandlimit_on=False), 1.3
    cut = 300000.0
    op = plan.grain_spec_op(p, SR, n, cut, st)
    if kind == "warp/on-kmax" and n >= 16:
        op.stretch_on, op.factor = 1, 1.0
    if op is None or (kind == "warp/on-kmax" and n < 16):
        return None
    return p, st, cut, op


def grain_reference(x, p, st, cut):
    """lowpass_fft -> fft_warp_power -> fft_partial_stretch -> unfold_multiband, as the oracle writes them."""
    g = x
    if p["bandlimit_on"]:
        g = O.fft_lowpass(g, SR, cut, roll=p["bandlimit_roll_hz"])
    if p["nl_warp_on"]:
        g = O.spectrum_power_warp(g, p["nl_warp_power"])
    g = O.spectrum_stretch(g, st)
    if p["unfold_mode"] != "Classic reinterpret":
        b1, b2, b3 = p["mb_b1"], p["mb_b2"], p["mb_b3"]
        g = O.multiband_unfold(g, SR, [(0, b1), (b1, b2), (b2, b3)], [p["mb_u1"], p["mb_u2"], p["mb_u3"]], p["mb_roll"])
    return g


def tilt_op(n, db):
    return plan.tilt_spec_op(n, SR, db)


def tilt_reference(x, alpha):
    spec = np.fft.rfft(x)
    k = np.arange(spec.size, dtype=np.float64)
    return np.fft.irfft(spec * np.maximum(k, 1.0) ** alpha, n=len(x))


def rot_op(theta):
    op = _abi.SpecOp()
    op.kind, op.alpha = _abi.OP_ROT, theta
    return op


def rot_reference(x, theta):
    """The right channel of stereo_diffuse without its shift, for odd and even n: kmax = n // 2 (rfft's last bin)."""
    spec = np.fft.rfft(x)
    k = np.arange(spec.size, dtype=np.float64)
    return np.fft.irfft(spec * np.exp(1j * theta * np.sin(2 * np.pi * k / max(1.0, k[-1]))), n=len(x))


def op_cases(n):
    """[(label, (op_a, ref_a), (op_b, ref_b) or None)] for one length: paired and unpaired jobs, different operators on
    a and b.  ref_*: x -> float64 reference."""
    none = (_abi.SpecOp(), lambda x: x)
    t6, tm = tilt_op(n, 6.0), tilt_op(n, -4.5)
    tilt6 = (t6, lambda x, a=t6.alpha: tilt_reference(x, a))
    tiltm = (tm, lambda x, a=tm.alpha: tilt_reference(x, a))
    rot = (rot_op(0.81), lambda x: rot_reference(x, 0.81))
    rot2 = (rot_op(0.27), lambda x: rot_reference(x, 0.27))
    grains = {}
    for kind in ("lp-cos/stretch-up", "lp-brick/stretch-down", "warp/on-kmax", "bands-zero-brick", "bands-cos/lp", "stretch-only"):
        g = grain_case(n, kind)
        if g is not None:
            p, st, cut, op = g
            grains[kind] = (op, lambda x, p=p, st=st, cut=cut: grain_reference(x, p, st, cut))
    cases = [("none", none, None), ("none/none", none, none), ("rot/tilt-", rot, tiltm), ("tilt+", tilt6, None),
             ("rot", rot2, None)]
    g = list(grains.items())
    if g:
        cases.append(("grain/tilt pair", g[0][1], tilt6))
    for i, (kind, gv) in enumerate(g):
        partner = [rot, none, g[(i + 1) % len(g)][1], None, rot2][i % 5]
        cases.append((kind, gv, partner))
    return cases


# ---- the checks ----------------------------------------------------------------------------------------------------------
def check_forward(dev, precision, n, rng):
    real = _real(precision)
    a, b = rng.standard_normal(n).astype(real), rng.standard_normal(n).astype(real)
    z, names = fft_pair(dev, precision, a, b)
    want = np.fft.fft(a.astype(np.float64) + 1j * b.astype(np.float64))
    err = float(np.max(np.abs(z - want)) / np.max(np.abs(want)))
    assert err < FWD_TOL[precision], (precision, n, "forward", err)
    return err, names


def run_inverse_cases(dev, precision, n, rng, runs=1):
    """Every operator case of `n` as one ms_spectral_apply (one length class).  Checks every job against its reference,
    the sentinel gaps of dst, and src.  Returns ({label: error}, kernel names, the per-job outputs)."""
    real = _real(precision)
    cases = op_cases(n)
    recs, at, total = layout([(n, ca[0], cb[0] if cb else None) for _, ca, cb in cases])
    src = np.full(total, SENTINEL)
    xs = []
    for (ia, ib), (_, ca, cb) in zip(at, cases):
        xa = rng.standard_normal(n) * rng.uniform(0.5, 2.0)
        src[ia:ia + n] = xa
        xb = None
        if cb is not None:
            xb = rng.standard_normal(n) * rng.uniform(0.5, 2.0)
            src[ib:ib + n] = xb
        xs.append((xa, xb))
    outs, src_after, names = spectral_apply(dev, precision, recs, src, runs=runs)
    srcq = src.astype(real).astype(np.float64)
    assert np.array_equal(src_after, srcq), (precision, n, "src modified")
    errors, per_job = {}, []
    written = np.zeros(total, bool)
    for (ia, ib), (label, ca, cb), (xa, xb) in zip(at, cases, xs):
        ra = ca[1](xa.astype(real).astype(np.float64))
        rb = cb[1](xb.astype(real).astype(np.float64)) if cb is not None else None
        sc = max(float(np.max(np.abs(ra))), float(np.max(np.abs(rb))) if rb is not None else 0.0, 1e-300)
        got_a = outs[0][ia:ia + n]
        e = float(np.max(np.abs(got_a - ra))) / sc
        written[ia:ia + n] = True
        job = [got_a]
        if rb is not None:
            got_b = outs[0][ib:ib + n]
            e = max(e, float(np.max(np.abs(got_b - rb))) / sc)
            written[ib:ib + n] = True
            job.append(got_b)
            if label == "grain/tilt pair":
                errors["grain/tilt pair: grain rel. own peak"] = float(np.max(np.abs(got_a - ra))) / max(1e-300, float(np.max(np.abs(ra))))
        errors[label] = e
        assert e < inv_tol(precision, n, label), (precision, n, label, e)
        per_job.append(job)
    assert np.all(np.isnan(outs[0][~written])), (precision, n, "write outside the jobs' outputs")
    for o in outs[1:]:
        assert np.array_equal(o, outs[0], equal_nan=True), (precision, n, "repeat run differs")
    return errors, names, per_job


def check_catalogue(dev, precision, big=False):
    """Each catalogued length alone: its route from the launch log (forward and inverse), the forward transform and
    every operator case.  Returns ({n: route}, worst errors)."""
    rng = np.random.default_rng(31 if precision == "f64" else 32)
    seen, worst, pair = {}, {"forward": 0.0, "inverse": 0.0}, 0.0
    for n, want in catalogue(big):
        ef, fwd = check_forward(dev, precision, n, rng)
        errs, names, _ = run_inverse_cases(dev, precision, n, rng)
        r = route_of(n, fwd, names)
        assert r == want[precision], (precision, n, "route", want[precision], fwd, names)
        seen[n] = r
        worst["forward"] = max(worst["forward"], ef)
        worst["inverse"] = max(worst["inverse"], max(v for k, v in errs.items() if not k.startswith("grain/tilt pair:")))
        pair = max(pair, errs.get("grain/tilt pair: grain rel. own peak", 0.0))
    worst["grain/tilt pair, grain rel. own peak"] = pair
    routes = set(seen.values())
    assert routes == REACHABLE[precision], (precision, sorted(REACHABLE[precision] - routes), sorted(routes - REACHABLE[precision]))
    assert "mixed-static-128" not in routes
    return seen, worst


def check_mixed_batch(dev, precision, big=False):
    """One ms_spectral_apply holding a length of every route (several jobs each), shuffled: every job equals its
    single-length result within the tolerance."""
    rng = np.random.default_rng(77)
    by_route = {}
    for n, want in catalogue(big):
        by_route.setdefault(want[precision], []).append(n)
    lengths = [ns[len(ns) // 2] for _, ns in sorted(by_route.items())]
    single = {}
    for n in lengths:
        single[n] = run_inverse_cases(dev, precision, n, np.random.default_rng(n))[2]
    # the same jobs (same inputs: the per-length generator replays), all lengths in one call, shuffled
    specs, refs, xs = [], [], []
    for n in lengths:
        r = np.random.default_rng(n)
        cases = op_cases(n)
        for k, (_, ca, cb) in enumerate(cases):
            xa = r.standard_normal(n) * r.uniform(0.5, 2.0)
            xb = r.standard_normal(n) * r.uniform(0.5, 2.0) if cb is not None else None
            specs.append((n, ca[0], cb[0] if cb else None))
            xs.append((xa, xb))
            refs.append(single[n][k])
    order = rng.permutation(len(specs))
    specs, xs, refs = [specs[i] for i in order], [xs[i] for i in order], [refs[i] for i in order]
    recs, at, total = layout(specs)
    src = np.full(total, SENTINEL)
    for (ia, ib), (xa, xb) in zip(at, xs):
        src[ia:ia + len(xa)] = xa
        if xb is not None:
            src[ib:ib + len(xb)] = xb
    (out,), src_after, _ = spectral_apply(dev, precision, recs, src)
    assert np.array_equal(src_after, src.astype(_real(precision)).astype(np.float64))
    worst, written = 0.0, np.zeros(total, bool)
    for (ia, ib), (n, _, _), ref in zip(at, specs, refs):
        got = [out[ia:ia + n]] + ([out[ib:ib + n]] if ib >= 0 else [])
        sc = max(float(np.max(np.abs(v))) for v in ref)
        e = max(float(np.max(np.abs(g - v))) for g, v in zip(got, ref)) / max(sc, 1e-300)
        written[ia:ia + n] = True
        if ib >= 0:
            written[ib:ib + n] = True
        worst = max(worst, e)
        assert e < inv_tol(precision, n, "warp"), (precision, n, "batch vs single", e)
    assert np.all(np.isnan(out[~written]))
    return {"lengths": lengths, "jobs": len(specs), "worst vs single": worst}


def check_split_entry_points(dev, precision, lengths):
    """ms_spectral_create -> forward -> Z through ms_spectral_z_table (== fft(a + i b)) -> inverse: bitwise equal to
    ms_spectral_apply of the same jobs."""
    api, real = _abi.Api(dev.lib, precision), _real(precision)
    rng = np.random.default_rng(5)
    specs = []
    for i, n in enumerate(lengths):
        g = grain_case(n, "lp-cos/stretch-up")
        specs.append((n, g[3] if g else rot_op(0.5), tilt_op(n, 3.0) if i % 2 == 0 else None))
    recs, at, total = layout(specs)
    src = np.full(total, SENTINEL)
    for (ia, ib), (n, _, _) in zip(at, specs):
        src[ia:ia + n] = rng.standard_normal(n)
        if ib >= 0:
            src[ib:ib + n] = rng.standard_normal(n)
    (want,), _, _ = spectral_apply(dev, precision, recs, src, log=False)
    arr = (_abi.SpecJob * len(recs))(*recs)
    need = api.ms_spectral_workspace_bytes(C.addressof(arr), len(recs))
    ws = dev.zeros(need, np.uint8)
    dsrc = dev.upload(src.astype(real))
    dst = dev.upload(np.full(total, np.nan, real))
    h = C.c_void_p()
    assert api.ms_spectral_create(C.addressof(arr), len(recs), dev.ptr(dsrc), dev.ptr(dst), dev.ptr(ws), need,
                                  dev.stream_ptr(), C.byref(h)) == 0, dev.lib.ms_last_error()
    try:
        assert api.ms_spectral_forward(h, dev.stream_ptr()) == 0, dev.lib.ms_last_error()
        zoff = (C.c_int64 * len(recs))()
        zbase = C.c_size_t()
        assert api.ms_spectral_z_table(h, zoff, C.byref(zbase)) == 0
        wsb = _fetch(dev, ws, np.uint8, need)
        cpx = np.complex64 if precision == "f32" else np.complex128
        isz = np.dtype(cpx).itemsize
        srcq = src.astype(real).astype(np.float64)
        worst = 0.0
        for k, ((ia, ib), (n, _, _)) in enumerate(zip(at, specs)):
            o = zbase.value + isz * zoff[k]
            z = wsb[o:o + isz * n].view(cpx).astype(np.complex128)
            x = srcq[ia:ia + n] + (1j * srcq[ib:ib + n] if ib >= 0 else 0.0)
            zr = np.fft.fft(x)
            e = float(np.max(np.abs(z - zr)) / np.max(np.abs(zr)))
            worst = max(worst, e)
            assert e < FWD_TOL[precision], (precision, n, "Z", e)
        assert api.ms_spectral_inverse(h, dev.stream_ptr()) == 0, dev.lib.ms_last_error()
        got = _fetch(dev, dst, real, total).astype(np.float64)
    finally:
        api.ms_spectral_destroy(h)
    assert np.array_equal(got, want, equal_nan=True), (precision, "split entry points differ from ms_spectral_apply")
    return worst


def check_refused(dev, precision, n):
    api = _abi.Api(dev.lib, precision)
    assert api.ms_fft_pair_workspace_bytes(n) == 0, (precision, n)
    msg = (dev.lib.ms_last_error() or b"").decode()
    assert "unsupported" in msg and str(n) in msg, msg
    return msg


def check_schedules(dev, precision, big=False):
    """A batch of every route of the precision (f64: nine length classes, more than the five side streams plus the
    caller's stream) run with a launch hook (serial schedule) and without (ms_spectral_run forks the classes onto side
    streams where it can): bitwise equal, and repeat runs bitwise equal."""
    by_route = {}
    for n, want in catalogue(big):
        by_route.setdefault(want[precision], []).append(n)
    rng = np.random.default_rng(3)
    specs = []
    for _, ns in sorted(by_route.items()):
        for n in ns[-2:]:
            for _, ca, cb in op_cases(n)[:4]:
                specs.append((n, ca[0], cb[0] if cb else None))
    specs = [specs[i] for i in rng.permutation(len(specs))]
    recs, at, total = layout(specs)
    src = np.full(total, SENTINEL)
    for (ia, ib), (n, _, _) in zip(at, specs):
        src[ia:ia + n] = rng.standard_normal(n)
        if ib >= 0:
            src[ib:ib + n] = rng.standard_normal(n)
    serial, _, names = spectral_apply(dev, precision, recs, src, log=True)
    forked, _, _ = spectral_apply(dev, precision, recs, src, log=False, runs=3)
    assert not np.any(np.isnan(serial[0][[i for ia, ib in at for i in (ia, ib) if i >= 0]]))
    for o in forked:
        assert np.array_equal(o, serial[0], equal_nan=True), (precision, "forked schedule differs from the serial one")
    return {"jobs": len(specs), "classes": len(by_route), "launches (serial)": len(names)}


def check_big_class(dev, precision, jobs=40000, n=60):
    """One length class of more jobs than one launch takes (32768): every job against its reference, repeat runs
    bitwise equal."""
    rng = np.random.default_rng(8)
    real = _real(precision)
    t = tilt_op(n, 6.0)
    specs = [(n, t if i % 3 == 0 else rot_op(0.5) if i % 3 == 1 else _abi.SpecOp(), _abi.SpecOp() if i % 2 else None)
             for i in range(jobs)]
    recs, at, total = layout(specs)
    src = np.full(total, SENTINEL)
    ia = np.array([a for a, _ in at])
    ib = np.array([b for _, b in at])
    idx_a = ia[:, None] + np.arange(n)
    src[idx_a] = rng.standard_normal((jobs, n))
    pb = ib >= 0
    idx_b = ib[pb][:, None] + np.arange(n)
    src[idx_b] = rng.standard_normal((int(pb.sum()), n))
    outs, _, _ = spectral_apply(dev, precision, recs, src, log=False, runs=2)
    assert np.array_equal(outs[0], outs[1], equal_nan=True), (precision, "repeat run differs")
    q = src.astype(real).astype(np.float64)
    xa = q[idx_a]
    spec = np.fft.rfft(xa, axis=1)
    k = np.arange(spec.shape[1], dtype=np.float64)
    mul = np.ones((jobs, spec.shape[1]), complex)
    kind = np.arange(jobs) % 3
    mul[kind == 0] = np.maximum(k, 1.0) ** t.alpha
    mul[kind == 1] = np.exp(1j * 0.5 * np.sin(2 * np.pi * k / k[-1]))
    ra = np.fft.irfft(spec * mul, n=n, axis=1)
    rb = q[idx_b]
    sc = np.maximum(np.max(np.abs(ra), axis=1), 0.0)
    sc[pb] = np.maximum(sc[pb], np.max(np.abs(rb), axis=1))
    ea = np.max(np.abs(outs[0][idx_a] - ra), axis=1) / sc
    eb = np.max(np.abs(outs[0][idx_b] - rb), axis=1) / sc[pb]
    worst = float(max(ea.max(), eb.max()))
    assert worst < INV_TOL[precision], (precision, "big class", worst, int(np.argmax(ea)))
    written = np.zeros(total, bool)
    written[idx_a] = True
    written[idx_b] = True
    assert np.all(np.isnan(outs[0][~written]))
    return worst
