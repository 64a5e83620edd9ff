"""Host planner: turns a Microsound parameter dict into the flat, integer-exact plan the kernels consume.

Everything `render()` decides with Python scalars stays on the host and is decided the same way
the reference decides it (SURVEY.md Appendix C): Python `round()` (half-to-even) for every index,
numpy's own PCG64 Generators for every scalar draw (event times, amplitudes, grain offsets,
reflection taps, dust impulses), float64 for every threshold that selects a branch.  The bulk
arithmetic (normal noise, FFTs, overlap-add, convolution) is what goes to the GPU.

Reference lines are cited as M:<line> = microsound_0.2.1/main_v2.py.
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field
from typing import List, Optional

import numpy as np

from . import _abi
from .configs import BASIC_MODES

DESIGN_SR_CAP = 30_000_000          # M:597, M:646
IR_TAP_CAP = 8192                   # M:443: default of the optional key `space_ir_tap_cap`
IR_TAP_LIMIT = 1 << 21              # most IR taps the FIR stage takes (ms_fir_*: 10 s at 192 kHz)
EXPORT_RATIO_LIMIT = 640            # largest up or down of `export_sr` / base_sr in lowest terms (filter of 12801 taps)

MODE_GAUSS, MODE_DUST, MODE_NOISE, MODE_SKEW, MODE_RES, MODE_PLAIN, MODE_WAVELET, MODE_IRFRAG, MODE_SCANLINE, MODE_SILENT, MODE_CHAOS, MODE_STICK = range(12)
WAVELET_FLOOR = 128                 # M:319
_MODE_ID = {m: i for i, m in enumerate(BASIC_MODES)}


# --------------------------------------------------------------------------- breakpoint lanes (M:452-482)
_BP_CACHE = {}


def parse_breakpoints(text):
    """M:452-467.  Cached per text: a sweep repeats the same four lane strings thousands of times."""
    hit = _BP_CACHE.get(text)
    if hit is None:
        if len(_BP_CACHE) > 1024:
            _BP_CACHE.clear()
        hit = _BP_CACHE[text] = tuple(_parse_breakpoints(text))
    return list(hit)


def _parse_breakpoints(text):
    pts = []
    for part in (text or "").strip().split(","):
        part = part.strip()
        if not part or ":" not in part:
            continue
        t, v = part.split(":")               # "a:b:c" raises ValueError like the reference (M:461 is outside its try)
        try:
            pts.append((float(t.strip()), float(v.strip())))
        except Exception:
            continue
    pts.sort(key=lambda p: p[0])
    return pts


def eval_breakpoints(pts, t, default):
    if not pts:
        return default
    if t <= pts[0][0]:
        return pts[0][1]
    if t >= pts[-1][0]:
        return pts[-1][1]
    for (t0, v0), (t1, v1) in zip(pts[:-1], pts[1:]):
        if t0 <= t <= t1:
            a = (t - t0) / max(1e-12, t1 - t0)
            return (1 - a) * v0 + a * v1
    return default


# --------------------------------------------------------------------------- event field (M:507-558)
def generate_event_times(process, dur_s, rate, seed, cluster_size=6, cluster_spread_ms=25.0,
                         hawkes_gain=0.6, hawkes_decay_s=0.25):
    if process == "Single" or rate <= 0:
        return [0.0]                      # (the reference seeds a generator first; it is never drawn from)
    rng = np.random.default_rng(int(seed) + 9999)
    times = []
    if process == "Poisson":
        t = 0.0
        while t < dur_s:
            t += rng.exponential(1.0 / rate)
            if t < dur_s:
                times.append(t)
    elif process == "Clustered":
        parents, t = [], 0.0
        parent_rate = max(0.1, rate / max(1, cluster_size))
        while t < dur_s:
            t += rng.exponential(1.0 / parent_rate)
            if t < dur_s:
                parents.append(t)
        spread = cluster_spread_ms / 1000.0
        for p in parents:
            k = int(max(1, round(rng.uniform(0.6, 1.4) * cluster_size)))
            for _ in range(k):
                tt = p + rng.normal(0.0, spread)
                if 0.0 <= tt < dur_s:
                    times.append(tt)
        times.sort()
    elif process == "Hawkes":
        dt, activity = 0.002, 0.0
        decay = math.exp(-dt / max(1e-6, hawkes_decay_s))
        for i in range(int(math.ceil(dur_s / dt))):
            activity *= decay
            p = min(0.95, (rate + hawkes_gain * activity * rate) * dt)
            if rng.random() < p:
                times.append(i * dt + rng.uniform(0, dt))
                activity += 1.0
    return times


# --------------------------------------------------------------------------- spectral masks
def _edge():
    return _abi.BandEdge(0.0, 0.0, 0.0, 0.0, 0, 0, 0, 0)


def lowpass_edge(sr, cutoff, roll):
    """Mask of lowpass_fft (M:43-58) as a falling skirt."""
    nyq = 0.5 * sr
    fc = float(min(max(cutoff, 1.0), nyq))            # np.clip (M:44)
    width = float(max(0.0, roll))
    e = _edge()
    if width <= 0:
        e.hi_mode, e.hi_f0, e.hi_f1 = 1, fc, fc
    else:
        e.hi_mode, e.hi_f0, e.hi_f1 = 2, fc, min(nyq, fc + width)
    return e


def bandpass_edge(sr, lo, hi, roll):
    """Mask of bandpass_fft (M:64-100)."""
    lo = max(0.0, float(lo))
    hi = max(lo, float(hi))
    nyq = 0.5 * sr
    hi = min(hi, nyq)
    e = _edge()
    if hi <= 0:
        e.zero = 1
        return e
    width = float(max(0.0, roll))
    if lo > 0:
        if width <= 0:
            e.lo_mode, e.lo_f0, e.lo_f1 = 1, lo, lo
        else:
            e.lo_mode, e.lo_f0, e.lo_f1 = 2, max(0.0, lo - width), lo
    if hi < nyq:
        if width <= 0:
            e.hi_mode, e.hi_f0, e.hi_f1 = 1, hi, hi
        else:
            e.hi_mode, e.hi_f0, e.hi_f1 = 2, hi, min(nyq, hi + width)
    return e


def bin_spacing(n, sr):
    """np.fft.rfftfreq(n, d=1/sr)[k] == k * bin_spacing (numpy computes val = 1.0/(n*d))."""
    return 1.0 / (n * (1.0 / sr))


def grain_spec_op(params, gen_sr, n, cutoff_gen, stretch, pre=True, post=True, keep=False, mb=True):
    """Spectral operator of one event: lowpass_fft -> fft_warp_power -> fft_partial_stretch -> unfold_multiband
    (M:690-727), or None when every stage is an identity (unless `keep`).  `pre` / `post` select the stages before
    (low-pass, warp) and after (stretch, multiband) the point where partial_lock_stretch sits."""
    op = _abi.SpecOp()
    op.kind = _abi.OP_GRAIN
    op.df = bin_spacing(n, gen_sr)
    op.factor = 1.0
    if not pre:
        params = dict(params, bandlimit_on=False, nl_warp_on=False)
    if not post:
        params, stretch = dict(params, unfold_mode="Classic reinterpret"), 1.0
    if not mb:
        params = dict(params, unfold_mode="Classic reinterpret")
    if params["bandlimit_on"] and n >= 8:
        op.lp_on = 1
        op.lp = lowpass_edge(gen_sr, cutoff_gen, float(params["bandlimit_roll_hz"]))
    if params["nl_warp_on"] and n >= 16:                               # fft_warp_power (M:103-115, called at M:694-695)
        op.warp_exp = 1.0 / max(1e-6, float(params["nl_warp_power"]))
    stretch = float(stretch)
    if n >= 16 and not abs(stretch - 1.0) < 1e-9:
        op.stretch_on = 1
        op.factor = stretch
    if params["unfold_mode"] != "Classic reinterpret" and n >= 8:
        b1, b2, b3 = float(params["mb_b1"]), float(params["mb_b2"]), float(params["mb_b3"])
        us = [float(params["mb_u1"]), float(params["mb_u2"]), float(params["mb_u3"])]
        roll = float(params["mb_roll"])
        op.n_bands = 3
        for i, ((lo, hi), u) in enumerate(zip([(0.0, b1), (b1, b2), (b2, b3)], us)):
            op.mb[i] = bandpass_edge(gen_sr, lo * u, hi * u, roll)
    if not (op.lp_on or op.stretch_on or op.n_bands or op.warp_exp) and not keep:
        return None
    return op


def tilt_spec_op(n, gen_sr, tilt_db_per_oct):
    """Spectral shaping of tilted_noise (M:227-232): (f/f[1])**alpha with f[0] := f[1]."""
    op = _abi.SpecOp()
    op.kind = _abi.OP_TILT
    op.df = bin_spacing(n, gen_sr)
    op.alpha = math.log(10.0 ** (tilt_db_per_oct / 20.0), 2.0)
    return op


# --------------------------------------------------------------------------- plan records
@dataclass
class EventPlan:
    index: int
    t0: float
    amp: float
    ufac: float
    gen_sr: int
    n: int
    seed: int
    mode: int
    cutoff_gen: float
    stretch: float
    start: int
    offset: int = 0
    length: int = 0
    placed: bool = False
    spec: Optional[object] = None           # _abi.SpecOp or None
    plock: Optional[tuple] = None           # (factor, top_n, neigh, pre-operator) when partial_lock_stretch is active
    cep: Optional[tuple] = None             # (factor, pre-operator, operator of its last inverse) when cepstral_warp is active
    stick_noise: float = 0.0
    note: str = ""                          # generator note carried by the progress message (M:651, 682-684, 758)
    wg: Optional[np.ndarray] = None         # waveguide lines: float64 [L, 3] = delay in samples, loop gain, mix
    res: Optional[tuple] = None             # (modes float64 [K, 3] = f/sr, phase, weight ; decay per sample) for resonator_bank
    spec_b: Optional[object] = None         # multiband operator applied AFTER the resonator bank
    tilt: Optional[object] = None           # _abi.SpecOp for the tilted-noise modes
    dust_pos: Optional[np.ndarray] = None   # sorted unique impulse positions (int32)
    dust_val: Optional[np.ndarray] = None   # float64 values (last write wins, M:243)
    table: Optional[np.ndarray] = None      # IR fragment / image row to be resampled to n samples (float64)
    atoms: Optional[np.ndarray] = None      # wavelet atoms: float64 [count, 4] = f0/sr, 1/(sigma*sr), phase, weight
    atom_shift: Optional[np.ndarray] = None # int32 [count] circular shifts
    # mode constants (float64)
    f_over_sr: float = 0.0
    ring_decay: float = 0.0                 # 1 / (tau * gen_sr)
    env_decay: float = 0.0                  # 1 / (T * gen_sr) for the mode's exponential envelope
    sigma: int = 1
    fade: int = 8
    ker_len: int = 8


@dataclass
class RenderPlan:
    base_sr: int
    out_n: int
    design_sr_base: int
    events: List[EventPlan] = field(default_factory=list)
    adsr: tuple = (0, 0, 0, 1.0, 1.0)       # A, D, R samples, sustain, curve
    imprint: Optional[tuple] = None         # (amount, smooth) when SpectralImprint is active (M:625, 736-738)
    feedback: Optional[float] = None        # event_feedback_amt when event feedback is on (M:731-734)
    er_offs: Optional[np.ndarray] = None    # int32 tap delays (0 < off < out_n)
    er_gains: Optional[np.ndarray] = None   # float64
    ir: Optional[np.ndarray] = None         # float64 mono taps (<= space_ir_tap_cap) or None; with ir_r: the left channel
    ir_r: Optional[np.ndarray] = None       # space_ir_stereo with a two-column IR: float64 right-channel taps, else None
    stereo_on: bool = False
    stereo_dl: int = 0
    stereo_dr: int = 0
    stereo_theta: float = 0.0
    drive: float = 1.0
    peak: float = 0.98
    export: Optional[tuple] = None          # (up, down) of the optional key `export_sr`, or None: delivered at base_sr
    pcm: Optional[tuple] = None             # (bits, dither, seed mod 2^64) of the optional key `export_format`, or None: float32
    progress_msgs: list = field(default_factory=list)


def design_rate(base_sr, unfold):
    return int(min(max(int(round(base_sr * unfold)), base_sr), DESIGN_SR_CAP))     # np.clip on scalars (M:597, M:646)


def grain_length(gen_sr, micro_ms, floor=16):
    return int(max(floor, round(gen_sr * micro_ms / 1000.0)))      # M:221 (gen_basic, floor 16), M:319 (wavelet atoms, 128)


def plan_render(params) -> RenderPlan:
    """Scalar half of render() (M:589-646, 742-753, 760-781)."""
    cap = ir_tap_cap(params)
    stereo_ir = ir_stereo(params)
    export = export_ratio(params)
    pcm = pcm_format(params)
    ir_conv = conv_ir(params)
    base_sr = int(params["base_sr"])
    out_dur = float(params["out_dur_s"])
    out_n = int(max(1, round(out_dur * base_sr)))
    base_unfold = max(1.0, float(params["time_unfold"]))
    rp = RenderPlan(base_sr=base_sr, out_n=out_n, design_sr_base=design_rate(base_sr, base_unfold))

    lanes = [parse_breakpoints(params[k]) for k in ("bp_density", "bp_unfold", "bp_cutoff", "bp_stretch")]
    rate = float(params["grains_per_sec"])
    times = generate_event_times(params["event_process"], out_dur, rate, int(params["seed"]),
                                 int(params["cluster_size"]), float(params["cluster_spread_ms"]),
                                 float(params["hawkes_gain"]), float(params["hawkes_decay_s"]))
    times = times[:int(params["max_grains"])]
    rng = np.random.default_rng(int(params["seed"]) + 123456)
    seed = int(params["seed"])
    micro_ms = float(params["micro_ms"])
    micro_s = micro_ms / 1000.0
    spread = float(params["grain_amp_rand"])
    gmode = params["gen_mode"]
    dust_density = tilt = ring_hz = ring_decay_ms = 0.0
    ir_audio, img_gray = params.get("_ir_audio"), params.get("_img_gray")
    digest = params.get("_ir_digest")          # pooled batches ship the IR pre-digested (digest_params) instead of `_ir_audio`
    frag_src = None
    floor = 16
    note = ""
    if gmode == "Wavelet atoms":
        mode, floor = MODE_WAVELET, WAVELET_FLOOR
    elif gmode == "Crackle / corona":
        mode = MODE_DUST                       # same device kernel as the dust mode: sparse impulses * exp kernel, no fades
    elif gmode == "IR fragment":               # M:335-337: silence of gen_basic's length when no IR is loaded
        if digest is not None:
            frag_src = digest["frag"]
        elif ir_audio is not None and np.asarray(ir_audio).size >= 32:                # M:335
            frag_src = _mono64(ir_audio)
        mode, floor = (MODE_SILENT, 16) if frag_src is None else (MODE_IRFRAG, 64)
        note = "No IR loaded" if frag_src is None else "IR fragment"                  # M:336, 348
    elif gmode == "Image scanline":
        mode, floor = (MODE_SILENT if img_gray is None else MODE_SCANLINE), 64
        note = "No image loaded" if img_gray is None else ""                          # M:354 (else: the scan line, per event)
    elif gmode == "Micro-chaos":
        mode, floor = MODE_CHAOS, 64
    elif gmode == "Stick–slip friction":
        mode, floor = MODE_STICK, 64
    elif gmode in _MODE_ID:
        mode = _MODE_ID[gmode]
        dust_density, tilt = float(params["dust_density"]), float(params["noise_tilt"])
        ring_hz, ring_decay_ms = float(params["ring_hz"]), float(params["ring_decay_ms"])
    else:       # unknown generator string: M:686
        mode, dust_density, tilt, ring_hz, ring_decay_ms = MODE_NOISE, 0.01, -3.0, 4000.0, 12.0
    offset_on = bool(params["grain_offset_on"])
    max_off = int(round((float(params["grain_offset_max_ms"]) / 1000.0) * base_sr)) if offset_on else 0
    bl_default = float(params["bandlimit_out_hz"])
    st_default = float(params["partial_stretch"])

    for i, t0 in enumerate(times):
        dens = eval_breakpoints(lanes[0], t0, rate)
        ufac = eval_breakpoints(lanes[1], t0, base_unfold)
        cutoff_out = eval_breakpoints(lanes[2], t0, bl_default)
        stretch = eval_breakpoints(lanes[3], t0, st_default)
        amp = 1.0
        if rate > 0:
            amp *= min(max(dens / max(1e-6, rate), 0.15), 4.0)          # np.clip (M:641)
        amp *= rng.uniform(1.0 - spread, 1.0 + spread)
        ufac = max(1.0, float(ufac))
        sr_evt = design_rate(base_sr, ufac)
        n = grain_length(sr_evt, micro_ms, floor)
        ev = EventPlan(index=i, t0=t0, amp=float(amp), ufac=ufac, gen_sr=sr_evt, n=n, seed=seed + i, mode=mode,
                       cutoff_gen=cutoff_out * ufac, stretch=float(stretch), start=int(round(t0 * base_sr)), note=note)
        if ev.start < out_n:
            if offset_on and max_off > 0:
                ev.offset = int(rng.integers(0, max(1, min(max_off, n))))
            ev.length = max(0, min(out_n - ev.start, n - ev.offset))
            ev.placed = ev.length > 0
        res_on = bool(params["res_bank_on"]) and n >= 32                 # M:372
        wg_on = bool(params["wg_on"]) and n >= 64                        # M:389
        mb_here = not (res_on or wg_on)                                  # the multiband unfold follows them (M:719-727)
        if params["cep_warp_on"] and n >= 64:
            # M:696-697: cepstral_warp sits between low-pass / power warp and the stretch; its three elementwise steps
            # run between transforms of their own, the stage's inverse applies what follows (stretch + multiband) --
            # unless an active partial lock follows: then the inverse is plain and the lock stage takes over from there
            pl_active = bool(params["partial_lock_on"]) and not abs(ev.stretch - 1.0) < 1e-9
            pre = grain_spec_op(params, sr_evt, n, ev.cutoff_gen, 1.0, post=False, keep=True)
            if pl_active:
                ident = grain_spec_op(params, sr_evt, n, ev.cutoff_gen, 1.0, pre=False, post=False, keep=True)
                ev.cep = (float(params["cep_factor"]), pre, ident)
                ev.plock = (ev.stretch, int(params["pl_top_n"]), int(params["pl_neigh"]), ident)
                ev.spec = grain_spec_op(params, sr_evt, n, ev.cutoff_gen, 1.0, pre=False, keep=True, mb=mb_here)
            else:
                ev.spec = grain_spec_op(params, sr_evt, n, ev.cutoff_gen, 1.0 if params["partial_lock_on"] else ev.stretch, pre=False,
                                        keep=True, mb=mb_here)
                ev.cep = (float(params["cep_factor"]), pre, ev.spec)
        elif params["partial_lock_on"]:
            # M:699-702: partial_lock_stretch REPLACES fft_partial_stretch; it is the identity for n < 64 or a factor of 1
            if n >= 64 and not abs(ev.stretch - 1.0) < 1e-9:
                ev.plock = (ev.stretch, int(params["pl_top_n"]), int(params["pl_neigh"]),
                            grain_spec_op(params, sr_evt, n, ev.cutoff_gen, 1.0, post=False, keep=True))
                ev.spec = grain_spec_op(params, sr_evt, n, ev.cutoff_gen, 1.0, pre=False, keep=True, mb=mb_here)
            else:
                ev.spec = grain_spec_op(params, sr_evt, n, ev.cutoff_gen, 1.0, mb=mb_here)
        else:
            ev.spec = grain_spec_op(params, sr_evt, n, ev.cutoff_gen, ev.stretch, mb=mb_here)
        if res_on:
            ev.res = _plan_resonator(params, seed + i, sr_evt)
        if wg_on:
            ev.wg = _plan_waveguide(params, seed + i, sr_evt)
        if res_on or wg_on:
            ev.spec_b = grain_spec_op(params, sr_evt, n, ev.cutoff_gen, 1.0, pre=False)       # multiband only, or None
        ev.fade = max(8, int(0.01 * n))
        if mode == MODE_GAUSS:
            ev.sigma = max(1, int(0.0025 * n))
        elif gmode == "Crackle / corona":
            _plan_crackle(ev, float(params["crackle_alpha"]), float(params["crackle_density"]), int(params["crackle_kernel"]))
        elif mode == MODE_DUST:
            _plan_dust(ev, dust_density)
        elif mode == MODE_IRFRAG:
            _plan_ir_fragment(ev, frag_src)
        elif mode == MODE_SCANLINE:
            _plan_scanline(ev, img_gray)
        elif mode == MODE_STICK:               # M:283-301: threshold, build, decay, noise ride in the mode constants
            ev.f_over_sr, ev.ring_decay = float(params["ss_threshold"]), float(params["ss_build"])
            ev.env_decay, ev.stick_noise = float(params["ss_decay"]), float(params["ss_noise"])
            ev.fade = 0
        elif mode == MODE_CHAOS:               # M:303-315: r, gate, y0 = (seed % 10000) / 10000 ride in the mode constants
            ev.f_over_sr, ev.ring_decay = float(params["chaos_r"]), float(params["chaos_gate"])
            ev.env_decay = (int(ev.seed) % 10000) / 10000.0
            ev.ker_len, ev.fade = 48, 0
        elif mode in (MODE_NOISE, MODE_SKEW):
            ev.tilt = tilt_spec_op(n, sr_evt, tilt)
            T = max(1e-6, micro_s * (0.25 if mode == MODE_NOISE else 0.2))
            ev.env_decay = 1.0 / (T * sr_evt)
        elif mode == MODE_WAVELET:
            _plan_wavelet(ev, micro_ms, float(params["wav_base_hz"]), int(params["wav_count"]), float(params["wav_spread"]))
        elif mode == MODE_RES:
            ev.f_over_sr = max(10.0, ring_hz) / sr_evt
            ev.ring_decay = 1.0 / (max(1e-6, ring_decay_ms / 1000.0) * sr_evt)
            ev.env_decay = 1.0 / (max(1e-6, micro_s * 0.15) * sr_evt)
        rp.events.append(ev)

    a = max(0, int(round(base_sr * float(params["env_a"]) / 1000.0)))
    d = max(0, int(round(base_sr * float(params["env_d"]) / 1000.0)))
    r = max(0, int(round(base_sr * float(params["env_r"]) / 1000.0)))
    rp.adsr = (a, d, r, float(min(max(float(params["env_s"]), 0.0), 1.0)), float(max(1e-6, float(params["env_curve"]))))

    if params["event_feedback_on"]:
        rp.feedback = float(params["event_feedback_amt"])
    if params["spectral_imprint_on"]:
        rp.imprint = (float(params["spectral_imprint_amt"]), float(params["spectral_imprint_smooth"]))
    if params["er_cloud_on"]:
        offs, gains = reflection_taps(base_sr, int(params["er_taps"]), float(params["er_max_ms"]), seed)
        keep = (offs > 0) & (offs < out_n)
        rp.er_offs, rp.er_gains = offs[keep].astype(np.int32), gains[keep]
    if params["space_ir_on"]:
        if digest is not None:
            rp.ir, rp.ir_r = digest["taps"], digest.get("taps_r")
        elif ir_conv is not None:
            rp.ir, rp.ir_r = ir_pair(ir_conv, int(params["space_ir_max_samps"]), cap, stereo_ir)
    if params["stereo_on"] and out_n >= 64:   # M:426: shorter outputs are duplicated
        w = float(min(max(float(params["stereo_width"]), 0.0), 1.0))
        rp.stereo_on = True
        rp.stereo_dl = int(round((1 + 7 * w) * 0.0005 * base_sr))
        rp.stereo_dr = int(round((1 + 9 * w) * 0.0007 * base_sr))
        rp.stereo_theta = w * 0.9
    rp.drive = float(params["sat_drive"])
    rp.peak = float(params["peak"])
    rp.export = export
    if pcm is not None:
        rp.pcm = pcm + (seed % (1 << 64),)
    return rp


_TAPS_CACHE = {}


def array_signature(a):
    """Cheap identity-and-content key of an array-valued parameter (`_ir_audio`, `_img_gray`) for the planner's caches:
    the object, its shape / dtype, and a checksum over 64 strided samples plus the last one -- so an array edited IN PLACE
    between two renders is seen as new (the reference keeps no caches: whatever the array holds at call time is used)."""
    if a is None:
        return None
    a = np.asarray(a)
    flat = a.reshape(-1)
    step = max(1, flat.size // 64)
    return (id(a), a.shape, a.dtype.str, float(np.sum(flat[::step], dtype=np.float64)), float(flat[-1]) if flat.size else 0.0)


def ir_tap_cap(params):
    """The optional key `space_ir_tap_cap`: how many rows of the IR convolve_ir_short keeps (M:443 keeps 8192, the
    default).  An int >= 1, or None for no cap beyond `space_ir_max_samps`.  Caps above 8192 are an EXTENSION of the
    reference: the FIR stage then runs its partitioned route, checked against float64 convolution."""
    cap = params.get("space_ir_tap_cap", IR_TAP_CAP)
    if cap is None:
        return None
    if isinstance(cap, (bool, np.bool_)) or not isinstance(cap, (int, np.integer)) or cap < 1:
        raise ValueError(f"space_ir_tap_cap must be an int >= 1 or None, not {cap!r}")
    return int(cap)


def ir_stereo(params):
    """The optional key `space_ir_stereo` (EXTENSION; the reference mixes every IR to mono, M:438-445): True convolves
    the render with each channel of a two-column IR separately (`ir_pair`).  Only a bool (numpy's included) is taken."""
    on = params.get("space_ir_stereo", False)
    if not isinstance(on, (bool, np.bool_)):
        raise ValueError(f"space_ir_stereo must be a bool, not {on!r}")
    return bool(on)


def export_ratio(params):
    """The optional key `export_sr` (EXTENSION; the reference delivers every render at base_sr): the rate the output is
    resampled to after the normalisation, as scipy.signal.resample_poly(x, up, down) does it.  Returns (up, down) in
    lowest terms, or None when the key is absent, None or equal to int(base_sr).  Only an int >= 1 (numpy's included, not
    a bool) is taken, with up and down at most EXPORT_RATIO_LIMIT."""
    sr = params.get("export_sr", None)
    if sr is None:
        return None
    if isinstance(sr, (bool, np.bool_)) or not isinstance(sr, (int, np.integer)) or sr < 1:
        raise ValueError(f"export_sr must be an int >= 1 or None, not {sr!r}")
    base, sr = int(params["base_sr"]), int(sr)
    if sr == base:
        return None
    g = math.gcd(base, sr)
    up, down = sr // g, base // g
    if max(up, down) > EXPORT_RATIO_LIMIT:
        raise ValueError(f"export_sr {sr} from base_sr {base} is the ratio {up}/{down}: up and down must be at most "
                         f"{EXPORT_RATIO_LIMIT}")
    return up, down


IR_RESAMPLED = "_ir_resampled"      # private key: the IR at base_sr under `space_ir_sr` (engine.resolve_ir_rate puts it there)


def ir_rate(params):
    """The optional key `space_ir_sr` (EXTENSION; the reference plays the IR at base_sr whatever its file rate): the rate
    of `_ir_audio`.  The convolution then reads scipy.signal.resample_poly(ir, up, down) of every column, resampled to
    base_sr on the device (engine.resolve_ir_rate), and the tap keys count rows of that.  Returns (up, down) in lowest
    terms, or None when the key is absent, None or equal to int(base_sr).  Only an int >= 1 (numpy's included, not a
    bool) is taken, with up and down at most EXPORT_RATIO_LIMIT."""
    sr = params.get("space_ir_sr", None)
    if sr is None:
        return None
    if isinstance(sr, (bool, np.bool_)) or not isinstance(sr, (int, np.integer)) or sr < 1:
        raise ValueError(f"space_ir_sr must be an int >= 1 or None, not {sr!r}")
    base, sr = int(params["base_sr"]), int(sr)
    if sr == base:
        return None
    g = math.gcd(base, sr)
    up, down = base // g, sr // g
    if max(up, down) > EXPORT_RATIO_LIMIT:
        raise ValueError(f"space_ir_sr {sr} to base_sr {base} is the ratio {up}/{down}: up and down must be at most "
                         f"{EXPORT_RATIO_LIMIT}")
    return up, down


def ir_rate_rows(params):
    """Rows of the resampled IR the convolution can read: min(space_ir_max_samps, max(cap, 8)) -- the "< 8 values" test
    sees the slice before the cut to `space_ir_tap_cap`, so at least 8 rows are kept for it -- or None for all of them
    (a negative space_ir_max_samps slices from the end)."""
    max_samps, cap = int(params["space_ir_max_samps"]), ir_tap_cap(params)
    if max_samps < 0:
        return None
    return max_samps if cap is None else min(max_samps, max(cap, 8))


def conv_ir(params):
    """The impulse response the convolution reads: `_ir_audio`, or under `space_ir_sr` (with the IR on) its resampled rows
    at IR_RESAMPLED.  The planners never touch the device: a render whose IR has not been resampled is refused."""
    ir = params.get("_ir_audio")
    if ir_rate(params) is None or ir is None or not params["space_ir_on"]:
        return ir
    h = params.get(IR_RESAMPLED)
    if h is None:
        raise ValueError("space_ir_sr: the impulse response has not been resampled to base_sr "
                         "(engine.resolve_ir_rate runs before planning)")
    return h


def export_frames(n, ratio):
    """Frames of a render of n frames at base_sr after the export resampler: ceil(n up / down)."""
    return n if ratio is None else -(-n * ratio[0] // ratio[1])


PCM_FORMATS = {"pcm16": 16, "pcm24": 24}


def pcm_format(params):
    """The optional keys `export_format` and `export_dither` (EXTENSION; the reference returns float samples): integer PCM
    quantised on the GPU after everything else (include/microsound_b200.h, ms_post_pcm).  Returns (bits, dither) -- bits 16
    or 24 for "pcm16" / "pcm24", dither 1 for TPDF dither (the default), 0 without -- or None for float32 output (the key
    absent, None or "float32"; `export_dither` is then not looked at).  Any other value raises ValueError."""
    fmt = params.get("export_format", None)
    if fmt is None or isinstance(fmt, str) and fmt == "float32":
        return None
    bits = PCM_FORMATS.get(fmt) if isinstance(fmt, str) else None
    if bits is None:
        raise ValueError(f"export_format must be None, 'float32', 'pcm16' or 'pcm24', not {fmt!r}")
    dither = params.get("export_dither", True)
    if not isinstance(dither, (bool, np.bool_)):
        raise ValueError(f"export_dither must be a bool, not {dither!r}")
    return bits, int(bool(dither))


def output_slots(n, bits=None):
    """8-byte slots of the output arena that n frames take: one float32 frame each, ceil(n / 2) for pcm16 and ceil(3 n / 4)
    for pcm24 (6 bytes a frame).  Every render starts on a slot."""
    return n if bits is None else (n + 1) // 2 if bits == 16 else (3 * n + 3) // 4


_PAIR_CACHE = {}


def ir_pair(ir, max_samps, cap=IR_TAP_CAP, stereo=False):
    """(left taps, right taps) of the IR: (`_ir_taps`, None) unless `stereo` and the IR has two columns; then the
    reference's slice, "< 8 values" test and cut to `cap` rows, and instead of the mono mix column 0 and column 1 as
    contiguous float64 arrays, each at most IR_TAP_LIMIT taps.  More than two columns raise ValueError.  Cached per IR
    object, so a sweep shares one pair of arrays (and one copy of each in the IR pool of its tables)."""
    a = np.asarray(ir)
    if stereo and (a.ndim > 2 or (a.ndim == 2 and a.shape[1] > 2)):
        raise ValueError(f"space_ir_stereo takes an impulse response of one or two channels, not shape {a.shape}")
    if not stereo or a.ndim < 2 or a.shape[1] == 1:
        return _ir_taps(ir, max_samps, cap), None
    key = (array_signature(ir), max_samps, cap)
    hit = _PAIR_CACHE.get(key)
    if hit is not None and hit[0] is ir:
        return hit[1]
    h = a[:max_samps]
    pair = (None, None)
    if h.size >= 8:                           # the reference's test: size counts both channels
        h = h if cap is None else h[:cap]
        if h.shape[0] > IR_TAP_LIMIT:
            raise ValueError(f"an impulse response of {h.shape[0]} taps per channel is outside the accelerated path "
                             f"(at most {IR_TAP_LIMIT}; lower space_ir_tap_cap or space_ir_max_samps)")
        pair = (np.array(h[:, 0], dtype=np.float64), np.array(h[:, 1], dtype=np.float64))
    if len(_PAIR_CACHE) > 64:
        _PAIR_CACHE.clear()
    _PAIR_CACHE[key] = (ir, pair)
    return pair


def _ir_taps(ir, max_samps, cap=IR_TAP_CAP):
    """convolve_ir_short's view of the IR (M:438-443): None if the slice has fewer than 8 values, else the
    float64 mono mix of its first `cap` rows (None: all of them).  Cached per IR object: a sweep shares one IR.
    More than IR_TAP_LIMIT kept taps raise ValueError: the FIR stage does not take them."""
    key = (array_signature(ir), max_samps, cap)
    hit = _TAPS_CACHE.get(key)
    if hit is not None and hit[0] is ir:
        return hit[1]
    h = np.asarray(ir)[:max_samps]
    taps = None
    if h.size >= 8:                           # size counts both channels of a 2-D IR
        h = (h if cap is None else h[:cap]).astype(np.float64)      # the mono mix is row-wise, so cut to `cap` rows first
        taps = h.mean(axis=1) if h.ndim > 1 else h
        if taps.size > IR_TAP_LIMIT:
            raise ValueError(f"an impulse response of {taps.size} taps is outside the accelerated path "
                             f"(at most {IR_TAP_LIMIT}; lower space_ir_tap_cap or space_ir_max_samps)")
    if len(_TAPS_CACHE) > 64:
        _TAPS_CACHE.clear()
    _TAPS_CACHE[key] = (ir, taps)
    return taps


def reflection_taps(sr, taps, max_ms, seed):
    """Delays in samples and gains of early_reflection_cloud (M:410-417)."""
    rng = np.random.default_rng(int(seed) + 202)
    delays = rng.uniform(0.3, max_ms, size=int(max(1, taps))) / 1000.0
    gains = rng.uniform(-1.0, 1.0, size=delays.size)
    gains *= np.exp(-delays * 42.0)
    offs = np.rint(delays * sr).astype(np.int64)      # np.rint is half-to-even like Python round()
    return offs, gains


def _plan_wavelet(ev, micro_ms, base_hz, count, spread):
    """Scalar draws of gen_wavelet_atoms (M:322-327) in the reference's stream order."""
    n = ev.n
    if grain_length(ev.gen_sr, micro_ms, 16) != n:
        # morlet_atom builds its atoms with gen_basic's length rule (M:166): shorter than the 128-sample grain here
        raise ValueError(f"operands could not be broadcast together with shapes ({n},) ({grain_length(ev.gen_sr, micro_ms, 16)},)")
    rng = np.random.default_rng(int(ev.seed))
    count = int(max(1, count))
    atoms = np.zeros((count, 4), dtype=np.float64)
    shifts = np.zeros(count, dtype=np.int32)
    for k in range(count):
        f0 = base_hz * (2.0 ** rng.uniform(-spread, spread))
        sigma_ms = max(0.03, micro_ms * rng.uniform(0.04, 0.18))
        phase = rng.uniform(0, 2 * np.pi)
        shifts[k] = int(rng.integers(-n // 8, n // 8))
        sigma = max(1e-9, sigma_ms / 1000.0)
        atoms[k] = (f0 / ev.gen_sr, 1.0 / (sigma * ev.gen_sr), phase, 1.0 / (1 + k * 0.6))
    ev.atoms, ev.atom_shift = atoms, shifts


def _plan_resonator(params, seed, sr):
    """Scalar draws of resonator_bank (M:370, 377-380)."""
    rng = np.random.default_rng(int(seed) + 321)
    modes = int(max(1, int(params["res_modes"])))
    f_min, f_max = float(params["res_fmin"]), float(params["res_fmax"])
    rows = np.zeros((modes, 3), dtype=np.float64)
    for k in range(modes):
        f = f_min * ((f_max / max(1.0, f_min)) ** (k / max(1, modes - 1)))
        f *= 2.0 ** rng.uniform(-0.02, 0.02)
        rows[k] = (f / sr, rng.uniform(0, 2 * np.pi), 1.0 / (1 + k * 0.35))
    tau = max(1e-6, float(params["res_decay_ms"]) / 1000.0)
    return rows, 1.0 / (tau * sr)


def _plan_waveguide(params, seed, sr):
    """Scalar draws of waveguide_splinters (M:387, 391-396)."""
    rng = np.random.default_rng(int(seed) + 777)
    lines = int(max(1, int(params["wg_lines"])))
    max_ms, fb = float(params["wg_max_ms"]), float(params["wg_fb"])
    rows = np.zeros((lines, 3), dtype=np.float64)
    for k in range(lines):
        d = int(max(1, round((rng.uniform(0.4, max_ms) / 1000.0) * sr)))
        g = fb * rng.uniform(0.6, 0.98)
        rows[k] = (d, g, rng.uniform(0.15, 0.45))
    return rows


def _plan_crackle(ev, alpha, density, kernel):
    """Scalar draws of gen_crackle (M:272-279): Pareto gaps -> impulse times; amplitudes on one sample add up."""
    rng = np.random.default_rng(int(ev.seed))
    n = ev.n
    times = np.cumsum(rng.pareto(alpha, int(max(8, density))))
    times = times[times < n].astype(int)
    dense = np.zeros(n, dtype=np.float64)
    for ti in times:
        dense[ti] += rng.uniform(-1, 1)
    pos = np.unique(times)
    ev.dust_pos, ev.dust_val = pos.astype(np.int32), dense[pos]
    ev.ker_len = max(8, int(kernel))
    ev.fade = 0                                  # gen_crackle has no fades


_MONO_CACHE = {}


def _mono64(ir):
    key = array_signature(ir)
    hit = _MONO_CACHE.get(key)
    if hit is None or hit[0] is not ir:
        src = np.asarray(ir).astype(np.float64)
        if src.ndim > 1:
            src = src.mean(axis=1)
        if len(_MONO_CACHE) > 16:
            _MONO_CACHE.clear()
        _MONO_CACHE[key] = hit = (ir, src)
    return hit[1]


def _plan_ir_fragment(ev, src):
    """gen_ir_fragment (M:333-348): the host draws the start and hands the 256-sample piece of the mono mix `src`
    (float64, full length) to the device."""
    rng = np.random.default_rng(int(ev.seed))
    start = int(rng.integers(0, max(1, src.size - 256)))
    ev.table = np.ascontiguousarray(src[start:start + 256])


def _plan_scanline(ev, img_gray):
    """gen_image_scanline (M:350-362): the host draws the row and centres it; the device resamples and smooths."""
    rng = np.random.default_rng(int(ev.seed))
    h, w = img_gray.shape
    y = int(rng.integers(0, h))
    ev.note = f"Image line y={y}"                                                   # M:362
    row = img_gray[y, :].astype(np.float64) / 255.0
    ev.table = (row - row.mean()) * 2.0
    ev.ker_len = 48


def _plan_dust(ev, density):
    """Dust impulses (M:240-244): the index/value draws happen on the host so the stream is numpy's."""
    rng = np.random.default_rng(int(ev.seed))
    n = ev.n
    k = int(max(1, round(density * n)))
    where = rng.integers(0, n, size=k)
    vals = rng.uniform(-1, 1, size=k)
    dense = np.zeros(n, dtype=np.float64)
    dense[where] = vals                                  # duplicates: last write wins
    hit = np.zeros(n, dtype=bool)
    hit[where] = True
    pos = np.flatnonzero(hit)                            # sorted unique positions
    ev.dust_pos = pos.astype(np.int32)
    ev.dust_val = dense[pos]
    ev.ker_len = max(8, int(0.01 * n))


# --------------------------------------------------------------------------- batch planning
def _slim_params(p):
    """Copy of a parameter dict for the planning workers: the impulse response is replaced by what the planner
    keeps of it -- `_ir_digest = {"taps": convolve_ir_short's view (M:439-443: float64 mono mix of the first
    min(space_ir_max_samps, space_ir_tap_cap) rows, None when that slice has fewer than 8 values), "frag": gen_ir_fragment's
    source (M:335-340: the float64 mono mix of the WHOLE response, None when it has fewer than 32 values), "taps_r": the
    right channel under space_ir_stereo (`ir_pair`; "taps" is then the left one), else None}` -- so a
    multi-second stereo IR is not pickled per render and both size tests are made on the original array.  Under
    `space_ir_sr` "taps" / "taps_r" come from the resampled IR (conv_ir) and "frag" from `_ir_audio`.  The
    digests are cached per IR object, so renders sharing an IR share the arrays (one pickle memo entry per piece)."""
    ir = p.get("_ir_audio")
    if ir is None or "_ir_digest" in p:
        return p
    q = dict(p)
    q["_ir_audio"] = None
    q.pop(IR_RESAMPLED, None)
    frag = None
    if p["gen_mode"] == "IR fragment" and np.asarray(ir).size >= 32:
        frag = _mono64(ir)
    taps, taps_r = ir_pair(conv_ir(p),int(p["space_ir_max_samps"]), ir_tap_cap(p), ir_stereo(p)) if p["space_ir_on"] else (None, None)
    q["_ir_digest"] = {"taps": taps, "taps_r": taps_r, "frag": frag}
    return q
