"""Job tables: RenderPlans -> flat, relocatable numpy tables -> one merged batch.

`pack_chunk(plans)` lays a list of render plans out in chunk-local coordinates (every offset starts at
0) and returns plain numpy arrays, so chunks can be built by worker processes and pickled cheaply;
`merge_chunks` concatenates them and shifts every offset field (RELOC) by the chunk's base in its buffer.
`pair_jobs` / `single_jobs` turn spectral items into the device's job records (two signals of equal
length share one complex transform).  A single in-process chunk goes through exactly the same code.

Every table is a record array with the layout of its struct in include/microsound_b200.h (SpecItem:
`struct Item` of csrc/ms_hostplan.cpp), so it is uploaded as it stands.  Fields only the device
workspace can supply (the `z*` spectrum offsets, scratch offsets) stay 0 here and are filled on upload.

Buffers (offsets in elements): pool (real; per-event signals), mono (real; per chunk:
[OLA plane | FIR plane | right channels / odd-length scratch / right-channel FIR outputs]), out (float32 frames, at the
export rate of renders with `export_sr`), hpool (real; combined FIR taps), taps (reflection delays/gains), irs
(deduplicated IR taps), dust (impulses), bank (polyphase banks of the export resampler, one per ratio and chunk).
"""
from __future__ import annotations

import math
import os
from dataclasses import dataclass, field, fields

import numpy as np

from . import _abi, decimate, plan as P

_SPEC_OP_BYTES = np.dtype(_abi.SpecOp).itemsize
_SPEC_JOB = np.dtype(_abi.SpecJob)
_ZERO_OP = np.zeros(_SPEC_OP_BYTES, np.uint8)

# one spectral work item: a signal of n samples from pool[src] to pool[dst] through one operator
SPEC_ITEM = np.dtype([("n", np.int64), ("src", np.int64), ("dst", np.int64), ("op", np.uint8, (_SPEC_OP_BYTES,))])
# odd-length stereo: rolled copy of mono[y_at : y_at + n] by dr into mono[scratch]
ODD = np.dtype([("y_at", np.int64), ("scratch", np.int64), ("n", np.int64), ("dr", np.int64)])
# per render: pool offsets of the last event's raw and final grain (-1 if none), its length
LAST = np.dtype([("micro", np.int64), ("grain", np.int64), ("n", np.int64)])
# one event of a render with event feedback, processed rank by rank: feedback from the previous event's final grain
# (fb.dst = -1 at rank 0), then the imprint step (imp_item.dst = -1 when the imprint is off or the grain is short)
SEQ = np.dtype([("render", np.int64), ("rank", np.int64), ("fb", np.dtype(_abi.FeedbackEvt)),
                ("imp", np.dtype(_abi.ImprintStepEvt)), ("imp_item", SPEC_ITEM)])


def _recs(ctype, n):
    return np.zeros(n, dtype=np.dtype(ctype))


def _structs(ctype, rows):
    """ctypes structs -> record array of their bytes (padding included)."""
    return np.frombuffer(bytearray(b"".join(map(bytes, rows))), np.dtype(ctype)) if rows else _recs(ctype, 0)


def spec_items(rows):
    """[(n, src, dst, SpecOp or None)] -> SPEC_ITEM array"""
    return np.array([(n, s, d, _ZERO_OP if op is None else np.frombuffer(bytes(op), np.uint8)) for n, s, d, op in rows], SPEC_ITEM)


_BESSEL = {}


def bessel_coeffs(theta, K=_abi.POST_K):
    """J_m(theta), m = -K..K by the ascending series (theta <= 0.9 here).  exp(i theta sin(phi)) =
    sum_m J_m(theta) exp(i m phi): for even n the rotation of spectral_diffusion_stereo (main_v2.py:432-435)
    is exactly a (2K+1)-tap circular FIR with taps at even lags."""
    hit = _BESSEL.get(theta)
    if hit is not None:
        return hit
    out = np.zeros(2 * K + 1)
    for m in range(K + 1):
        s, k = 0.0, 0
        while True:
            term = (-1.0) ** k * (theta / 2.0) ** (2 * k + m) / (math.factorial(k) * math.factorial(k + m))
            s += term
            k += 1
            if abs(term) < 1e-22 or k > 40:
                break
        out[K + m] = s
        out[K - m] = s * (-1.0) ** m
    if len(_BESSEL) > 256:
        _BESSEL.clear()
    _BESSEL[theta] = out
    return out


def _empty(dtype, *shape):
    return field(default_factory=lambda: np.zeros((0,) + shape, dtype))


@dataclass
class Tables:
    sy1: np.ndarray = _empty(_abi.SynthEvt)
    sy2: np.ndarray = _empty(_abi.SynthEvt)
    ola_r: np.ndarray = _empty(_abi.OlaRender)
    env_reps: np.ndarray = _empty(_abi.OlaRender)    # one OlaRender per shared envelope table (its .env = table offset)
    env_n: int = 0
    ola_e: np.ndarray = _empty(_abi.OlaEvt)
    fir: np.ndarray = _empty(_abi.FirRender)
    post: np.ndarray = _empty(_abi.PostRender)
    tap_off: np.ndarray = _empty(np.int32)
    tap_gain: np.ndarray = _empty(np.float64)
    irs: np.ndarray = _empty(np.float64)
    dust_pos: np.ndarray = _empty(np.int32)
    dust_val: np.ndarray = _empty(np.float64)
    atoms: np.ndarray = _empty(np.float64, 4)        # wavelet atoms, float64 [N, 4]
    atom_shift: np.ndarray = _empty(np.int32)
    seq: np.ndarray = _empty(SEQ)                    # events of renders with event feedback, in render / event order
    wg: np.ndarray = _empty(_abi.WgEvt)
    wg_lines: np.ndarray = _empty(_abi.WgLine)
    res: np.ndarray = _empty(_abi.ResEvt)
    res_modes: np.ndarray = _empty(_abi.ResMode)
    post_grain: np.ndarray = _empty(SPEC_ITEM)       # spectral items applied after the resonator bank (multiband)
    cep: np.ndarray = _empty(_abi.CepEvt)            # cepstral warp (`pre` operator filled) ...
    cep_items: np.ndarray = _empty(SPEC_ITEM)        # ... and its outer forward / inverse transform
    plock: np.ndarray = _empty(_abi.PlockEvt)        # partial lock (`pre` operator filled) ...
    plock_items: np.ndarray = _empty(SPEC_ITEM)      # ... and its outer transforms
    imprint: np.ndarray = _empty(_abi.ImprintEvt)    # spectral imprint without feedback, in event order per render ...
    imprint_items: np.ndarray = _empty(SPEC_ITEM)
    imprint_r: np.ndarray = _empty(_abi.ImprintRender)
    tilt: np.ndarray = _empty(SPEC_ITEM)
    grain: np.ndarray = _empty(SPEC_ITEM)
    rot: np.ndarray = _empty(SPEC_ITEM)
    odd: np.ndarray = _empty(ODD)
    export: np.ndarray = _empty(_abi.ExportRender)   # renders with an export rate, in render order ...
    export_of: np.ndarray = _empty(np.int64)         # ... and their render indices
    bank: np.ndarray = _empty(np.float64)            # polyphase banks of the export resampler (decimate.polyphase_bank)
    pool_n: int = 0
    mono_n: int = 0
    frames: int = 0
    h_total: int = 0
    max_h: int = 0
    max_out_n: int = 0
    out_at: np.ndarray = _empty(np.int64)            # per render: first frame
    out_n: np.ndarray = _empty(np.int64)             # per render: frames (at the export rate, if any)
    y_at: np.ndarray = _empty(np.int64)
    last: np.ndarray = _empty(LAST)
    srs: np.ndarray = _empty(np.int64, 2)            # per render: base_sr, design_sr_base
    alg: dict = field(default_factory=dict)          # algorithmic element counts per stage (SURVEY 8d)


# Every offset field of the tables: (table, field) -> (buffer it indexes, whether -1 means "none" and stays -1).
# Field None: the table is a plain per-render array of offsets.
RELOC = {
    ("sy1", "out"): ("pool", False), ("sy1", "dust_begin"): ("dust", False), ("sy1", "atom_begin"): ("atoms", False),
    ("sy2", "out"): ("pool", False), ("sy2", "aux"): ("pool", False),
    ("ola_r", "out"): ("mono", False), ("ola_r", "ev_begin"): ("ola_e", False), ("ola_r", "ev_end"): ("ola_e", False),
    ("ola_r", "env"): ("env", True), ("env_reps", "env"): ("env", False),
    ("ola_e", "grain"): ("pool", False),
    ("fir", "ir"): ("irs", False), ("fir", "h"): ("h", False), ("fir", "tap_begin"): ("taps", False), ("fir", "tap_end"): ("taps", False),
    ("fir", "x"): ("mono", False), ("fir", "y"): ("mono", False),
    ("post", "y"): ("mono", False), ("post", "rbuf"): ("mono", False), ("post", "out"): ("frames", False),
    ("seq", "render"): ("renders", False), ("seq", "fb.cur"): ("pool", False), ("seq", "fb.prev"): ("pool", True),
    ("seq", "fb.dst"): ("pool", True), ("seq", "imp_item.src"): ("pool", False), ("seq", "imp_item.dst"): ("pool", True),
    ("wg", "src"): ("pool", False), ("wg", "dst"): ("pool", False), ("wg", "line_begin"): ("wg_lines", False),
    ("res", "src"): ("pool", False), ("res", "dst"): ("pool", False), ("res", "mode_begin"): ("res_modes", False),
    ("imprint_r", "ev_begin"): ("imprint", False), ("imprint_r", "ev_end"): ("imprint", False),
    ("odd", "y_at"): ("mono", False), ("odd", "scratch"): ("mono", False),
    ("out_at", None): ("frames", False), ("y_at", None): ("mono", False),
    ("export", "out"): ("frames", False), ("export", "out_end"): ("frames", False),
    ("export", "bank"): ("bank", False), ("export", "bank_end"): ("bank", False), ("export_of", None): ("renders", False),
    ("last", "micro"): ("pool", True), ("last", "grain"): ("pool", True),
}
for _t, _buf in (("tilt", "pool"), ("grain", "pool"), ("post_grain", "pool"), ("cep_items", "pool"), ("plock_items", "pool"),
                 ("imprint_items", "pool"), ("rot", "mono")):
    RELOC[(_t, "src")] = RELOC[(_t, "dst")] = (_buf, False)

# size of each buffer in a chunk: the base of the next chunk's offsets
BUFFERS = {
    "pool": lambda t: t.pool_n, "mono": lambda t: t.mono_n, "frames": lambda t: t.frames, "h": lambda t: t.h_total,
    "env": lambda t: t.env_n, "ola_e": lambda t: len(t.ola_e), "taps": lambda t: len(t.tap_off), "irs": lambda t: len(t.irs),
    "dust": lambda t: len(t.dust_pos), "atoms": lambda t: len(t.atom_shift), "res_modes": lambda t: len(t.res_modes),
    "wg_lines": lambda t: len(t.wg_lines), "imprint": lambda t: len(t.imprint), "renders": lambda t: len(t.post),
    "bank": lambda t: len(t.bank),
}


def column(arr, name):
    """arr["a"]["b"] for name "a.b"; arr itself for None."""
    for f in (name.split(".") if name else ()):
        arr = arr[f]
    return arr


def pack_chunk(plans) -> Tables:
    R = len(plans)
    n_evt = sum(len(rp.events) for rp in plans)
    sy1, sy2 = _recs(_abi.SynthEvt, n_evt), _recs(_abi.SynthEvt, n_evt)
    ola_r, post = _recs(_abi.OlaRender, R), _recs(_abi.PostRender, R)
    ola_e = []
    fir = []
    tilt, grain, rot, post_grain = [], [], [], []
    dust_pos, dust_val, n_dust = [], [], 0
    atoms, atom_shift, n_atoms = [], [], 0
    imprint, imprint_items, imprint_r = [], [], []
    plock, plock_items, cep, cep_items = [], [], [], []
    res, res_modes, n_modes = [], [], 0
    wg, wg_lines, n_lines = [], [], 0
    seq = []
    tap_off, tap_gain, n_taps = [], [], 0
    irs, ir_index, n_ir = [], {}, 0
    pool_n = mono_n = h_total = max_h = 0
    mono_at = []
    last = np.zeros(R, LAST)
    last[:] = (-1, -1, -1)
    fir_of, fir_r_of = {}, {}

    def ir_slot(h):
        """(offset, length) of taps `h` in the deduplicated IR pool"""
        nonlocal n_ir
        key = h.ctypes.data if h.flags.owndata else h.tobytes()
        hit = ir_index.get(key)
        if hit is None or (not isinstance(key, bytes) and hit[2] is not h):
            hit = ir_index[key] = (n_ir, h.size, h)
            irs.append(h)
            n_ir += h.size
        return hit
    alg = dict(synth=0, tilt_spectral=0, grain_spectral=0, overlap_add=0, fir_in=0, fir_taps=0, post=0)
    env_seen = {}
    e = 0
    for r, rp in enumerate(plans):
        a, d, rel, S, curve = rp.adsr
        n = rp.out_n
        if a > n:
            raise ValueError(f"could not broadcast input array from shape ({a},) into shape ({n},)")   # main_v2.py:182
        d_end = min(n, a + d) if d > 0 else a
        sus_end = max(d_end, n - rel)
        ev_begin = len(ola_e)
        imp_begin = len(imprint)
        max_len = 0
        x_begin, x_end = n, 0
        prev_final, prev_n, rank = -1, 0, 0
        for ev in rp.events:
            st = np.random.PCG64(ev.seed).state["state"]
            s_hi, s_lo = st["state"] >> 64, st["state"] & 0xFFFFFFFFFFFFFFFF
            i_hi, i_lo = st["inc"] >> 64, st["inc"] & 0xFFFFFFFFFFFFFFFF
            micro = pool_n
            pool_n += ev.n
            out1, mode2, aux2, dust_b, dust_c = micro, -1, 0, 0, 0
            atom_b, atom_c = 0, 0
            alg["synth"] += ev.n
            if ev.mode == P.MODE_WAVELET:
                atom_b, atom_c = n_atoms, len(ev.atom_shift)
                atoms.append(ev.atoms)
                atom_shift.append(ev.atom_shift)
                n_atoms += atom_c
            if ev.mode == P.MODE_DUST:
                dust_b, dust_c = n_dust, len(ev.dust_pos)
                dust_pos.append(ev.dust_pos)
                dust_val.append(ev.dust_val)
                n_dust += dust_c
            elif ev.mode in (P.MODE_IRFRAG, P.MODE_SCANLINE):        # table rides in the impulse arrays (positions unused)
                dust_b, dust_c = n_dust, len(ev.table)
                dust_pos.append(np.zeros(dust_c, np.int32))
                dust_val.append(ev.table)
                n_dust += dust_c
                if ev.mode == P.MODE_SCANLINE:
                    aux2 = pool_n                                     # windowed, unsmoothed line
                    pool_n += ev.n
            elif ev.mode in (P.MODE_CHAOS, P.MODE_STICK):
                aux2 = pool_n                                         # gated logistic-map samples / the event's normals
                pool_n += ev.n
            elif ev.mode in (P.MODE_NOISE, P.MODE_SKEW):
                raw, tilted = pool_n, pool_n + ev.n
                pool_n += 2 * ev.n
                out1, mode2, aux2 = raw, ev.mode, tilted
                tilt.append((ev.n, raw, tilted, ev.tilt))
                alg["tilt_spectral"] += 2 * ev.n
            common = (s_hi, s_lo, i_hi, i_lo, ev.n)
            tail = (ev.fade, ev.sigma)
            inv_fade = 1.0 / ev.fade if ev.fade > 0 else (ev.stick_noise if ev.mode == P.MODE_STICK else 0.0)
            sy1[e] = common + (ev.mode,) + tail + (out1, ev.f_over_sr, inv_fade, ev.ring_decay, ev.env_decay,
                                                     dust_b, dust_c, ev.ker_len, aux2 if ev.mode in (P.MODE_SCANLINE, P.MODE_CHAOS, P.MODE_STICK) else 0,
                                                     atom_b, atom_c, 0)
            sy2[e] = common + (mode2,) + tail + (micro, ev.f_over_sr, inv_fade, ev.ring_decay, ev.env_decay,
                                                  0, 0, ev.ker_len, aux2, 0, 0, 0)
            g_at = micro
            if ev.cep is not None:
                g_at = pool_n
                pool_n += ev.n
                cep.append(_abi.CepEvt(n=ev.n, factor=ev.cep[0], pre=ev.cep[1]))
                cep_items.append((ev.n, micro, g_at, ev.cep[2]))
                alg["grain_spectral"] += 2 * ev.n * (1 + int(ev.cep[1].lp_on) + (1 if ev.cep[1].warp_exp else 0)
                                                     + int(ev.cep[2].stretch_on) + (1 if ev.cep[2].n_bands else 0))
            if ev.plock is not None:
                pl_src = g_at                      # the raw transient, or the cepstrally warped grain
                g_at = pool_n
                pool_n += ev.n
                plock.append(_abi.PlockEvt(n=ev.n, top_n=ev.plock[1], neigh=ev.plock[2], factor=ev.plock[0], pre=ev.plock[3]))
                plock_items.append((ev.n, pl_src, g_at, ev.spec))
                alg["grain_spectral"] += 2 * ev.n * (1 + int(ev.plock[3].lp_on) + (1 if ev.plock[3].warp_exp else 0) + (1 if ev.spec.n_bands else 0))
            elif ev.cep is None and ev.spec is not None:
                g_at = pool_n
                pool_n += ev.n
                grain.append((ev.n, micro, g_at, ev.spec))
                alg["grain_spectral"] += 2 * ev.n * (int(ev.spec.lp_on) + int(ev.spec.stretch_on) + (1 if ev.spec.n_bands else 0)
                                                     + (1 if ev.spec.warp_exp else 0))
            if ev.res is not None:
                r_at = pool_n                      # the resonator reads the grain so far and writes a new one
                pool_n += ev.n
                res.append(_abi.ResEvt(src=g_at, dst=r_at, n=ev.n, mode_begin=n_modes, mode_count=len(ev.res[0]), decay=ev.res[1]))
                res_modes.append(ev.res[0])
                n_modes += len(ev.res[0])
                g_at = r_at
            if ev.wg is not None:
                w_at = pool_n                      # the combs run in place on a copy of the grain so far
                pool_n += ev.n
                wg.append(_abi.WgEvt(src=g_at, dst=w_at, n=ev.n, line_begin=n_lines, line_count=len(ev.wg)))
                wg_lines.append(ev.wg)
                n_lines += len(ev.wg)
                g_at = w_at
            if ev.res is not None or ev.wg is not None:
                if ev.spec_b is not None:
                    b_at = pool_n
                    pool_n += ev.n
                    post_grain.append((ev.n, g_at, b_at, ev.spec_b))
                    alg["grain_spectral"] += 2 * ev.n
                    g_at = b_at
            last[r] = (micro, g_at, ev.n)
            if rp.feedback is not None:
                # M:731-740: feedback from the previous event's FINAL grain, then the imprint, rank by rank
                cur, fb_dst, imp_dst = g_at, -1, -1
                if prev_final >= 0:
                    fb_dst = pool_n
                    pool_n += ev.n
                    g_at = fb_dst
                imp_on = rp.imprint is not None and ev.n >= 64 and rp.imprint[0] > 0
                if imp_on:
                    imp_dst = pool_n
                    pool_n += ev.n
                amount, smooth = rp.imprint if imp_on else (0.0, 0.0)
                seq.append((r, rank, (cur, prev_final, fb_dst, ev.n, prev_n, rp.feedback), (0, ev.n, 0, amount, smooth),
                            (ev.n, g_at, imp_dst, _ZERO_OP)))       # the imprint reads the fed-back grain, or the grain itself
                g_at = imp_dst if imp_on else g_at
                prev_final, prev_n, rank = g_at, ev.n, rank + 1
            elif rp.imprint is not None and ev.n >= 64 and rp.imprint[0] > 0:         # M:570: short grains / amount <= 0 pass through
                src = g_at
                g_at = pool_n                      # imprinted grain (grain_last keeps the grain before it, M:729)
                pool_n += ev.n
                imprint.append(_abi.ImprintEvt(n=ev.n))
                imprint_items.append((ev.n, src, g_at, None))
            if ev.placed:
                ola_e.append((g_at + ev.offset, ev.start, ev.length, ev.amp))
                max_len = max(max_len, ev.length)
                # (no "grain[0] == 0" shortcut here: that holds for a raw gen_basic transient only, not after the
                #  band-limit / stretch / multiband operators or for the generators without a fade-in)
                x_begin = min(x_begin, ev.start)
                x_end = max(x_end, ev.start + ev.length)
                alg["overlap_add"] += ev.length
            e += 1
        if len(imprint) > imp_begin:
            imprint_r.append(_abi.ImprintRender(imp_begin, len(imprint), *rp.imprint))
        env_key = (n, a, d_end, sus_end, 1 if (rel > 0 and n > sus_end) else 0,
                   1.0 / a if a > 0 else 0.0, 1.0 / (d_end - a) if d_end > a else 0.0,
                   1.0 / (n - sus_end - 1) if n - sus_end > 1 else 0.0, S, curve)
        env_seen.setdefault(env_key, []).append(r)
        ola_r[r] = (mono_n, n, ev_begin, len(ola_e), max_len) + env_key[1:] + (-1,)
        alg["overlap_add"] += n
        # FIR: reflection cloud folded into the impulse response
        has_er = rp.er_offs is not None and rp.er_offs.size > 0
        if has_er or rp.ir is not None:
            if rp.ir is not None:
                hit = ir_slot(rp.ir)
                alg["fir_in"] += 2 * n
                alg["fir_taps"] += rp.ir.size
            else:
                hit = ir_index.get(b"delta")
                if hit is None:
                    hit = ir_index[b"delta"] = (n_ir, 1, None)
                    irs.append(np.ones(1))
                    n_ir += 1
            ir_at, ir_len = hit[0], hit[1]
            t0 = n_taps
            h_len = ir_len
            if has_er:
                if rp.er_offs.size > 4096:
                    raise ValueError("er_taps > 4096 is outside the accelerated path")
                tap_off.append(rp.er_offs)
                tap_gain.append(rp.er_gains)
                n_taps += rp.er_offs.size
                h_len = ir_len + int(rp.er_offs.max())
                alg["fir_in"] += 2 * n
            if x_begin == 0 and a > 0:
                x_begin = 1                      # env[0] = 0 ** curve = 0 (main_v2.py:181-182)
            fir_of[r] = len(fir)
            fir.append((ir_at, ir_len, h_len, h_total, t0, n_taps, mono_n, 0, n, min(x_begin, x_end), x_end, 0))
            if rp.ir_r is not None:              # space_ir_stereo: the right channel's row differs only in `ir` and `y`
                fir_r_of[r] = len(fir)
                fir.append((ir_slot(rp.ir_r)[0],) + fir[-1][1:])
                alg["fir_in"] += 2 * n * (2 if has_er else 1)
                alg["fir_taps"] += rp.ir_r.size
            h_total += h_len
            max_h = max(max_h, h_len)
        mono_at.append(mono_n)
        mono_n += n
    plane = mono_n
    extra = 0
    frames = 0
    odd = []
    out_at, out_n, y_at = np.zeros(R, np.int64), np.zeros(R, np.int64), np.zeros(R, np.int64)
    export, export_of, banks, bank_at, n_bank = [], [], [], {}, 0
    fir_arr = np.array(fir, np.dtype(_abi.FirRender))
    for r, rp in enumerate(plans):
        n = rp.out_n
        y = mono_at[r]
        if r in fir_of:
            y = plane + mono_at[r]
            fir_arr[fir_of[r]]["y"] = y
        mode, dl, dr, rbuf = 0, 0, 0, 0
        coef = np.zeros(2 * _abi.POST_K + 1)
        if r in fir_r_of:
            # space_ir_stereo: the right channel's FIR output yR opens the render's extra region, the right channel
            # proper is made from it: [yR | right] (even n, Bessel FIR in the max pass), [yR | rolled copy | right]
            # (odd n), or [yR] itself (no stereo diffusion)
            y_r = 2 * plane + extra
            fir_arr[fir_r_of[r]]["y"] = y_r
            extra += n
            if not rp.stereo_on:
                mode, rbuf = 2, y_r
            elif n % 2 == 0:
                mode, coef, rbuf, dl, dr = 3, bessel_coeffs(rp.stereo_theta), y_r + n, rp.stereo_dl, rp.stereo_dr
                extra += n
            else:
                mode, rbuf, dl, dr = 2, y_r + 2 * n, rp.stereo_dl, rp.stereo_dr
                odd.append((y_r, y_r + n, n, dr))
                op = _abi.SpecOp()
                op.kind, op.alpha = _abi.OP_ROT, rp.stereo_theta
                rot.append((n, y_r + n, y_r + 2 * n, op))
                extra += 2 * n
        elif rp.stereo_on:
            dl, dr = rp.stereo_dl, rp.stereo_dr
            if n % 2 == 0:
                mode, coef, rbuf = 1, bessel_coeffs(rp.stereo_theta), 2 * plane + extra     # right channel, written by the max pass
                extra += n
            else:
                mode, rbuf = 2, 2 * plane + extra + n                                        # [rolled copy | right channel]
                odd.append((y, 2 * plane + extra, n, dr))
                op = _abi.SpecOp()
                op.kind, op.alpha = _abi.OP_ROT, rp.stereo_theta
                rot.append((n, 2 * plane + extra, 2 * plane + extra + n, op))
                extra += 2 * n
        post[r] = (y, frames, rbuf, n, mode, dl, dr, rp.drive, 1.0 / math.tanh(rp.drive) if rp.drive > 0 else 1.0, rp.peak, coef)
        n_x = P.export_frames(n, rp.export)
        if rp.export is not None:                # export_sr: the output is resampled by up / down through the ratio's bank
            half, taps, bk = decimate.polyphase_bank(*rp.export)
            at = bank_at.get(rp.export)
            if at is None:
                at = bank_at[rp.export] = n_bank
                banks.append(bk.reshape(-1))
                n_bank += bk.size
            export.append((frames, frames + n_x, at, at + bk.size, rp.export + (half, taps)))
            export_of.append(r)
        out_at[r], out_n[r], y_at[r] = frames, n_x, y
        frames += n_x
        alg["post"] += n
    # envelopes shared by several renders are tabulated once (ms_adsr_tables) instead of one pow() per sample
    env_n = 0
    reps = []
    for key, members in env_seen.items():
        if len(members) >= 2:
            ola_r["env"][members] = env_n
            reps.append(ola_r[members[0]].copy())
            env_n += int(key[0])
    t = Tables()
    if reps:
        t.env_reps = np.array(reps, dtype=ola_r.dtype)
    t.env_n = env_n
    t.sy1, t.sy2, t.ola_r, t.post, t.fir = sy1, sy2, ola_r, post, fir_arr
    t.ola_e = np.array(ola_e, np.dtype(_abi.OlaEvt))
    for name, parts in (("tap_off", tap_off), ("tap_gain", tap_gain), ("irs", irs), ("dust_pos", dust_pos), ("dust_val", dust_val),
                        ("atoms", atoms), ("atom_shift", atom_shift)):
        if parts:
            setattr(t, name, np.concatenate(parts).astype(getattr(t, name).dtype))
    t.cep, t.cep_items = _structs(_abi.CepEvt, cep), spec_items(cep_items)
    t.plock, t.plock_items = _structs(_abi.PlockEvt, plock), spec_items(plock_items)
    t.res = _structs(_abi.ResEvt, res)
    if res_modes:
        t.res_modes = np.ascontiguousarray(np.concatenate(res_modes), np.float64).view(t.res_modes.dtype).reshape(-1)
    t.wg, t.wg_lines = _structs(_abi.WgEvt, wg), _recs(_abi.WgLine, n_lines)
    if wg_lines:
        lines = np.concatenate(wg_lines)
        t.wg_lines["d"], t.wg_lines["g"], t.wg_lines["mix"] = lines[:, 0], lines[:, 1], lines[:, 2]
    t.seq = np.array(seq, SEQ)
    t.imprint, t.imprint_items, t.imprint_r = _structs(_abi.ImprintEvt, imprint), spec_items(imprint_items), _structs(_abi.ImprintRender, imprint_r)
    t.tilt, t.grain, t.rot, t.post_grain = spec_items(tilt), spec_items(grain), spec_items(rot), spec_items(post_grain)
    t.odd = np.array(odd, ODD)
    if export:
        t.export, t.export_of = np.array(export, t.export.dtype), np.array(export_of, np.int64)
        t.bank = np.concatenate(banks)
    t.pool_n, t.mono_n, t.frames, t.h_total, t.max_h = pool_n, 2 * plane + extra, frames, h_total, max_h
    t.max_out_n = max((rp.out_n for rp in plans), default=0)
    t.out_at, t.out_n, t.y_at, t.last = out_at, out_n, y_at, last
    t.srs = np.asarray([(rp.base_sr, rp.design_sr_base) for rp in plans], np.int64).reshape(-1, 2)
    t.alg = alg
    return t


def merge_chunks(chunks) -> Tables:
    """One Tables of consecutive chunks: tables concatenated, offsets shifted by the chunk's base in their buffer.
    The chunks themselves are left as they are."""
    if len(chunks) == 1:
        return chunks[0]
    m = Tables()
    for f in fields(Tables):
        if f.name != "alg" and isinstance(getattr(m, f.name), np.ndarray):
            setattr(m, f.name, np.concatenate([getattr(c, f.name) for c in chunks]))
    bases = {buf: np.cumsum([0] + [size(c) for c in chunks[:-1]]) for buf, size in BUFFERS.items()}

    def shift(table, buf):
        return np.repeat(bases[buf], [len(getattr(c, table)) for c in chunks])
    for (table, name), (buf, keep_none) in RELOC.items():
        col, add = column(getattr(m, table), name), shift(table, buf)
        col += np.where(col >= 0, add, 0) if keep_none else add
    # sy1.aux is a pool offset only for these generators (the scratch they synthesise through); 0 for the others
    m.sy1["aux"] += np.where(np.isin(m.sy1["mode"], (P.MODE_SCANLINE, P.MODE_CHAOS, P.MODE_STICK)), shift("sy1", "pool"), 0)
    for k in ("pool_n", "mono_n", "frames", "h_total", "env_n"):
        setattr(m, k, sum(getattr(c, k) for c in chunks))
    m.max_h, m.max_out_n = max(c.max_h for c in chunks), max(c.max_out_n for c in chunks)
    for c in chunks:
        for k, v in c.alg.items():
            m.alg[k] = m.alg.get(k, 0) + v
    return m


def _op_bytes(jobs, i):
    """Raw bytes of jobs["op"][:, i] (SpecOp has nested structs: operators are copied as bytes)."""
    op0 = _SPEC_JOB.fields["op"][1] + i * _SPEC_OP_BYTES
    return jobs.view(np.uint8).reshape(len(jobs), _SPEC_JOB.itemsize)[:, op0:op0 + _SPEC_OP_BYTES]


def single_jobs(items):
    """SPEC_ITEM array -> one SpecJob per item, in item order (for stages that address each job's spectrum)."""
    jobs = np.zeros(len(items), _SPEC_JOB)
    jobs["n"], jobs["in_a"], jobs["out_a"], jobs["in_b"], jobs["out_b"] = items["n"], items["src"], items["dst"], -1, -1
    _op_bytes(jobs, 0)[:] = items["op"]
    return jobs


def pair_jobs(items):
    """SPEC_ITEM array -> SpecJob record array.  Two signals of equal n share one complex transform;
    the leftover of an odd group rides alone."""
    k = len(items)
    if k == 0:
        return np.zeros(0, _SPEC_JOB)
    items = items[np.argsort(items["n"], kind="stable")]
    n, src, dst, ops = items["n"], items["src"], items["dst"], items["op"]
    starts = np.flatnonzero(np.r_[True, n[1:] != n[:-1]])
    pos = np.arange(k) - np.repeat(starts, np.diff(np.r_[starts, k]))      # index inside its equal-n group
    first = pos % 2 == 0
    has_partner = np.zeros(k, bool)
    has_partner[:-1] = first[:-1] & (n[1:] == n[:-1]) & (pos[1:] == pos[:-1] + 1)
    a = np.flatnonzero(first)
    b = a + 1
    paired = has_partner[a]
    jobs = np.zeros(a.size, _SPEC_JOB)
    jobs["n"] = n[a]
    jobs["in_a"], jobs["out_a"] = src[a], dst[a]
    bb = np.where(paired, np.minimum(b, k - 1), 0)
    jobs["in_b"] = np.where(paired, src[bb], -1)
    jobs["out_b"] = np.where(paired, dst[bb], -1)
    _op_bytes(jobs, 0)[:] = ops[a]
    _op_bytes(jobs, 1)[:] = np.where(paired[:, None], ops[bb], _ZERO_OP[None, :])
    return jobs


# --------------------------------------------------------------------------- worker pool
class _Pending:
    """Results of _WorkerPool.submit, retrievable in any order while the workers are still busy."""

    def __init__(self, n):
        import threading
        self.results, self.ready, self.error, self.cv, self.threads = [None] * n, [False] * n, None, threading.Condition(), []

    def put(self, i, value):
        with self.cv:
            self.results[i], self.ready[i] = value, True
            self.cv.notify_all()

    def fail(self, err):
        with self.cv:
            if self.error is None:
                self.error = err
            self.cv.notify_all()

    def get(self, i):
        with self.cv:
            while not self.ready[i] and self.error is None:
                self.cv.wait()
            if not self.ready[i]:
                raise self.error
            out, self.results[i] = self.results[i], None
            return out


class _WorkerPool:
    """Persistent `python -m audio_suite_b200.plan_worker` subprocesses, one feeder thread each."""

    def __init__(self, size):
        import os
        import subprocess
        import sys
        root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
        env = dict(os.environ)
        env["PYTHONPATH"] = root + os.pathsep + env.get("PYTHONPATH", "")
        env["OMP_NUM_THREADS"] = env["OPENBLAS_NUM_THREADS"] = "1"
        self.size = size
        self.procs = [subprocess.Popen([sys.executable, "-m", "audio_suite_b200.plan_worker"], stdin=subprocess.PIPE,
                                       stdout=subprocess.PIPE, env=env) for _ in range(size)]
        # one worker per core, leaving the first cores of the affinity mask to the parent (kernel launches, table
        # uploads, the copy stream): measured on the 16-core B200 hosts, workers floating over all cores stall
        # the parent's CUDA calls for tens of ms at a time
        try:
            cores = sorted(os.sched_getaffinity(0))
            spare = int(os.environ.get("MS_PLAN_SPARE_CORES", "2")) if len(cores) >= 8 else 0
            usable = cores[spare:] or cores
            # (pinning only helps when this process owns the box; ranks of a torchrun job share it unpinned)
            if os.environ.get("MS_PLAN_PIN", "0") == "1":
                for i, p in enumerate(self.procs):
                    os.sched_setaffinity(p.pid, {usable[i % len(usable)]})
        except Exception:
            pass
        try:                                    # 1 MiB pipes: a request or a packed piece fits without blocking the writer
            import fcntl
            for p in self.procs:
                for f in (p.stdin, p.stdout):
                    fcntl.fcntl(f.fileno(), 1031, 1 << 20)          # F_SETPIPE_SZ
        except Exception:
            pass

    def submit(self, chunks, prep=None):
        """Start planning `chunks` (lists of parameter dicts); returns a _Pending whose get(i) blocks until
        chunk i is packed.  Chunks are handed out in order, so early chunks finish first.  `prep` (optional)
        is applied to a chunk by the feeder thread right before it is sent."""
        import pickle
        import struct
        import threading
        pend = _Pending(len(chunks))
        todo = list(enumerate(chunks))
        lock = threading.Lock()

        def serve(proc):
            # two requests in flight per worker: the worker finds its next piece already in the pipe when it
            # finishes one, instead of waiting for this thread to be scheduled on a box whose cores are all busy
            from collections import deque
            inflight = deque()

            def send_next():
                with lock:
                    if not todo or pend.error is not None:
                        return
                    i, chunk = todo.pop(0)
                if prep is not None:
                    chunk = prep(chunk)
                blob = pickle.dumps(chunk, protocol=pickle.HIGHEST_PROTOCOL)
                proc.stdin.write(struct.pack("<Q", len(blob)))
                proc.stdin.write(blob)
                proc.stdin.flush()
                inflight.append(i)
            try:
                send_next()
                send_next()
                while inflight:
                    i = inflight.popleft()
                    head = proc.stdout.read(8)
                    if len(head) < 8:
                        raise RuntimeError("planning worker died")
                    status, payload = pickle.loads(proc.stdout.read(struct.unpack("<Q", head)[0]))
                    if status != "ok":
                        raise payload
                    pend.put(i, payload)
                    send_next()
            except BaseException as e:
                pend.fail(e)
        pend.threads = [threading.Thread(target=serve, args=(p,), daemon=True) for p in self.procs]
        for t in pend.threads:
            t.start()
        return pend

    def map(self, chunks):
        pend = self.submit(chunks)
        try:
            return [pend.get(i) for i in range(len(chunks))]
        except BaseException:
            self.close()
            raise

    def close(self):
        for p in self.procs:
            try:
                p.stdin.close()
                p.terminate()
            except Exception:
                pass
        self.procs = []


_POOL = None


def shutdown_pool():
    global _POOL
    if _POOL is not None:
        _POOL.close()
        _POOL = None


def _pool(workers):
    import atexit
    global _POOL
    if _POOL is None or _POOL.size != workers or not _POOL.procs:
        shutdown_pool()
        _POOL = _WorkerPool(workers)
        atexit.register(shutdown_pool)
    return _POOL


def default_workers():
    """Planning worker processes per rank: the cores this process may run on, shared between the ranks of the box
    (torchrun sets LOCAL_WORLD_SIZE), minus two per rank for the parent (kernel launches, uploads, copy stream)."""
    import os
    forced = int(os.environ.get("MS_PLAN_WORKERS", "0"))
    if forced:
        return forced
    cores = len(os.sched_getaffinity(0))
    ranks = max(1, int(os.environ.get("LOCAL_WORLD_SIZE", "1")))
    share = cores // ranks
    return min(32, max(1, share - 2 if share >= 8 else share - 1 if share >= 3 else share))


def plan_stream(params_list, chunk, workers=None, piece=32):
    """Generator of packed Tables for consecutive slices of `chunk` renders.  The whole list is handed to the
    worker pool at once (pieces of `piece` renders, in order); slice k is yielded as soon as its pieces are
    packed, while the workers carry on with the later ones -- the caller renders slice k meanwhile."""
    n = len(params_list)
    workers = default_workers() if workers is None else workers
    # slice boundaries; `chunk` may be a list of sizes (the last one repeats): a short first slice starts the GPU and
    # the device->host drain early
    sizes = list(chunk) if isinstance(chunk, (list, tuple)) else [int(chunk)]
    cuts, a = [], 0
    while a < n:
        c = max(1, int(sizes[min(len(cuts), len(sizes) - 1)]))
        cuts.append((a, min(n, a + c)))
        a += c
    # slices whose renders all belong to the native planner's family are planned in-process by libms_hostplan.so
    # (hostplan.plan_slice: no pickling, ~10x the Python planner's speed); the others go to the worker processes
    from . import hostplan
    have_native = hostplan.lib() is not None and not os.environ.get("MS_PLAN_PYTHON")

    def is_native(a, b):
        return have_native and all(hostplan.supported(p) for p in params_list[a:b])
    if have_native and len(cuts) > 1 and workers > 1 and is_native(*cuts[0]):
        # Optimistic native path: the first slice is planned before anything else is looked at; then two Python threads
        # alternate over the remaining slices (one converts the parameters of slice k+1 while the native call of slice k --
        # which releases the GIL and plans blocks of renders on its own threads -- runs).  Slices come out in order.  The
        # conversion itself notices a render outside the native family (hostplan.Unsupported): from that slice on the
        # batch goes through the general path below.
        from concurrent.futures import ThreadPoolExecutor
        nthr = max(1, min(hostplan.default_threads(), workers))
        yield hostplan.plan_chunk(params_list[cuts[0][0]:cuts[0][1]], nthr)
        rest = None
        with ThreadPoolExecutor(max_workers=2, thread_name_prefix="ms-hostplan") as ex:
            futs = [ex.submit(hostplan.plan_chunk, params_list[a:b], nthr) for a, b in cuts[1:]]
            for k, f in enumerate(futs):
                try:
                    tb = f.result()
                except hostplan.Unsupported:
                    for g in futs[k + 1:]:
                        g.cancel()
                    rest = k + 1
                    break
                yield tb
        if rest is not None:
            yield from plan_stream(params_list[cuts[rest][0]:], sizes[rest:] if len(sizes) > rest else sizes[-1:], workers=workers, piece=piece)
        return
    native = [is_native(a, b) for a, b in cuts]
    if workers <= 1 or all(native):
        for (a, b), nat in zip(cuts, native):
            yield hostplan.plan_slice(params_list[a:b]) if nat else pack_chunk([P.plan_render(p) for p in params_list[a:b]])
        return
    bounds = []
    for (a, b), nat in zip(cuts, native):
        bounds.append(None if nat else [(i, min(b, i + piece)) for i in range(a, b, piece)])
    flat = [ab for bs in bounds if bs is not None for ab in bs]
    # Static round-robin assignment: piece i belongs to worker i % W and is answered in order; the parent reads the
    # answers in piece order straight from the pipes (1 MiB pipes let a worker run a few pieces ahead).  Impulse
    # responses are digested before pickling (P._slim_params).
    import pickle
    import struct
    pool = _pool(workers)
    W = len(pool.procs)

    def send(w, obj):
        blob = pickle.dumps(obj, protocol=pickle.HIGHEST_PROTOCOL)
        f = pool.procs[w].stdin
        f.write(struct.pack("<Q", len(blob)))
        f.write(blob)
        f.flush()

    def slim(i):
        a, b = flat[i]
        return [P._slim_params(p) for p in params_list[a:b]]

    def recv(w):
        f = pool.procs[w].stdout
        head = f.read(8)
        if len(head) < 8:
            raise RuntimeError("planning worker died")
        status, payload = pickle.loads(f.read(struct.unpack("<Q", head)[0]))
        if status != "ok":
            raise payload
        return payload
    # Requests go out piece by piece, round-robin (piece i -> worker i % W), from a FEEDER THREAD: the thread that
    # reads the answers never blocks on a write.  (Writing from the reading thread can deadlock: a request larger than
    # the free space of a worker's stdin pipe blocks the parent while that worker is itself blocked writing an answer
    # nobody reads -- reproduced with 4 MB `_img_gray` arrays per piece.)  Every piece below the one being read has been
    # consumed, so the worker that owns it can always finish it: the pipeline cannot stall for good.
    import threading
    feed_err = []

    def feed():
        try:
            for i in range(len(flat)):
                send(i % W, slim(i))
        except BaseException as e:          # a closed pool (abandoned generator) ends the feeder quietly;
            feed_err.append(e)              # anything else (e.g. an unpicklable parameter) must not leave the reader waiting
            if not isinstance(e, (BrokenPipeError, ValueError, OSError)):
                shutdown_pool()
    feeder = threading.Thread(target=feed, daemon=True)
    feeder.start()
    try:
        k = 0
        for (a, b), bs in zip(cuts, bounds):
            if bs is None:
                yield hostplan.plan_slice(params_list[a:b])
                continue
            parts = [recv((k + t) % W) for t in range(len(bs))]
            k += len(bs)
            yield merge_chunks(parts)
        feeder.join()
    except BaseException as e:
        shutdown_pool()          # pipes may hold unread answers: start from fresh workers next time
        if feed_err and not isinstance(feed_err[0], (BrokenPipeError, ValueError, OSError)) and isinstance(e, RuntimeError):
            raise feed_err[0]
        raise


def plan_and_pack(params_list, workers=None):
    """Returns (Tables, plans or None).  Small batches are planned in-process (plans kept for progress /
    inspection); large ones by a persistent pool of worker processes that return packed chunks."""
    import os
    from . import hostplan
    n = len(params_list)
    if hostplan.lib() is not None and not os.environ.get("MS_PLAN_PYTHON") and all(hostplan.supported(p) for p in params_list):
        return hostplan.plan_slice(params_list), None
    if workers is None:
        workers = default_workers()
    min_batch = int(os.environ.get("MS_PLAN_MIN_BATCH", "256"))
    if n < min_batch or workers <= 1:
        plans = [P.plan_render(p) for p in params_list]
        return pack_chunk(plans), plans
    slim = [P._slim_params(p) for p in params_list]      # do not pickle multi-MB impulse responses per render
    per = max(min(32, max(1, n // workers)), (n + 2 * workers - 1) // (2 * workers))
    chunks = _pool(workers).map([slim[i:i + per] for i in range(0, n, per)])
    return merge_chunks(chunks), None
