"""Native host planner binding (csrc/ms_hostplan.cpp -> libms_hostplan.so): parameter dicts of the common family of
renders -> packed job tables, 10-20x faster than the Python planner (plan.py + tables.pack_chunk), which stays the
specification (tests/test_hostplan.py: identical tables) and the path for everything outside the family.

Family: the five gen_basic generators, `event_process` Single or Poisson, no partial lock / cepstral warp / resonator /
waveguide / event feedback / spectral imprint.  That is every render of a seed x unfold x stretch sweep of such a preset
(the reference's batch dialog, main_v2.py:1578-1593) and all of BASELINE.json's configs.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import _abi, decimate, plan as P
from .configs import BASIC_MODES

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "libms_hostplan.so")

FIELDS = ("base_sr", "out_dur_s", "time_unfold", "peak", "sat_drive", "stereo_on", "stereo_width", "gen_mode", "micro_ms", "seed",
          "dust_density", "noise_tilt", "ring_hz", "ring_decay_ms", "unfold_mode", "partial_stretch", "nl_warp_on", "nl_warp_power",
          "mb_b1", "mb_b2", "mb_b3", "mb_u1", "mb_u2", "mb_u3", "mb_roll", "bandlimit_on", "bandlimit_out_hz", "bandlimit_roll_hz",
          "event_process", "grains_per_sec", "max_grains", "grain_amp_rand", "grain_offset_on", "grain_offset_max_ms",
          "bp_density", "bp_unfold", "bp_cutoff", "bp_stretch", "er_cloud_on", "er_taps", "er_max_ms", "space_ir_on", "_ir",
          "_ir_r", "env_a", "env_d", "env_s", "env_r", "env_curve", "_bessel", "export_sr",
          "export_format", "export_dither")
_MODE = {m: float(i) for i, m in enumerate(BASIC_MODES)}
_PROCESS = {"Single": 0.0, "Poisson": 1.0}
_OFF_FLAGS = ("partial_lock_on", "cep_warp_on", "res_bank_on", "wg_on", "event_feedback_on", "spectral_imprint_on")
_HP_NAMES = ("sy1", "ola_r", "env_reps", "ola_e", "fir", "post", "tap_off", "dust_pos", "tilt", "grain", "rot", "odd", "irs", "export", "ratios", "pcm")   # ms_hp_sizes

_lib = None


def lib():
    """The native planner, or None when it has not been built (callers then use the Python planner -- same tables)."""
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            _lib = False
        else:
            l = C.CDLL(LIB_PATH)
            l.ms_hp_field_count.restype = C.c_int
            l.ms_hp_plan.restype = C.c_void_p
            l.ms_hp_plan.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int]
            l.ms_hp_error.restype = C.c_char_p
            l.ms_hp_error.argtypes = [C.c_void_p, C.POINTER(C.c_int)]
            l.ms_hp_sizes.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
            l.ms_hp_export.argtypes = [C.c_void_p] * 28
            l.ms_hp_free.argtypes = [C.c_void_p]
            l.ms_hp_pcg64_seed.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
            l.ms_hp_draws.argtypes = [C.c_int64, C.c_int, C.c_uint64, C.c_int, C.c_void_p]
            if l.ms_hp_field_count() != len(FIELDS):
                raise RuntimeError("libms_hostplan.so does not match hostplan.FIELDS; rebuild (make -C audio_suite_b200/csrc)")
            _lib = l
    return _lib or None


def supported(p) -> bool:
    """True when render `p` belongs to the family the native planner covers."""
    if p["gen_mode"] not in _MODE or p["event_process"] not in _PROCESS:
        return False
    for k in _OFF_FLAGS:
        if p[k]:
            return False
    return int(p["seed"]) >= 0


def pcg64_states(seeds):
    """numpy's PCG64(seed).state for every seed: uint64 [n, 4] = state hi, state lo, inc hi, inc lo."""
    s = np.ascontiguousarray(seeds, dtype=np.int64)
    out = np.zeros((s.size, 4), np.uint64)
    lib().ms_hp_pcg64_seed(s.ctypes.data, int(s.size), out.ctypes.data)
    return out


_NUM = ("base_sr", "out_dur_s", "time_unfold", "peak", "sat_drive", "stereo_on", "stereo_width", "micro_ms", "seed",
        "dust_density", "noise_tilt", "ring_hz", "ring_decay_ms", "partial_stretch", "nl_warp_on", "nl_warp_power",
        "mb_b1", "mb_b2", "mb_b3", "mb_u1", "mb_u2", "mb_u3", "mb_roll", "bandlimit_on", "bandlimit_out_hz", "bandlimit_roll_hz",
        "grains_per_sec", "max_grains", "grain_amp_rand", "grain_offset_on", "grain_offset_max_ms",
        "er_cloud_on", "er_taps", "er_max_ms", "space_ir_on", "env_a", "env_d", "env_s", "env_r", "env_curve")
_NUM_COL = [FIELDS.index(k) for k in _NUM]
_INT_COL = [FIELDS.index(k) for k in ("base_sr", "seed", "max_grains", "er_taps")]           # int(params[k]) in the reference
_BOOL_COL = [FIELDS.index(k) for k in ("stereo_on", "nl_warp_on", "bandlimit_on", "grain_offset_on", "er_cloud_on", "space_ir_on")]
_get_num = _get_side = None


class Unsupported(Exception):
    """A render of the list is outside the native planner's family (`supported()` is False for it); args[0] = its index."""
_CLASSIC = "Classic reinterpret"


def _marshal(params_list):
    """Parameter dicts -> float64 rows in FIELDS order plus the side tables (lanes, impulse responses, Bessel taps)."""
    import operator
    from . import tables as T
    global _get_num, _get_side
    if _get_num is None:
        _get_num = operator.itemgetter(*(_NUM + _OFF_FLAGS))     # the flags ride along: the support check costs no second pass

        _get_side = operator.itemgetter("gen_mode", "unfold_mode", "event_process", "bp_density", "bp_unfold", "bp_cutoff",
                                        "bp_stretch", "space_ir_on", "space_ir_max_samps")
    R = len(params_list)
    rows = np.zeros((R, len(FIELDS)), np.float64)
    try:
        # (blocks of 64 with a GIL hand-over in between: a planning thread must not keep the launching thread waiting for
        #  the ~3 ms a 512-render slice takes to convert)
        import time as _time
        num = []
        for b in range(0, R, 64):
            num += [_get_num(p) for p in params_list[b:b + 64]]
            if b + 64 < R:
                _time.sleep(0)
        num = np.array(num, dtype=np.float64).reshape(R, len(_NUM) + len(_OFF_FLAGS))
        rows[:, _NUM_COL] = num[:, :len(_NUM)]
        bad = np.flatnonzero((num[:, len(_NUM):] != 0.0).any(axis=1) | (num[:, _NUM.index("seed")] < 0))
        if bad.size:
            raise Unsupported(int(bad[0]))
    except (TypeError, ValueError):          # numbers given as strings and the like: the reference's float() / int() accept them
        for r, p in enumerate(params_list):
            if not supported(p):
                raise Unsupported(r)
        rows[:, _NUM_COL] = np.array([[float(p[k]) for k in _NUM] for p in params_list], dtype=np.float64)
    rows[:, _INT_COL] = np.trunc(rows[:, _INT_COL])
    rows[:, _BOOL_COL] = rows[:, _BOOL_COL] != 0.0
    lanes, lane_of = [], {"": -1.0}
    irs, ir_of = [], {}
    bess, bess_of = [], {}

    def lane_id(text):
        i = lane_of.get(text)
        if i is None:
            pts = P.parse_breakpoints(text)
            if not pts:
                i = lane_of[text] = -1.0
            else:
                i = lane_of[text] = float(len(lanes))
                lanes.append(pts)
        return i

    def ir_index(taps):
        j = ir_of.get(id(taps))
        if j is None or irs[j] is not taps:
            j = ir_of[id(taps)] = len(irs)
            irs.append(taps)
        return float(j)
    # the non-numeric fields: one small tuple per render; a sweep repeats the same strings / IR object, so the converted
    # values are memoised per distinct tuple (arrays enter by id(); the objects themselves are kept alive by `params_list`)
    uniq, uniq_of, idx = [], {}, []
    pcm_rows, pcm_vals = [], []
    widths = rows[:, 6].tolist()
    gs = _get_side
    for r, p in enumerate(params_list):
        ir, dig = p.get("_ir_audio"), p.get("_ir_digest")
        if p.get("space_ir_sr") is not None:                     # optional key: the convolution reads the resampled IR
            ir = P.conv_ir(p)
        cap = p.get("space_ir_tap_cap", P.IR_TAP_CAP)           # optional keys: not in the itemgetter
        if cap.__class__ is not int or cap < 1:
            cap = P.ir_tap_cap(p)
        stereo = p.get("space_ir_stereo", False)
        if stereo.__class__ is not bool:
            stereo = P.ir_stereo(p)
        ex = p.get("export_sr")                                  # optional key, 0 = none (also when equal to base_sr)
        if ex is not None:
            rows[r, _EXPORT_COL] = 0.0 if P.export_ratio(p) is None else float(ex)
        if p.get("export_format") is not None:                   # optional key: bits (0 = float32) and dither
            pcm = P.pcm_format(p)
            if pcm is not None:
                pcm_rows.append(r)
                pcm_vals.append(pcm)
        key = gs(p) + (cap, stereo, id(ir), id(dig), widths[r])
        k = uniq_of.get(key)
        if k is None:
            gen_mode, unfold_mode, process, l0, l1, l2, l3, ir_on, max_samps, _, _, _, _, w = key
            ir_id = ir_r_id = -1.0
            if ir_on:
                if dig is not None:
                    pair = dig["taps"], dig.get("taps_r")
                else:
                    pair = P.ir_pair(ir, int(max_samps), cap, stereo) if ir is not None else (None, None)
                if pair[0] is not None:
                    ir_id = ir_index(pair[0])
                    if pair[1] is not None:
                        ir_r_id = ir_index(pair[1])
            theta = (0.0 if w < 0.0 else 1.0 if w > 1.0 else float(w)) * 0.9
            b = bess_of.get(theta)
            if b is None:
                b = bess_of[theta] = float(len(bess))
                bess.append(T.bessel_coeffs(theta))
            k = uniq_of[key] = len(uniq)
            if gen_mode not in _MODE or process not in _PROCESS:
                raise Unsupported(r)
            uniq.append((_MODE[gen_mode], 0.0 if unfold_mode == _CLASSIC else 1.0, _PROCESS[process],
                         lane_id(l0), lane_id(l1), lane_id(l2), lane_id(l3), ir_id, ir_r_id, b))
        idx.append(k)
    if pcm_rows:
        rows[np.ix_(pcm_rows, _PCM_COL)] = pcm_vals
    rows[:, _SIDE_COL] = np.array(uniq, dtype=np.float64).reshape(len(uniq), len(_SIDE_COL))[np.array(idx, dtype=np.intp)]
    lane_ptr = np.zeros(len(lanes) + 1, np.int64)
    for i, pts in enumerate(lanes):
        lane_ptr[i + 1] = lane_ptr[i] + len(pts)
    flat = [q for pts in lanes for q in pts]
    lane_t = np.array([q[0] for q in flat] or [0.0], np.float64)
    lane_v = np.array([q[1] for q in flat] or [0.0], np.float64)
    ir_len = np.array([a.size for a in irs] or [0], np.int64)
    btab = np.ascontiguousarray(np.array(bess, np.float64).reshape(len(bess), -1))
    return rows, lane_ptr, lane_t, lane_v, irs, ir_len, btab


_EXPORT_COL = FIELDS.index("export_sr")
_PCM_COL = [FIELDS.index("export_format"), FIELDS.index("export_dither")]
_SIDE_COL = [FIELDS.index(k) for k in ("gen_mode", "unfold_mode", "event_process", "bp_density", "bp_unfold", "bp_cutoff", "bp_stretch", "_ir", "_ir_r", "_bessel")]


def default_threads():
    """Native planning threads per slice: the cores this process may use, less two for the launching and the prefetching
    thread, shared between the ranks of the node."""
    # (more than four slowed the launching thread's own slice set-up on the 16-core B200 hosts: 86.7 -> 79.4 ms per sweep)
    return max(1, min(4, (len(os.sched_getaffinity(0)) - 2) // max(1, int(os.environ.get("LOCAL_WORLD_SIZE", "1")))))


def plan_chunk(params_list, threads=None):
    """Packed Tables (tables.Tables) of a list of supported renders -- what tables.pack_chunk(plan_render(p) ...) returns.
    `threads` (default: default_threads()): the native call plans blocks of 32 renders on that many threads and appends
    them in order (same tables)."""
    from . import tables as T
    l = lib()
    R = len(params_list)
    rows, lane_ptr, lane_t, lane_v, irs, ir_len, btab = _marshal(params_list)
    h = l.ms_hp_plan(rows.ctypes.data, R, lane_ptr.ctypes.data, lane_t.ctypes.data, lane_v.ctypes.data, ir_len.ctypes.data,
                     btab.ctypes.data, int(btab.shape[1]), max(1, int(default_threads() if threads is None else threads)))
    try:
        bad = C.c_int(-1)
        err = l.ms_hp_error(h, C.byref(bad))
        if err:
            # conditions the reference answers with an exception: let the Python planner raise it, message and all
            T.pack_chunk([P.plan_render(params_list[bad.value])])
            raise RuntimeError("native planner rejected render %d (%s) but the Python planner accepted it" % (bad.value, err.decode()))
        sizes = np.zeros(len(_HP_NAMES), np.int64)
        sc = np.zeros(14, np.int64)
        l.ms_hp_sizes(h, sizes.ctypes.data, sc.ctypes.data)
        n = dict(zip(_HP_NAMES, sizes.tolist()))
        t = T.Tables()
        n["sy2"], n["dust_val"] = n["sy1"], n["dust_pos"]
        for k in ("sy1", "sy2", "ola_r", "env_reps", "ola_e", "fir", "post", "tap_off", "dust_pos", "dust_val", "tilt", "grain", "rot", "odd"):
            setattr(t, k, np.zeros(n[k], getattr(t, k).dtype))
        delay, raw, ir_order = np.zeros(n["tap_off"]), np.zeros(n["tap_off"]), np.zeros(n["irs"], np.int64)
        t.out_at, t.out_n, t.y_at = np.zeros(R, np.int64), np.zeros(R, np.int64), np.zeros(R, np.int64)
        t.last, t.srs = np.zeros(R, T.LAST), np.zeros((R, 2), np.int64)
        t.export, t.export_of, ratios = np.zeros(n["export"], t.export.dtype), np.zeros(n["export"], np.int64), np.zeros((n["ratios"], 2), np.int64)
        t.pcm, t.pcm_of = np.zeros(n["pcm"], t.pcm.dtype), np.zeros(n["pcm"], np.int64)
        args = [t.sy1, t.sy2, t.ola_r, t.env_reps, t.ola_e, t.fir, t.post, t.tap_off, delay, raw, t.dust_pos, t.dust_val,
                t.tilt, t.grain, t.rot, t.odd, ir_order, t.out_at, t.out_n, t.y_at, t.last, t.srs, t.export, t.export_of, ratios,
                t.pcm, t.pcm_of]
        l.ms_hp_export(h, *[a.ctypes.data for a in args])
    finally:
        l.ms_hp_free(h)
    # gains *= exp(-delays * 42) (main_v2.py:415) with numpy's own exp, as the reference computes it
    t.tap_gain = raw * np.exp(-delay * 42.0)
    t.irs = np.concatenate([np.ones(1) if k == -2 else irs[k] for k in ir_order.tolist()]).astype(np.float64) if n["irs"] else np.zeros(0)
    if len(ratios):                       # the banks are designed in numpy, as the Python planner does (bit-identical pools)
        t.bank = np.concatenate([decimate.polyphase_bank(u, d)[2].reshape(-1) for u, d in ratios.tolist()])
    t.pool_n, t.mono_n, t.frames, t.h_total, t.max_h, t.max_out_n, t.env_n = (int(v) for v in sc[:7])
    t.alg = dict(zip(("synth", "tilt_spectral", "grain_spectral", "overlap_add", "fir_in", "fir_taps", "post"), (int(v) for v in sc[7:])))
    return t
