"""The relocatable job tables: chunks packed on their own and merged must describe the same batch as one chunk packed
whole, for every table and every offset field (tables.RELOC), with the stages outside the native planner's family in
every chunk."""
import copy

import numpy as np
import pytest

from audio_suite_b200 import _abi, configs, plan as P, tables as T

# integer fields that are not offsets into a relocated buffer (operators are skipped as a whole)
NOT_OFFSETS = {
    **{("sy1", f): "" for f in ("s_hi", "s_lo", "i_hi", "i_lo", "n", "mode", "fade", "sigma", "dust_count", "ker_len", "atom_count", "_pad")},
    ("sy1", "aux"): "a pool offset for scanline / chaos / stick-slip only: merge_chunks' special case",
    **{("sy2", f): "" for f in ("s_hi", "s_lo", "i_hi", "i_lo", "n", "mode", "fade", "sigma", "dust_count", "ker_len", "atom_count", "_pad")},
    ("sy2", "dust_begin"): "0 in sy2", ("sy2", "atom_begin"): "0 in sy2",
    **{("ola_r", f): "" for f in ("out_n", "max_len", "A", "D_end", "sus_end", "has_release")},
    **{("env_reps", f): "ms_adsr_tables reads the envelope shape and env only"
       for f in ("out", "out_n", "ev_begin", "ev_end", "max_len", "A", "D_end", "sus_end", "has_release")},
    ("ola_e", "start"): "", ("ola_e", "len"): "",
    **{("fir", f): "" for f in ("ir_len", "h_len", "out_n", "x_begin", "x_end", "_pad")},
    **{("post", f): "" for f in ("n", "stereo_mode", "dl", "dr")},
    ("seq", "rank"): "", ("seq", "fb.n_cur"): "", ("seq", "fb.n_prev"): "", ("seq", "imp.n"): "", ("seq", "imp_item.n"): "",
    ("seq", "imp.z"): "filled on upload", ("seq", "imp.slot"): "filled on upload",
    ("wg", "tmp"): "unused", ("wg", "n"): "", ("wg", "line_count"): "", ("wg", "_pad"): "", ("wg_lines", "d"): "", ("wg_lines", "_pad"): "",
    ("res", "n"): "", ("res", "mode_count"): "", ("res", "_pad"): "",
    **{("cep", f): "filled on upload" for f in ("z1", "z2", "z3", "xp", "cep", "cep2")}, ("cep", "n"): "", ("cep", "_pad"): "",
    ("plock", "z"): "filled on upload", ("plock", "scratch"): "filled on upload",
    **{("plock", f): "" for f in ("n", "top_n", "neigh", "_pad")},
    ("imprint", "z"): "filled on upload", ("imprint", "n"): "", ("imprint", "_pad"): "",
    **{(t, "n"): "" for t in ("tilt", "grain", "rot", "post_grain", "cep_items", "plock_items", "imprint_items")},
    ("odd", "n"): "", ("odd", "dr"): "", ("last", "n"): "",
    ("tap_off", None): "delays", ("dust_pos", None): "positions inside the event", ("atom_shift", None): "",
    ("out_n", None): "", ("srs", None): "sample rates",
}
_OPS = (np.dtype(_abi.SpecOp), T.SPEC_ITEM.fields["op"][0])


def _int_fields(name, dtype, prefix=""):
    if dtype.names is None:
        return [(name, prefix[:-1] or None)] if dtype.kind in "iu" and dtype not in _OPS else []
    out = []
    for f in dtype.names:
        sub = dtype.fields[f][0]
        if sub not in _OPS:
            out += _int_fields(name, sub, prefix + f + ".")
    return out


def test_every_integer_field_is_relocated_or_declared_not_an_offset():
    t = T.Tables()
    seen = set()
    for name, v in vars(t).items():
        if isinstance(v, np.ndarray):
            seen.update(_int_fields(name, v.dtype))
    assert not seen - set(T.RELOC) - set(NOT_OFFSETS), sorted(seen - set(T.RELOC) - set(NOT_OFFSETS))
    assert not set(T.RELOC) & set(NOT_OFFSETS)
    assert not (set(T.RELOC) | set(NOT_OFFSETS)) - seen       # no stale entries


def _chunk(k):
    """Five renders with every stage outside the native family; the IR differs per chunk."""
    W = configs.with_defaults
    dur = 0.2 if k < 2 else 0.21                # chunks 0 and 1 share their envelope table in the whole batch
    ir = configs.synth_ir(0.01 + 0.002 * k, 48000, 50 + k)
    base = dict(event_process="Poisson", grains_per_sec=30.0, micro_ms=2.0, seed=100 + 10 * k, out_dur_s=dur, er_cloud_on=False)
    return [
        W(base, gen_mode="Micro-chaos", cep_warp_on=True, partial_lock_on=True, partial_stretch=1.2, res_bank_on=True, wg_on=True,
          wg_max_ms=1.0, unfold_mode="Multi-band unfold", event_feedback_on=True, spectral_imprint_on=True),
        W(base, gen_mode="Wavelet atoms", spectral_imprint_on=True, seed=101 + 10 * k, base_sr=44100, out_dur_s=(4411 + 442 * k) / 44100,
          stereo_on=True, er_cloud_on=True, er_taps=40, space_ir_on=True, _ir_audio=ir),
        W(base, gen_mode="Dust impulses", event_feedback_on=True, seed=102 + 10 * k, er_cloud_on=True, er_taps=30),
        W(base, gen_mode="Image scanline", seed=103 + 10 * k, space_ir_on=True, _ir_audio=ir,
          _img_gray=np.random.default_rng(k).integers(0, 256, (20, 100)).astype(np.uint8)),
        W(base, gen_mode="Noise burst", seed=104 + 10 * k, partial_lock_on=True, stereo_on=True),
    ]


def _mono_regions(t):
    """(start, length, (render, kind)) of every region of the mono buffer, sorted; checks they do not overlap."""
    regs = []
    for r, (o, p) in enumerate(zip(t.ola_r, t.post)):
        n, mode = int(p["n"]), int(p["stereo_mode"])
        regs.append((int(o["out"]), n, (r, "ola")))
        if p["y"] != o["out"]:
            regs.append((int(p["y"]), n, (r, "fir")))
        if mode:
            regs.append((int(p["rbuf"]) - (n if mode == 2 else 0), mode * n, (r, "stereo")))
    regs.sort()
    for (a, n, _), (b, _, _) in zip(regs, regs[1:]):
        assert a + n <= b, "mono regions overlap"
    assert regs[-1][0] + regs[-1][1] <= t.mono_n
    return regs


def _mono_canon(t, offsets):
    """mono offsets -> (render, region, offset inside it): the same in any layout of the buffer."""
    regs = _mono_regions(t)
    starts = np.array([s for s, _, _ in regs])
    out = []
    for v in np.asarray(offsets).tolist():
        i = int(np.searchsorted(starts, v, side="right")) - 1
        s, n, key = regs[i]
        assert 0 <= v - s <= n
        out.append((key, v - s))
    return out


MONO = {("ola_r", "out"), ("fir", "x"), ("fir", "y"), ("post", "y"), ("post", "rbuf"), ("odd", "y_at"), ("odd", "scratch"),
        ("rot", "src"), ("rot", "dst"), ("y_at", None)}


_READ_WHERE = {
    ("sy1", "dust_begin"): lambda t: t.sy1["dust_count"] > 0,
    ("sy1", "atom_begin"): lambda t: t.sy1["atom_count"] > 0,
    ("sy2", "aux"): lambda t: np.isin(t.sy1["mode"], (P.MODE_SCANLINE, P.MODE_CHAOS, P.MODE_STICK, P.MODE_NOISE, P.MODE_SKEW)),
}


def _envelopes(t):
    """per render: the envelope record its shared table was made from (None when it has its own)."""
    shape = ("out_n", "A", "D_end", "sus_end", "has_release", "inv_A", "inv_D", "inv_R", "S", "curve")
    rep_at = {int(e["env"]): e for e in t.env_reps}
    ends = sorted((int(e["env"]), int(e["env"]) + int(e["out_n"])) for e in t.env_reps)
    assert all(a[1] <= b[0] for a, b in zip(ends, ends[1:])) and (not ends or ends[-1][1] <= t.env_n)
    out = []
    for o in t.ola_r:
        if o["env"] < 0:
            out.append(None)
        else:
            rep = rep_at[int(o["env"])]
            assert all(rep[f] == o[f] for f in shape)
            out.append(tuple(rep[f] for f in shape))
    return out


def _impulse_responses(t):
    return [t.irs[int(f["ir"]):int(f["ir"]) + int(f["ir_len"])].tolist() for f in t.fir]


def assert_same_batch(got, want):
    for name, w in vars(want).items():
        g = getattr(got, name)
        if name in ("env_reps", "env_n", "irs"):
            continue
        if not isinstance(w, np.ndarray):
            assert g == w, name
            continue
        assert g.dtype == w.dtype and g.shape == w.shape, name
        for f in (w.dtype.names or (None,)):
            if (name, f) in MONO:
                assert _mono_canon(got, T.column(g, f)) == _mono_canon(want, T.column(w, f)), (name, f)
            elif (name, f) in _READ_WHERE:                 # merge_chunks shifts these in every row; only some rows are read
                used = _READ_WHERE[name, f](want)
                assert np.array_equal(g[f][used], w[f][used]), (name, f)
            elif (name, f) not in (("ola_r", "env"), ("fir", "ir")):
                assert np.array_equal(T.column(g, f), T.column(w, f)), (name, f)
    assert _envelopes(got) == _envelopes(want)
    assert _impulse_responses(got) == _impulse_responses(want)


@pytest.fixture(scope="module")
def three_chunks():
    chunks = [[P.plan_render(p) for p in _chunk(k)] for k in range(3)]
    return chunks, [T.pack_chunk(c) for c in chunks]


def test_merged_chunks_equal_the_batch_packed_whole(three_chunks):
    plans, packed = three_chunks
    before = copy.deepcopy(packed)
    merged = T.merge_chunks(packed)
    whole = T.pack_chunk([rp for c in plans for rp in c])
    for name in ("cep", "plock", "res", "wg", "seq", "imprint", "post_grain", "tilt", "grain", "rot", "odd", "atoms", "dust_pos",
                 "fir", "env_reps"):
        assert all(len(getattr(c, name)) for c in packed), name                 # every chunk holds every kind of table
    assert (merged.seq["imp_item"]["dst"] >= 0).any() and (merged.seq["fb"]["dst"] >= 0).any()
    assert len(merged.env_reps) != len(whole.env_reps) and merged.irs.size != whole.irs.size       # deduplicated across the cuts
    assert_same_batch(merged, whole)
    for b, a in zip(before, packed):                                              # the inputs are left as they were
        for name, v in vars(b).items():
            w = getattr(a, name)
            assert (np.array_equal(v, w) if isinstance(v, np.ndarray) else v == w), name
