"""ctypes binding of the C ABI in include/microsound_b200.h.

The product has exactly one compute path: the CUDA shared library built from csrc/ for sm_100a.
If it is missing or was not built from the CUDA sources, importing this module's `lib()` raises --
there is no CPU fallback (the block-emulator build under tests/host_emul is test infrastructure and
can only be selected explicitly by tests through `load_library(path)`).
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# MS_LIB_PATH: A/B-test another build of the same CUDA library (development only; still no CPU fallback)
LIB_PATH = os.environ.get("MS_LIB_PATH") or os.path.join(_HERE, "csrc", "libmicrosound_b200.so")


class BandEdge(C.Structure):
    _fields_ = [("lo_f0", C.c_double), ("lo_f1", C.c_double), ("hi_f0", C.c_double), ("hi_f1", C.c_double),
                ("lo_mode", C.c_int32), ("hi_mode", C.c_int32), ("zero", C.c_int32), ("_pad", C.c_int32)]


class SpecOp(C.Structure):
    _fields_ = [("kind", C.c_int32), ("n_bands", C.c_int32), ("lp_on", C.c_int32), ("stretch_on", C.c_int32),
                ("df", C.c_double), ("factor", C.c_double), ("alpha", C.c_double), ("warp_exp", C.c_double),
                ("lp", BandEdge), ("mb", BandEdge * 3)]


class SpecJob(C.Structure):
    _fields_ = [("n", C.c_int32), ("_pad", C.c_int32),
                ("in_a", C.c_int64), ("in_b", C.c_int64), ("out_a", C.c_int64), ("out_b", C.c_int64),
                ("op", SpecOp * 2)]


OP_NONE, OP_GRAIN, OP_TILT, OP_ROT = 0, 1, 2, 3
POST_K = 12


class SynthEvt(C.Structure):
    _fields_ = [("s_hi", C.c_uint64), ("s_lo", C.c_uint64), ("i_hi", C.c_uint64), ("i_lo", C.c_uint64),
                ("n", C.c_int32), ("mode", C.c_int32), ("fade", C.c_int32), ("sigma", C.c_int32),
                ("out", C.c_int64), ("f_over_sr", C.c_double), ("inv_fade", C.c_double),
                ("ring_decay", C.c_double), ("env_decay", C.c_double),
                ("dust_begin", C.c_int64), ("dust_count", C.c_int32), ("ker_len", C.c_int32), ("aux", C.c_int64),
                ("atom_begin", C.c_int64), ("atom_count", C.c_int32), ("_pad", C.c_int32)]


class FeedbackEvt(C.Structure):
    _fields_ = [("cur", C.c_int64), ("prev", C.c_int64), ("dst", C.c_int64), ("n_cur", C.c_int32), ("n_prev", C.c_int32),
                ("fb", C.c_double)]


class ImprintStepEvt(C.Structure):
    _fields_ = [("z", C.c_int64), ("n", C.c_int32), ("slot", C.c_int32), ("amount", C.c_double), ("smooth", C.c_double)]


class WgLine(C.Structure):
    _fields_ = [("d", C.c_int32), ("_pad", C.c_int32), ("g", C.c_double), ("mix", C.c_double)]


class WgEvt(C.Structure):
    _fields_ = [("src", C.c_int64), ("dst", C.c_int64), ("tmp", C.c_int64), ("n", C.c_int32), ("line_begin", C.c_int32),
                ("line_count", C.c_int32), ("_pad", C.c_int32)]


class ResMode(C.Structure):
    _fields_ = [("f_over_sr", C.c_double), ("phase", C.c_double), ("weight", C.c_double)]


class ResEvt(C.Structure):
    _fields_ = [("src", C.c_int64), ("dst", C.c_int64), ("n", C.c_int32), ("mode_begin", C.c_int32),
                ("mode_count", C.c_int32), ("_pad", C.c_int32), ("decay", C.c_double)]


class PlockEvt(C.Structure):
    _fields_ = [("z", C.c_int64), ("scratch", C.c_int64), ("n", C.c_int32), ("top_n", C.c_int32), ("neigh", C.c_int32),
                ("_pad", C.c_int32), ("factor", C.c_double), ("pre", SpecOp)]


class CepEvt(C.Structure):
    _fields_ = [("z1", C.c_int64), ("z2", C.c_int64), ("z3", C.c_int64), ("xp", C.c_int64), ("cep", C.c_int64),
                ("cep2", C.c_int64), ("n", C.c_int32), ("_pad", C.c_int32), ("factor", C.c_double), ("pre", SpecOp)]


class ImprintEvt(C.Structure):
    _fields_ = [("z", C.c_int64), ("n", C.c_int32), ("_pad", C.c_int32)]


class ImprintRender(C.Structure):
    _fields_ = [("ev_begin", C.c_int32), ("ev_end", C.c_int32), ("amount", C.c_double), ("smooth", C.c_double)]


class WaveletAtom(C.Structure):
    _fields_ = [("f0_over_sr", C.c_double), ("inv_sigma", C.c_double), ("phase", C.c_double), ("weight", C.c_double)]


class OlaRender(C.Structure):
    _fields_ = [("out", C.c_int64), ("out_n", C.c_int32), ("ev_begin", C.c_int32), ("ev_end", C.c_int32),
                ("max_len", C.c_int32), ("A", C.c_int32), ("D_end", C.c_int32), ("sus_end", C.c_int32),
                ("has_release", C.c_int32), ("inv_A", C.c_double), ("inv_D", C.c_double), ("inv_R", C.c_double),
                ("S", C.c_double), ("curve", C.c_double), ("env", C.c_int64)]


class OlaEvt(C.Structure):
    _fields_ = [("grain", C.c_int64), ("start", C.c_int32), ("len", C.c_int32), ("amp", C.c_double)]


class FirRender(C.Structure):
    _fields_ = [("ir", C.c_int64), ("ir_len", C.c_int32), ("h_len", C.c_int32), ("h", C.c_int64),
                ("tap_begin", C.c_int32), ("tap_end", C.c_int32), ("x", C.c_int64), ("y", C.c_int64),
                ("out_n", C.c_int32), ("x_begin", C.c_int32), ("x_end", C.c_int32), ("_pad", C.c_int32)]


class PostRender(C.Structure):
    _fields_ = [("y", C.c_int64), ("out", C.c_int64), ("rbuf", C.c_int64), ("n", C.c_int32),
                ("stereo_mode", C.c_int32), ("dl", C.c_int32), ("dr", C.c_int32),
                ("drive", C.c_double), ("inv_tanh_drive", C.c_double), ("peak", C.c_double),
                ("coef", C.c_double * (2 * POST_K + 1))]


class ExportRender(C.Structure):
    _fields_ = [("out", C.c_int64), ("out_end", C.c_int64), ("bank", C.c_int64), ("bank_end", C.c_int64),
                ("rate", C.c_int32 * 4)]             # up, down, half, taps per phase


_P, _I, _Z = C.c_void_p, C.c_int, C.c_size_t
_COMMON = {
    "ms_version": (C.c_int, []),
    "ms_last_error": (C.c_char_p, []),
    "ms_is_cuda_build": (C.c_int, []),
    "ms_launch_count": (C.c_ulonglong, []),
    "ms_h2d_bytes": (C.c_ulonglong, []),
    "ms_set_launch_hook": (None, [C.c_void_p]),
}
LAUNCH_HOOK = C.CFUNCTYPE(None, C.c_char_p, C.c_void_p)
# every stage exists as <name>_f32 and <name>_f64 (include/microsound_b200.h, MS_DECLARE_API)
_STAGES = {
    "ms_spectral_workspace_bytes": (_Z, [_P, _I]),
    "ms_spectral_apply": (_I, [_P, _I, _P, _P, _P, _Z, _P]),
    "ms_spectral_create": (_I, [_P, _I, _P, _P, _P, _Z, _P, C.POINTER(C.c_void_p)]),
    "ms_spectral_run": (_I, [_P, _P]),
    "ms_spectral_forward": (_I, [_P, _P]),
    "ms_spectral_inverse": (_I, [_P, _P]),
    "ms_spectral_z_table": (_I, [_P, _P, C.POINTER(C.c_size_t)]),
    "ms_imprint": (_I, [_P, _P, _I, _I, _P, _P]),
    "ms_partial_lock": (_I, [_P, _I, _P, _P, _P]),
    "ms_resonator": (_I, [_P, _I, _P, _P, _P]),
    "ms_waveguide": (_I, [_P, _I, _P, _P, _P]),
    "ms_feedback": (_I, [_P, _I, _I, _P, _P]),
    "ms_imprint_step": (_I, [_P, _I, _I, _P, _P, _P, _P]),
    "ms_cepstral": (_I, [_I, _P, _I, _I, _P, _P, _P, _P, _P]),
    "ms_spectral_destroy": (None, [_P]),
    "ms_fft_pair_forward": (_I, [_P, _P, _I, _P, _P, _Z, _P]),
    "ms_fft_pair_workspace_bytes": (_Z, [_I]),
    "ms_synth_normal": (_I, [_P, _I, _P, _P]),
    "ms_synth_dust": (_I, [_P, _I, _P, _P, _P, _P]),
    "ms_synth_tilt_finish": (_I, [_P, _I, _P, _P]),
    "ms_synth_wavelet": (_I, [_P, _I, _P, _P, _P, _P]),
    "ms_synth_table": (_I, [_P, _I, _P, _P, _P]),
    "ms_adsr_tables": (_I, [_P, _I, _I, _P, _P]),
    "ms_overlap_add": (_I, [_P, _I, _I, _P, _P, _P, _P, _P]),
    "ms_fir_workspace_bytes": (_Z, [_P, _I]),
    "ms_fir_create": (_I, [_P, _I, _P, _P, _P, _P, _P, _P, _Z, _P, C.POINTER(C.c_void_p)]),
    "ms_fir_run": (_I, [_P, _P]),
    "ms_fir_destroy": (None, [_P]),
    "ms_post": (_I, [_P, _I, _I, _P, _P, _P, _P]),
    "ms_post_export": (_I, [_P, _P, _I, _I, _I, _P, _P, _P, _P, _P]),
    "ms_roll": (_I, [_P, _P, _I, _I, _P]),
    "ms_polyphase_decimate": (_I, [_P, C.c_int64, _I, _I, _P, _I, _I, _P, C.c_int64, _P]),
}
PRECISIONS = ("f32", "f64")


class MicrosoundLibraryError(RuntimeError):
    pass


def exported_symbols():
    """Names include/microsound_b200.h declares (checked by tests/test_abi_symbols.py)."""
    return sorted(list(_COMMON) + [f"{n}_{p}" for n in _STAGES for p in PRECISIONS])


def load_library(path):
    if not os.path.isfile(path):
        raise MicrosoundLibraryError(
            f"{path} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a). There is no CPU fallback.")
    lib = C.CDLL(path)
    for name, (res, args) in _COMMON.items():
        fn = getattr(lib, name)      # AttributeError here = header/library mismatch
        fn.restype, fn.argtypes = res, args
    for name, (res, args) in _STAGES.items():
        for p in PRECISIONS:
            fn = getattr(lib, f"{name}_{p}")
            fn.restype, fn.argtypes = res, args
    return lib


class Api:
    """View of the library for one precision: api.ms_post -> lib.ms_post_f64 etc."""

    def __init__(self, lib, precision):
        if precision not in PRECISIONS:
            raise ValueError(f"precision must be one of {PRECISIONS}")
        self.lib, self.precision = lib, precision
        for name in _COMMON:
            setattr(self, name, getattr(lib, name))
        for name in _STAGES:
            setattr(self, name, getattr(lib, f"{name}_{precision}"))


_lib = None


def lib():
    global _lib
    if _lib is None:
        l = load_library(LIB_PATH)
        if l.ms_version() != 1:
            raise MicrosoundLibraryError(f"ABI version mismatch: library {l.ms_version()}, binding 1")
        if not l.ms_is_cuda_build():
            raise MicrosoundLibraryError("libmicrosound_b200.so is not a CUDA build")
        _lib = l
    return _lib


def check(rc, l=None):
    if rc != 0:
        l = l or lib()
        raise RuntimeError("microsound_b200: " + (l.ms_last_error() or b"unknown error").decode())
