"""EXTENSION (SURVEY a14, "parity unpinned"): band-limited polyphase decimation on the GPU.

Microsound's render() never decimates -- its rate change is a relabel (main_v2.py:489-490) and its band-limit is the
whole-grain rFFT mask lowpass_fft (main_v2.py:39-59) -- so nothing on the parity path calls this.  It is the stage the
task statement describes ("band-limited polyphase decimation stages filter taps in shared memory and reduces with warp
shuffles"), offered as a stand-alone operator with scipy.signal.resample_poly's conventions and checked against scipy
in float64 (tests/test_decimate.py)."""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _abi


def resample_taps(up, down, half_len_per_q=10, beta=5.0):
    """The filter resample_poly(x, up, down) designs: up * firwin(2 * 10 q + 1, 1 / q, window=('kaiser', 5.0)) with
    q = max(up, down), restated with numpy (windowed sinc, unit DC gain before the factor up).  Float64 taps of odd length."""
    q = max(int(up), int(down))
    half = half_len_per_q * q
    m = np.arange(-half, half + 1, dtype=np.float64)
    h = (1.0 / q) * np.sinc(m / q) * np.kaiser(2 * half + 1, beta)
    return int(up) * (h / np.sum(h))


def design_taps(q, half_len_per_q=10, beta=5.0):
    """The low-pass resample_poly(x, 1, q) designs (resample_taps with up = 1)."""
    return resample_taps(1, q, half_len_per_q, beta)


_BANKS = {}


def polyphase_bank(up, down):
    """resample_taps(up, down) as the polyphase bank ms_post_export reads (include/microsound_b200.h): float64
    [up, taps], row p holding g[p + half - s up] for s = -A .. taps - 1 - A (zero outside g), A = half // up.
    Returns (half, taps, bank); cached per ratio, so a sweep shares one bank."""
    key = (int(up), int(down))
    hit = _BANKS.get(key)
    if hit is None:
        g = resample_taps(*key)
        half = (len(g) - 1) // 2
        u = key[0]
        a, b = half // u, (u - 1 + half) // u
        k = np.arange(u)[:, None] + half - np.arange(-a, b + 1)[None, :] * u
        bank = np.where((k >= 0) & (k <= 2 * half), g[np.clip(k, 0, 2 * half)], 0.0)
        hit = _BANKS[key] = (half, a + b + 1, np.ascontiguousarray(bank))
    return hit


def upfirdn_decimate(x, h, q, device, precision="f64"):
    """scipy.signal.upfirdn(h, x, up=1, down=q) along the last axis of `x` ([signals, n] or [n]) on the device."""
    api = _abi.Api(device.lib, precision)
    real = np.float32 if precision == "f32" else np.float64
    x2 = np.atleast_2d(np.asarray(x, real))
    s, n = x2.shape
    taps = int(len(h))
    n_out = (n + taps - 1 + q - 1) // q
    dx, dh = device.upload(np.ascontiguousarray(x2)), device.upload(np.asarray(h, real))
    dy = device.zeros(max(1, s * n_out), real)
    rc = api.ms_polyphase_decimate(device.ptr(dx), n, n, s, device.ptr(dh), taps, int(q), device.ptr(dy), n_out, device.stream_ptr())
    if rc != 0:
        raise RuntimeError("microsound_b200: " + (device.lib.ms_last_error() or b"unknown error").decode())
    device.synchronize()
    y = np.asarray(device.download(dy, 0, s * n_out)).view(real).reshape(s, n_out)
    return y[0] if np.ndim(x) == 1 else y


def resample_poly(x, up, down, device, precision="f64", n_out=None):
    """scipy.signal.resample_poly(x, up, down) along axis 0 of `x` ([n] or [n, signals]) on the device
    (ms_resample_poly, with the filter of polyphase_bank).  Returns ceil(n up / down) rows, or only the first `n_out` of
    them: every output is its own sum, so those rows are bitwise the rows of the full call."""
    up, down = int(up), int(down)
    api = _abi.Api(device.lib, precision)
    real = np.float32 if precision == "f32" else np.float64
    a = np.asarray(x)
    x2 = np.ascontiguousarray(np.atleast_2d(a.T if a.ndim > 1 else a), dtype=real)        # [signals, n]
    s, n = x2.shape
    full = -(-n * up // down)
    n_out = full if n_out is None else max(0, min(int(n_out), full))
    half, taps, bank = polyphase_bank(up, down)
    y = np.zeros((s, n_out), real)
    if n_out and s:
        dx, db = device.upload(x2), device.upload(bank.astype(real))
        dy = device.zeros(s * n_out, real)
        rc = api.ms_resample_poly(device.ptr(dx), n, n, s, device.ptr(db), up, down, half, taps, device.ptr(dy), n_out, n_out,
                                  device.stream_ptr())
        if rc != 0:
            raise RuntimeError("microsound_b200: " + (device.lib.ms_last_error() or b"unknown error").decode())
        device.synchronize()
        y = np.asarray(device.download(dy, 0, s * n_out)).view(real).reshape(s, n_out)
    return np.ascontiguousarray(y.T) if a.ndim > 1 else y[0]


def decimate(x, q, device, precision="f64", taps=None):
    """resample_poly(x, 1, q) along the last axis: the Kaiser-windowed FIR above, group delay removed, ceil(n / q) outputs."""
    h = design_taps(q) if taps is None else np.asarray(taps, np.float64)
    half = (len(h) - 1) // 2
    n = np.shape(x)[-1]
    # resample_poly pads the filter in front so that output 0 is centred on input 0: here the same alignment by padding
    # the taps with (q - half % q) % q leading zeros and dropping the first (half + pad) / q outputs
    pad = (q - half % q) % q
    hp = np.concatenate([np.zeros(pad), h])
    y = upfirdn_decimate(x, hp, q, device, precision)
    first = (half + pad) // q
    n_out = -(-n // q)
    return y[..., first:first + n_out]
