"""Headless preset / batch front end (SURVEY 8(f) rank 3): what the reference's Qt window does around `render` --
preset JSON merged over the factory defaults (main_v2.py:1279-1294), the batch dialog's seed x unfold x stretch sweep
with its file naming (main_v2.py:1553-1593) -- on top of the streamed `render_batch`.

Two quirks of the reference are kept visible rather than silently "fixed":
* the batch name is built as f"ms_seed{sd}_unf{u:g}_st{st:g}_{out_sr}Hz.wav".replace(".", "p"), which also turns the
  extension into "pwav" (main_v2.py:1587); `batch_name` reproduces the string, `batch_render` writes
  `<that name>.wav` so the files stay openable, and returns both;
* soundfile is not a dependency here: audio is written as RIFF/WAVE IEEE-float32 by hand (`write_wav_float32`).
"""
from __future__ import annotations

import json
import os
import struct

import numpy as np

from .configs import FACTORY_DEFAULTS
from .plan import export_ratio


def load_preset(source, ir_audio=None, img_gray=None):
    """Preset (path to a JSON file, or a dict) merged over the factory defaults the way on_load_preset does
    (main_v2.py:1286-1291).  Unknown keys (e.g. the dead `harm_*` keys of five shipped presets) are carried along and
    ignored by render(), as in the reference."""
    if isinstance(source, (str, os.PathLike)):
        with open(source, "r", encoding="utf-8") as f:
            source = json.load(f)
    p = dict(FACTORY_DEFAULTS)
    if isinstance(source, dict):
        p.update(source)
    p["_ir_audio"], p["_img_gray"] = ir_audio, img_gray
    return p


def read_wav(path):
    """(float64 samples [frames] or [frames, channels], sample rate) of a RIFF/WAVE file: PCM 8/16/24/32 bit scaled to
    [-1, 1) the way soundfile's default float64 read does (value / 2^(bits-1)), or IEEE float 32/64.  soundfile is not
    a dependency here."""
    with open(path, "rb") as f:
        raw = f.read()
    if raw[:4] != b"RIFF" or raw[8:12] != b"WAVE":
        raise ValueError(f"{path}: not a RIFF/WAVE file")
    at, fmt, data = 12, None, None
    while at + 8 <= len(raw):
        tag, size = raw[at:at + 4], struct.unpack("<I", raw[at + 4:at + 8])[0]
        body = raw[at + 8:at + 8 + size]
        if tag == b"fmt ":
            fmt = struct.unpack("<HHIIHH", body[:16])
            if fmt[0] == 0xFFFE and len(body) >= 26:            # WAVE_FORMAT_EXTENSIBLE: the sub-format's first two bytes
                fmt = (struct.unpack("<H", body[24:26])[0],) + fmt[1:]
        elif tag == b"data":
            data = body
        at += 8 + size + (size & 1)
    if fmt is None or data is None:
        raise ValueError(f"{path}: missing fmt or data chunk")
    kind, ch, sr, _, _, bits = fmt
    if kind == 3:
        a = np.frombuffer(data, dtype="<f4" if bits == 32 else "<f8").astype(np.float64)
    elif kind == 1 and bits == 8:
        a = (np.frombuffer(data, dtype=np.uint8).astype(np.float64) - 128.0) / 128.0
    elif kind == 1 and bits == 16:
        a = np.frombuffer(data, dtype="<i2").astype(np.float64) / 32768.0
    elif kind == 1 and bits == 24:
        b = np.frombuffer(data[:len(data) // 3 * 3], dtype=np.uint8).reshape(-1, 3).astype(np.int32)
        v = b[:, 0] | (b[:, 1] << 8) | (b[:, 2] << 16)
        a = np.where(v >= 1 << 23, v - (1 << 24), v).astype(np.float64) / float(1 << 23)
    elif kind == 1 and bits == 32:
        a = np.frombuffer(data, dtype="<i4").astype(np.float64) / 2147483648.0
    else:
        raise ValueError(f"{path}: unsupported WAVE format {kind}/{bits} bit")
    if ch > 1:
        a = a[:a.size // ch * ch].reshape(-1, ch)
    return a, int(sr)


def load_ir_wav(path, stereo=False, with_rate=False):
    """What on_load_ir hands to render() as `_ir_audio` (main_v2.py:1401-1413): the file as float64, the mean over
    its channels, normalised to a 0.9 peak (normalize, main_v2.py:26-29: untouched when silent).  The file's sample
    rate is ignored, as in the reference (it is only displayed there); `with_rate=True` (EXTENSION) returns
    `(ir, file_rate)`, the rate to pass as `space_ir_sr` so that the IR is resampled to base_sr.  `stereo=True`
    (EXTENSION, for `space_ir_stereo`) keeps every channel, float64 [frames, channels], with one gain for all of them so
    that their balance stays as recorded; a one-channel file gives the same 1-D array either way."""
    a, sr = read_wav(path)
    a = a.astype(np.float64)
    if a.ndim > 1 and not stereo:
        a = a.mean(axis=1)
    m = float(np.max(np.abs(a))) if a.size else 0.0
    a = a if m <= 0 else a * (0.9 / m)
    return (a, sr) if with_rate else a


def parse_list(text, cast=float):
    """Comma-separated list of the batch dialog; entries that do not parse are dropped (main_v2.py:1553-1562)."""
    out = []
    for part in str(text).split(","):
        part = part.strip()
        if not part:
            continue
        try:
            out.append(cast(part))
        except Exception:
            pass
    return out


def batch_name(seed, unfold, stretch, out_sr):
    """The reference's batch file name, dots and all (main_v2.py:1587)."""
    return f"ms_seed{seed}_unf{unfold:g}_st{stretch:g}_{out_sr}Hz.wav".replace(".", "p")


def batch_params(base_params, seeds, unfolds, stretches):
    """Parameter dicts of the sweep in the reference's loop order: seed outermost, stretch innermost (main_v2.py:1578-1584)."""
    out = []
    for sd in seeds:
        for u in unfolds:
            for st in stretches:
                p = dict(base_params)
                p["seed"], p["time_unfold"], p["partial_stretch"] = int(sd), float(u), float(st)
                out.append(p)
    return out


def write_wav_float32(path, audio, sample_rate):
    """RIFF/WAVE, WAVE_FORMAT_IEEE_FLOAT, 32 bit, interleaved channels."""
    a = np.ascontiguousarray(np.asarray(audio, dtype=np.float32))
    if a.ndim == 1:
        a = a[:, None]
    frames, ch = a.shape
    data = a.astype("<f4").tobytes()
    fmt = struct.pack("<HHIIHH", 3, ch, int(sample_rate), int(sample_rate) * ch * 4, ch * 4, 32)
    fact = struct.pack("<I", frames)
    body = b"WAVE" + b"fmt " + struct.pack("<I", len(fmt)) + fmt + b"fact" + struct.pack("<I", 4) + fact + \
           b"data" + struct.pack("<I", len(data)) + data
    with open(path, "wb") as f:
        f.write(b"RIFF" + struct.pack("<I", len(body)) + body)


def write_wav_pcm(path, data, sample_rate):
    """RIFF/WAVE, WAVE_FORMAT_PCM, stereo, from what a render with `export_format` returns: int16 [n, 2] is written as 16 bit,
    uint8 [n, 6] (L, R as three little-endian bytes each) as 24 bit -- the bytes as they are."""
    a = np.asarray(data)
    if a.dtype == np.int16 and a.ndim == 2 and a.shape[1] == 2:
        bits, data_bytes = 16, np.ascontiguousarray(a, dtype="<i2").tobytes()
    elif a.dtype == np.uint8 and a.ndim == 2 and a.shape[1] == 6:
        bits, data_bytes = 24, np.ascontiguousarray(a).tobytes()
    else:
        raise ValueError(f"write_wav_pcm takes int16 [n, 2] or uint8 [n, 6], not {a.dtype} {a.shape}")
    ch, block = 2, 2 * bits // 8
    fmt = struct.pack("<HHIIHH", 1, ch, int(sample_rate), int(sample_rate) * block, block, bits)
    body = b"WAVE" + b"fmt " + struct.pack("<I", len(fmt)) + fmt + b"data" + struct.pack("<I", len(data_bytes)) + data_bytes
    with open(path, "wb") as f:
        f.write(b"RIFF" + struct.pack("<I", len(body)) + body)


def batch_render(base_params, seeds, unfolds, stretches, folder, device=None, precision="auto", progress=None):
    """The batch dialog's sweep (main_v2.py:1524-1593) through the streamed GPU batch: returns [(reference name, path)].
    With `export_sr` in the parameters the files are written, and named, at that rate; with `export_format` "pcm16" /
    "pcm24" they are 16- / 24-bit PCM files (write_wav_pcm), else 32-bit float.
    `progress(done, total, name)` mirrors the dialog's progress bar / status line."""
    from . import engine
    plist = batch_params(base_params, seeds, unfolds, stretches)
    os.makedirs(folder, exist_ok=True)
    outs = engine.render_batch(plist, device=device, precision=precision)
    written, total = [], max(1, len(plist))
    for i, (p, audio) in enumerate(zip(plist, outs)):
        out_sr = int(p["base_sr"]) if export_ratio(p) is None else int(p["export_sr"])      # the optional key `export_sr`
        name = batch_name(p["seed"], p["time_unfold"], p["partial_stretch"], out_sr)
        path = os.path.join(folder, name + ".wav")
        if audio.dtype == np.float32:
            write_wav_float32(path, audio, out_sr)
        else:
            write_wav_pcm(path, audio, out_sr)
        written.append((name, path))
        if progress:
            progress(i + 1, total, name)
    return written
