"""Headless preset / batch front end (SURVEY 8(f) rank 3) against the reference's rules."""
import os
import struct

import numpy as np

from audio_suite_b200 import configs, frontend


def test_preset_merge_and_lists(tmp_path):
    f = tmp_path / "p.json"
    f.write_text('{"gen_mode": "Wavelet atoms", "micro_ms": 1.6, "harm_mix": 0.5}')
    p = frontend.load_preset(str(f))
    assert p["gen_mode"] == "Wavelet atoms" and p["micro_ms"] == 1.6 and p["harm_mix"] == 0.5
    assert p["event_process"] == "Single" and p["_ir_audio"] is None          # factory default survives (main_v2.py:1039)
    assert set(configs.FACTORY_DEFAULTS) <= set(p)
    assert frontend.parse_list("1001, 1002,x, ,1003", int) == [1001, 1002, 1003]
    assert frontend.parse_list("0.9,1.0,abc,1.2") == [0.9, 1.0, 1.2]


def test_batch_names_follow_the_reference_rule():
    # f"ms_seed{sd}_unf{u:g}_st{st:g}_{out_sr}Hz.wav".replace(".", "p")      main_v2.py:1587
    assert frontend.batch_name(1001, 15.0, 0.9, 48000) == "ms_seed1001_unf15_st0p9_48000Hzpwav"
    assert frontend.batch_name(7, 22.5, 1.0, 96000) == "ms_seed7_unf22p5_st1_96000Hzpwav"
    ps = frontend.batch_params(configs.with_defaults(), [1, 2], [15, 25], [0.9, 1.2])
    assert [(p["seed"], p["time_unfold"], p["partial_stretch"]) for p in ps][:3] == [(1, 15.0, 0.9), (1, 15.0, 1.2), (1, 25.0, 0.9)]
    assert len(ps) == 8 and ps[0] is not ps[1]


def test_wav_writer_round_trip(tmp_path):
    a = np.random.default_rng(0).uniform(-1, 1, (1000, 2)).astype(np.float32)
    path = tmp_path / "x.wav"
    frontend.write_wav_float32(str(path), a, 48000)
    raw = path.read_bytes()
    assert raw[:4] == b"RIFF" and raw[8:12] == b"WAVE" and struct.unpack("<I", raw[4:8])[0] == len(raw) - 8
    fmt, ch, sr, _, _, bits = struct.unpack("<HHIIHH", raw[20:36])
    assert (fmt, ch, sr, bits) == (3, 2, 48000, 32)
    at = raw.index(b"data")
    n = struct.unpack("<I", raw[at + 4:at + 8])[0]
    assert np.array_equal(np.frombuffer(raw[at + 8:at + 8 + n], "<f4").reshape(-1, 2), a)


def test_batch_render_through_the_engine(emul, tmp_path):
    base = configs.with_defaults(out_dur_s=0.05, er_cloud_on=False)
    seen = []
    out = frontend.batch_render(base, [5, 6], [20.0], [1.0, 1.1], str(tmp_path), device=emul, precision="f64",
                                progress=lambda d, t, n: seen.append((d, t)))
    assert len(out) == 4 and seen[-1] == (4, 4)
    assert all(os.path.getsize(p) == 12 + 8 + 16 + 12 + 8 + 2400 * 2 * 4 for _, p in out)
    assert out[0][0] == "ms_seed5_unf20_st1_48000Hzpwav"


def test_ir_loader_follows_on_load_ir(tmp_path):
    """frontend.load_ir_wav = on_load_ir (main_v2.py:1401-1413): float64, mean over channels, normalise to 0.9, rate
    ignored; PCM 16 / 24 / 32 bit and float32 files; the shipped IRs give what the reference's rule gives."""
    import wave
    rng = np.random.default_rng(4)
    x = rng.uniform(-0.5, 0.5, (300, 2))
    frontend.write_wav_float32(str(tmp_path / "f.wav"), x, 44100)
    a, sr = frontend.read_wav(str(tmp_path / "f.wav"))
    assert sr == 44100 and np.array_equal(a, x.astype(np.float32).astype(np.float64))
    ir = frontend.load_ir_wav(str(tmp_path / "f.wav"))
    mono = x.astype(np.float32).astype(np.float64).mean(axis=1)
    assert ir.ndim == 1 and np.allclose(ir, mono * (0.9 / np.max(np.abs(mono))), rtol=0, atol=1e-15) and abs(np.max(np.abs(ir)) - 0.9) < 1e-12
    q = np.round(x[:, 0] * 32767).astype("<i2")
    with wave.open(str(tmp_path / "p16.wav"), "wb") as w:
        w.setnchannels(1); w.setsampwidth(2); w.setframerate(48000); w.writeframes(q.tobytes())
    a, _ = frontend.read_wav(str(tmp_path / "p16.wav"))
    assert np.array_equal(a, q.astype(np.float64) / 32768.0)
    q24 = np.round(x[:, 0] * (2 ** 23 - 1)).astype(np.int32)
    raw = b"".join(int(v & 0xFFFFFF).to_bytes(3, "little") for v in q24)
    with wave.open(str(tmp_path / "p24.wav"), "wb") as w:
        w.setnchannels(1); w.setsampwidth(3); w.setframerate(48000); w.writeframes(raw)
    a, _ = frontend.read_wav(str(tmp_path / "p24.wav"))
    assert np.array_equal(a, q24.astype(np.float64) / float(2 ** 23))
    import kernel_checks as K
    (tmp_path / "irs").mkdir()
    for path, want in K.shipped_irs(tmp_path / "irs").items():
        assert np.array_equal(frontend.load_ir_wav(path), want), path
    from oracle import ref_loader
    if ref_loader.available():
        import glob
        ref = ref_loader.load()
        for f in glob.glob(os.path.join(ref_loader.REFERENCE_ROOT, "microsound_0.2.1", "irs", "*.wav")):
            with wave.open(f, "rb") as w:
                s = np.frombuffer(w.readframes(w.getnframes()), "<i2").astype(np.float64) / 32768.0
                s = s.reshape(-1, w.getnchannels()).mean(axis=1) if w.getnchannels() > 1 else s
            assert np.array_equal(frontend.load_ir_wav(f), ref.normalize(s, 0.9)), f


def test_shipped_preset_files_merge_like_on_load_preset(tmp_path):
    """The 27 shipped presets, as the reference's fixture stores them merged (tests/golden/presets.npz): a file with the
    values that differ from the factory defaults loads to the whole merged set, {**defaults, **file} (main_v2.py:1286-1291)."""
    import json
    import kernel_checks as K
    presets = K.preset_fixture()
    assert len(presets) == 27
    for name, (merged, *_) in presets.items():
        merged = {k: v for k, v in merged.items() if not k.startswith("_")}
        raw = {k: v for k, v in merged.items() if k not in configs.FACTORY_DEFAULTS or configs.FACTORY_DEFAULTS[k] != v}
        f = tmp_path / (name + ".json")
        f.write_text(json.dumps(raw))
        p = frontend.load_preset(str(f))
        assert all(p[k] == v for k, v in merged.items()) and set(configs.FACTORY_DEFAULTS) <= set(p), name
