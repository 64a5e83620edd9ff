"""The oracle (oracle/microsound_np.py) against (a) the unmodified reference where it exists (build
container) and (b) the golden fixtures the reference produced (tests/golden, oracle/make_golden.py)."""
import functools
import os

import numpy as np
import pytest

from audio_suite_b200 import configs
from oracle import microsound_np as O, ref_loader
from conftest import GOLDEN

TOL = 1e-12


def _g(name):
    return np.load(os.path.join(GOLDEN, name))


# ---------------------------------------------------------------- golden fixtures (travel everywhere)
def test_golden_stage_vectors():
    g = _g("stages.npz")
    x, xo = g["x"], g["x_odd"]
    assert np.max(np.abs(O.fft_lowpass(x, 96000.0, 18000.0, 2500.0) - g["lowpass_roll"])) < TOL
    assert np.max(np.abs(O.fft_lowpass(x, 96000.0, 18000.0, 0.0) - g["lowpass_brick"])) < TOL
    assert np.max(np.abs(O.fft_bandpass(x, 96000.0, 4000.0, 16000.0, 2000.0) - g["bandpass"])) < TOL
    assert np.max(np.abs(O.fft_bandpass(x, 96000.0, 4000.0, 16000.0, 0.0) - g["bandpass_brick"])) < TOL
    assert np.max(np.abs(O.spectrum_stretch(x, 4.0) - g["stretch_4"])) < TOL
    assert np.max(np.abs(O.spectrum_stretch(x, 0.3) - g["stretch_0p3"])) < TOL
    assert np.max(np.abs(O.spectrum_stretch(xo, 2.5) - g["stretch_odd_2p5"])) < TOL
    assert np.max(np.abs(O.fft_lowpass(xo, 48000.0 * 33.3, 18000.0 * 33.3, 2500.0) - g["lowpass_odd"])) < TOL
    mb = O.multiband_unfold(x, 1_200_000.0, [(0, 2000.0), (2000.0, 8000.0), (8000.0, 20000.0)], [35.0, 20.0, 12.0], 2000.0)
    assert np.max(np.abs(mb - g["multiband"])) < TOL
    assert np.max(np.abs(O.adsr_envelope(5000, 48000, 20.0, 30.0, 0.65, 40.0, 1.8) - g["adsr"])) < TOL
    assert np.max(np.abs(O.adsr_envelope(2000, 48000, 20.0, 250.0, 0.65, 1800.0, 1.8) - g["adsr_short"])) < TOL
    assert np.max(np.abs(O.reflection_cloud(x, 8000, 40, 45, 7) - g["er_cloud"])) < TOL
    assert np.max(np.abs(O.short_ir_convolve(x, g["ir"]) - g["conv_ir"])) < 1e-11
    assert np.max(np.abs(O.stereo_diffuse(x, 48000, 0.65) - g["stereo_even"])) < TOL
    assert np.max(np.abs(O.stereo_diffuse(xo, 48000, 0.65) - g["stereo_odd"])) < TOL
    assert np.max(np.abs(O.soft_saturate(x * 3.0, 1.7) - g["soft_clip"])) < TOL
    assert np.max(np.abs(O.peak_normalize(np.column_stack([x, -2 * x]), 0.98) - g["normalize"])) < TOL
    for mode in configs.BASIC_MODES:
        got = O.basic_transient(1_200_000, 1.5, 4242, mode, 0.02, -3.0, 4200.0, 12.0)
        assert np.max(np.abs(got - g["gen_" + mode.replace(" ", "_")])) < TOL, mode


def test_golden_event_fields():
    g = _g("events.npz")
    for proc in ("Single", "Poisson", "Clustered", "Hawkes"):
        got = np.array(O.event_times(proc, 3.0, 18.0, 12345, 6, 25.0, 0.6, 0.25))
        assert got.shape == g["times_" + proc].shape and np.array_equal(got, g["times_" + proc]), proc
    pts = O.parse_lane("0:18, 4:40, junk, 8:14, 2:x, :3")
    assert np.array_equal(np.array(pts), g["bp_points"])
    got = np.array([O.lane_value(pts, t, 7.0) for t in (-1.0, 0.0, 1.0, 4.0, 6.5, 8.0, 9.0)])
    assert np.array_equal(got, g["bp_eval"])


@pytest.mark.parametrize("name", ["C1b", "C1", "C2", "C3"])
def test_golden_renders(name):
    g = _g("renders.npz")
    audio, meta = O.render(configs.canonical(name))
    step = int(g[name + "_step"])
    assert np.max(np.abs(audio[::step] - g[name + "_audio"])) < TOL
    assert np.max(np.abs(meta["grain_last"][::step] - g[name + "_grain_last"])) < TOL
    assert np.max(np.abs(meta["micro_last"][::step] - g[name + "_micro_last"])) < TOL
    assert audio.dtype == np.float64 and audio.shape[1] == 2


@pytest.mark.parametrize("i", [0, 3, 5, 7, 11])
def test_golden_sweep_renders(i):
    g = _g("renders.npz")
    audio, _ = O.render(configs.c5_params(i))
    assert np.max(np.abs(audio[::8] - g[f"C5_{i}_audio"])) < TOL


# ---------------------------------------------------------------- the reference itself (build container only)
needs_ref = pytest.mark.skipif(not ref_loader.available(), reason="/root/reference not present on this machine")


def _cases():
    W = configs.with_defaults
    yield "poisson_lanes", W(event_process="Poisson", out_dur_s=2.0, bp_unfold="0:20, 1:33.3, 2:25",
                             bp_cutoff="0:9000,2:18000", bp_stretch="0:0.5, 2:2")
    yield "clustered", W(event_process="Clustered", out_dur_s=1.5, gen_mode="Noise burst")
    yield "hawkes", W(event_process="Hawkes", out_dur_s=0.6, gen_mode="Resonant strike")
    yield "multiband_dust", W(event_process="Poisson", out_dur_s=1.0, unfold_mode="Multi-band unfold",
                              bandlimit_roll_hz=0.0, gen_mode="Dust impulses")
    yield "skewed_44k_noclip", W(event_process="Poisson", out_dur_s=1.0, gen_mode="Skewed transient", sat_drive=0.0,
                                 stereo_on=False, base_sr=44100)
    yield "fallback_mode", W(gen_mode="Bogus", out_dur_s=1.0)
    yield "odd_length_stereo", W(base_sr=44100, out_dur_s=0.05, er_cloud_on=False)
    yield "max_grains_cut", W(event_process="Poisson", out_dur_s=2.0, max_grains=5, grains_per_sec=40.0)


@needs_ref
@pytest.mark.parametrize("name,params", list(_cases()))
def test_oracle_matches_reference(name, params):
    ref = ref_loader.load()
    a, ma = ref.render(params)
    b, mb = O.render(params)
    assert a.shape == b.shape
    assert np.max(np.abs(a - b)) < TOL
    assert np.max(np.abs(ma["micro_last"] - mb["micro_last"])) < TOL
    assert np.max(np.abs(ma["grain_last"] - mb["grain_last"])) < TOL
    assert ma["out_sr"] == mb["out_sr"] and ma["design_sr_base"] == mb["design_sr_base"]


@functools.lru_cache(maxsize=1)
def _preset_fixture():
    import kernel_checks as K
    return K.preset_fixture()


def test_oracle_progress_calls_match_reference():
    """The (pct, msg) calls the reference made while rendering the 27 shipped presets (tests/golden/presets.npz)."""
    longest = 0
    for name, (p, _, _, _, msgs) in sorted(_preset_fixture().items()):
        b = []
        O.render(p, progress=lambda pct, msg: b.append((int(pct), str(msg))))
        assert b == msgs, name
        longest = max(longest, len(b))
    assert longest >= 4


def test_ir_loader_matches_shipped_files(tmp_path):
    """The shipped impulse responses, rebuilt from what the preset fixture stores of them (kernel_checks.shipped_irs),
    load to the stored arrays; the files themselves too where the reference is present."""
    import kernel_checks as K
    for path, want in K.shipped_irs(tmp_path).items():
        a = ref_loader.load_ir_wav(path)
        assert a.ndim == 1 and abs(np.max(np.abs(a)) - 0.9) < 1e-12 and np.array_equal(a, want), path
    if ref_loader.available():
        d = os.path.join(ref_loader.REFERENCE_ROOT, "microsound_0.2.1", "irs")
        for f in sorted(os.listdir(d)):
            a = ref_loader.load_ir_wav(os.path.join(d, f))
            assert a.ndim == 1 and abs(np.max(np.abs(a)) - 0.9) < 1e-12


# ---------------------------------------------------------------- SURVEY 8(f) rows accelerated so far
def test_golden_next_rows():
    import kernel_checks as K
    g = _g("next_rows.npz")
    assert np.max(np.abs(O.wavelet_atoms(1_200_000, 1.6, 4242, 1800, 10, 0.9) - g["wavelet"])) < TOL
    assert np.max(np.abs(O.wavelet_atoms(1_200_000, 0.11, 7, 2400, 3, 0.6) - g["wavelet_floor"])) < TOL
    imp, at, out = O.ImprintMemory(), 0, []
    for n in (400, 400, 400, 401, 401, 63, 400):
        out.append(imp.apply(g["imprint_in"][at:at + n].copy(), 0.35, 0.9))
        at += n
    assert np.max(np.abs(np.concatenate(out) - g["imprint_out"])) < TOL
    for name in K.PRESET_LIKE:
        p = K.preset_like(name)
        p["out_dur_s"] = 2.0
        audio, _ = O.render(p)
        assert np.max(np.abs(audio[::4] - g["render_" + name])) < TOL, name


def test_wavelet_grain_shorter_than_its_atoms_fails_like_the_reference():
    # 128-sample floor for the grain (main_v2.py:319) but 16 for the atoms (:166): `x += atom[:n]` cannot broadcast
    with pytest.raises(ValueError):
        O.wavelet_atoms(48000, 1.0, 1, 2400, 2, 0.5)
    from audio_suite_b200 import plan as P
    with pytest.raises(ValueError):
        P.plan_render(configs.with_defaults(gen_mode="Wavelet atoms", time_unfold=1.0, micro_ms=1.0))


@pytest.mark.parametrize("name", ["opal_airfold", "opal_oval_breath", "basinski_melodic_loop", "basinski_oval_decay",
                                  "soft_ellipse_memory", "micro_carillon", "oval_glass_orbit", "glass_harmonic_arc",
                                  "01_corona_glass_fog", "corona_memory_glass", "melodic_dust_chime", "oval_room_trace",
                                  "room_as_particle", "image_grain_hallucination", "closed_curve_air",
                                  "drifting_mode_fragments", "ghost_formants", "corona_glass_fog", "chaotic_dustfield",
                                  "elliptical_insect_hum", "infra_mechanical_choir",
                                  "infra_tone_lattice", "03_wavelet_ice_bloom", "orbital_friction_loop",
                                  "02_friction_lattice", "friction_lattice", "wavelet_mist"])
def test_oracle_matches_reference_on_shipped_presets(name):
    """The shipped presets, merged over the factory defaults the way on_load_preset does (main_v2.py:1286-1291), with
    the shipped impulse responses: 2 s renders of the reference, every 8th frame stored as float32
    (tests/golden/presets.npz, oracle/make_golden_presets.py).  The oracle must match to TOL beyond that rounding.
    Where the reference is present, also every frame and grain_last of its own 1.5 s float64 renders, to TOL."""
    p, want, step, _, _ = _preset_fixture()[name]
    b, _ = O.render(p)
    half_ulp = 0.5 * np.spacing(np.abs(want)).astype(np.float64)
    assert b[::step].shape == want.shape
    assert np.max(np.abs(b[::step] - want.astype(np.float64)) - half_ulp) < TOL
    if ref_loader.available():
        import json
        ref = ref_loader.load()
        path = os.path.join(ref_loader.REFERENCE_ROOT, "microsound_0.2.1", "presets", name + ".json")
        p = configs.with_defaults(json.load(open(path)))
        p["out_dur_s"] = 1.5
        if name == "oval_room_trace":
            p["_ir_audio"] = configs.synth_ir(0.25, 48000, 11, channels=1)
        if name == "image_grain_hallucination":
            p["_img_gray"] = np.random.default_rng(5).integers(0, 256, (40, 300)).astype(np.uint8)
        a, ma = ref.render(p)
        b, mb = O.render(p)
        assert np.max(np.abs(a - b)) < TOL and np.max(np.abs(ma["grain_last"] - mb["grain_last"])) < TOL
