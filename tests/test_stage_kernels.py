"""The time-domain stages every render runs after the grains -- FIR (reflection cloud + impulse response, overlap-save),
overlap-add + ADSR, stereo / clip / normalise -- checked stage by stage against float64 restatements (stage_checks.py):
directly through the C ABI at the edges of each kernel, and in situ on real renders, each stage on the device's own
input.  The CPU tests run the kernel bodies on the block emulator at small sizes; the gpu tests repeat them at full size,
the FIR with a batch of many fused units as well.  Every test prints its per-case errors; the tolerances and the errors
measured on a B200 are listed in stage_checks.py."""
import numpy as np
import pytest

import kernel_checks as K
import stage_checks as S
from audio_suite_b200 import configs


def _report(title, errors):
    print("%s: worst %.3e" % (title, max(v for v in errors.values() if v is not None)))
    for k, v in errors.items():
        print("  %-50s %.3e" % (k, v))


def _in_situ_params(big):
    """C3 with a shipped-like IR; a C5 slab whose FIR stages fall in several block classes (IR + cloud in fused
    65536-point blocks, IR alone, cloud alone through the delta IR, no FIR at all) with one odd-length stereo render;
    two shipped presets (an IR without cloud, a cloud without IR)."""
    dur = 2.0 if big else 0.5
    ir = configs.synth_ir(0.25, 48000, 11, channels=1)
    c3 = configs.canonical("C3")
    c3.update(_ir_audio=ir * (0.9 / np.max(np.abs(ir))), space_ir_max_samps=12000)
    if not big:
        c3["out_dur_s"] = 0.25
    slab = [dict(configs.c5_params(i), out_dur_s=dur) for i in (0, 1, 2, 3, 4)]
    slab[1]["er_cloud_on"] = False                              # IR only
    slab[2]["space_ir_on"] = False                              # cloud only: delta IR, 8192-point blocks
    slab[3].update(er_cloud_on=False, space_ir_on=False)        # no FIR stage
    slab[4]["out_dur_s"] = dur + 1.0 / 48000                    # odd length: right channel by the FFT rotation
    assert int(round(slab[4]["out_dur_s"] * 48000)) % 2 == 1
    fx = K.preset_fixture()
    presets = [dict(fx[name][0], out_dur_s=dur) for name in ("oval_room_trace", "image_grain_hallucination")]
    return [("C3 shipped-like IR", [c3]), ("C5 slab", slab), ("presets", presets)]


def _check_in_situ(dev, title, params):
    errs = S.check_in_situ(dev, params)
    print(title)
    for e in errs:
        print("  n=%-8d ola %.3e  fir %s  post %.3e  (pre-clip peak %.1f)" % (
            e["n"], e["ola"], "%.3e" % e["fir"] if e["fir"] is not None else "   -     ", e["post"], e["peak_pre_clip"]))


# ---- CPU: block emulator --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("precision", ["f64", "f32"])
def test_fir_stage_emulated(emul, precision):
    """Every block class, tap sets reaching the self-partnered rows 0 / 128 and the 4096-tap limit, shared delays,
    support edges, one mixed batch run twice."""
    res = S.check_fir(emul, precision, big=False)
    _report("FIR %s" % precision, res["errors"])


@pytest.mark.parametrize("precision", ["f64", "f32"])
def test_overlap_add_adsr_emulated(emul, precision):
    _report("overlap-add + ADSR %s" % precision, S.check_ola(emul, precision))


@pytest.mark.parametrize("precision", ["f64", "f32"])
def test_post_emulated(emul, precision):
    _report("post %s" % precision, S.check_post(emul, precision))


@pytest.mark.parametrize("case", range(3))
def test_stages_in_situ_emulated(emul, case):
    title, params = _in_situ_params(big=False)[case]
    _check_in_situ(emul, title, params)


# ---- GPU --------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_fir_stage(cuda_dev):
    """Full-size cases plus a batch of 300 fused units sharing one IR spectrum, run twice (bitwise-equal repeats)."""
    for precision in ("f64", "f32"):
        res = S.check_fir(cuda_dev, precision, big=True, many=True)
        _report("FIR %s" % precision, res["errors"])
        print("  kernels:", ", ".join(k for k in res["kernels"] if k.startswith(("Fir", "ErScatter"))))


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["f64", "f32"])
def test_overlap_add_adsr(cuda_dev, precision):
    _report("overlap-add + ADSR %s" % precision, S.check_ola(cuda_dev, precision, big=True))


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["f64", "f32"])
def test_post(cuda_dev, precision):
    _report("post %s" % precision, S.check_post(cuda_dev, precision, big=True))


@pytest.mark.gpu
@pytest.mark.parametrize("case", range(3))
def test_stages_in_situ(cuda_dev, case):
    title, params = _in_situ_params(big=True)[case]
    _check_in_situ(cuda_dev, title, params)


@pytest.mark.gpu
def test_stages_in_situ_c4_shortened(cuda_dev):
    p = configs.canonical("C4")
    p["out_dur_s"] = 12.0
    _check_in_situ(cuda_dev, "C4 12 s", [p])
