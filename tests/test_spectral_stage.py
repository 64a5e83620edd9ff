"""The spectral engine -- the grain stage's transforms and operators -- checked stage by stage against float64 references
(spectral_checks.py): a catalogue of lengths with the route each must take, read from the launch log, both directions
with every operator, sentinels around unaligned jobs, shuffled mixed batches, the split entry points and the limits
of the Bluestein route.  The CPU tests run on the block emulator at small sizes; the gpu tests repeat them at full
size and add the side-stream schedule, a class of more jobs than one launch takes and a render at the largest
Bluestein length.  Tolerances and measured errors are listed in spectral_checks.py."""
import pytest

import kernel_checks as K
import spectral_checks as SP
from audio_suite_b200 import configs


def _print_catalogue(precision, seen, worst):
    print("routes %s:" % precision)
    by = {}
    for n, r in seen.items():
        by.setdefault(r, []).append(n)
    for r in SP.ROUTES:
        ns = by.get(r, [])
        print("  %-18s %s" % (r, ", ".join(str(n) for n in ns) if ns else "-"))
    for k, v in worst.items():
        print("  worst %-40s %.3e" % (k, v))


# ---- CPU: block emulator --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("precision", ["f64", "f32"])
def test_route_catalogue_emulated(emul, precision):
    """Every catalogued length takes its route, forward and inverse match the references with every operator."""
    seen, worst = SP.check_catalogue(emul, precision)
    _print_catalogue(precision, seen, worst)


@pytest.mark.parametrize("precision", ["f64", "f32"])
def test_mixed_batch_emulated(emul, precision):
    print(precision, SP.check_mixed_batch(emul, precision))


@pytest.mark.parametrize("precision", ["f64", "f32"])
def test_split_entry_points_emulated(emul, precision):
    lengths = [64, 1000, 2047, 4100, 4208, 9216, 4097]
    print(precision, "Z worst %.3e" % SP.check_split_entry_points(emul, precision, lengths))


@pytest.mark.parametrize("precision", ["f64", "f32"])
def test_lengths_beyond_the_largest_bluestein_size_are_refused(emul, precision):
    """M = 2^23 is refused with a message in both precisions (no device work: the plan fails first)."""
    for n in (2097153, 4194301):
        print(precision, SP.check_refused(emul, precision, n))


# ---- GPU --------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["f64", "f32"])
def test_route_catalogue(cuda_dev, precision):
    """Full-size catalogue, including n / 256 at MS_TILE_MAX / 4 and the largest accepted Bluestein size M = 2^22."""
    seen, worst = SP.check_catalogue(cuda_dev, precision, big=True)
    _print_catalogue(precision, seen, worst)


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["f64", "f32"])
def test_mixed_batch(cuda_dev, precision):
    print(precision, SP.check_mixed_batch(cuda_dev, precision, big=True))


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["f64", "f32"])
def test_split_entry_points(cuda_dev, precision):
    lengths = [64, 1000, 2047, 4100, 4208, 9216, 4097, 83040, 256000]
    print(precision, "Z worst %.3e" % SP.check_split_entry_points(cuda_dev, precision, lengths))


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["f64", "f32"])
def test_side_stream_schedule_equals_serial(cuda_dev, precision):
    print(precision, SP.check_schedules(cuda_dev, precision, big=True))


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["f64", "f32"])
def test_class_larger_than_one_launch(cuda_dev, precision):
    print(precision, "worst %.3e" % SP.check_big_class(cuda_dev, precision))


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["f64", "f32"])
def test_lengths_beyond_the_largest_bluestein_size_are_refused_on_the_device(cuda_dev, precision):
    for n in (2097153, 4194301):
        print(precision, SP.check_refused(cuda_dev, precision, n))


@pytest.mark.gpu
def test_render_with_a_grain_at_the_largest_bluestein_size(cuda_dev):
    """96 kHz at the 30 MHz design-rate cap with 51.7 ms grains: n = 1551000 = 517 * 3000, a Bluestein length with
    M = 2^22 in the default precision (f64), whose columns are 1024 rows long."""
    p = configs.with_defaults(base_sr=96000, time_unfold=400.0, micro_ms=51.7, event_process="Single")
    print("max-abs %.3e" % K.check_render(cuda_dev, p))
