"""Cost of the IR sample rate (`space_ir_sr`) on the GPU, in f64.

  * ms_resample_poly alone (CUDA events around `reps` calls on resident buffers) and decimate.resample_poly end to end
    (upload, kernel, download; host clock), for the shipped ir_tiny_room_250ms (48 kHz) at 96 kHz, and for the C3 and C4
    synthetic IRs taken as 44.1 kHz recordings at 48 / 96 / 192 kHz, mono (the mean of the columns) and stereo;
  * render() of C3 with a 44.1 kHz IR: the first call (resample, plan, upload, run) against the cached calls, with and
    without the key;
  * render_batch of the C5 sweep (4096 renders sharing one IR) with `space_ir_sr=44100` against the same sweep without
    the key, and, with --parent DIR, against the sweep as the parent commit's tree at DIR renders it (alternating).
Writes JSON with the GPU name and power limit read in the same run.

    python scripts/ir_rate_time.py --out profiles/ir_rate_time_b200.json [--parent DIR]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

SWEEP = r'''
import sys, time, json
sys.path.insert(0, %r)
import numpy as np
from audio_suite_b200 import configs, engine
dev = engine.CudaDevice(0)
ps = [configs.c5_params(i) for i in range(4096)]
key = %r
if key:
    ps = [dict(p, space_ir_sr=key) for p in ps]
engine.render_batch(ps, device=dev)                  # warm-up: modules, workers, arenas (and the resample cache)
ts = []
for _ in range(%d):
    t0 = time.perf_counter(); engine.render_batch(ps, device=dev); ts.append(time.perf_counter() - t0)
print(json.dumps(ts))
'''


def sweep(root, key, reps):
    out = subprocess.run([sys.executable, "-c", SWEEP % (root, key, reps)], capture_output=True, text=True, cwd=root)
    if out.returncode:
        raise RuntimeError(out.stderr[-3000:])
    return json.loads(out.stdout.strip().splitlines()[-1])


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "ir_rate_time_b200.json"))
    ap.add_argument("--parent", default=None, help="tree of the parent commit, built, for the sweep comparison")
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--sweep-reps", type=int, default=5)
    args = ap.parse_args()
    sys.path.insert(0, ROOT)
    import numpy as np
    import torch
    if not torch.cuda.is_available():
        sys.exit("ir_rate_time.py measures on a CUDA device; none found")
    from audio_suite_b200 import _abi, configs, decimate, engine
    dev = engine.CudaDevice(0)
    api = _abi.Api(dev.lib, "f64")
    res = {"gpu": gpu_info(), "precision": "f64", "resample": [], "render_c3": {}, "c5_sweep": {}}

    g = np.load(os.path.join(ROOT, "tests", "golden", "presets.npz"))
    room = np.array(g["ir_ir_tiny_room_250ms.wav"])
    c3_ir, c4_ir = configs.canonical("C3")["_ir_audio"], configs.canonical("C4")["_ir_audio"]
    cases = [("ir_tiny_room_250ms mono", room, 48000, 96000)]
    for name, ir in (("C3 IR (240000 x 2)", c3_ir), ("C4 IR (960000 x 2)", c4_ir)):
        for base in (48000, 96000, 192000):
            cases.append((name + " mono", ir.mean(axis=1), 44100, base))
            cases.append((name + " stereo", ir, 44100, base))
    for name, ir, sr, base in cases:
        import math
        gg = math.gcd(sr, base)
        up, down = base // gg, sr // gg
        x2 = np.ascontiguousarray(np.atleast_2d(ir.T if ir.ndim > 1 else ir))
        s, n = x2.shape
        n_out = -(-n * up // down)
        half, taps, bank = decimate.polyphase_bank(up, down)
        dx, db, dy = dev.upload(x2), dev.upload(bank), dev.zeros(s * n_out, np.float64)
        st = dev.stream_ptr()

        def call():
            _abi.check(api.ms_resample_poly(dev.ptr(dx), n, n, s, dev.ptr(db), up, down, half, taps, dev.ptr(dy), n_out, n_out, st), dev.lib)
        call()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(args.reps):
            call()
        b.record()
        b.synchronize()
        k_ms = a.elapsed_time(b) / args.reps
        e2e = []
        for _ in range(5):
            t0 = time.perf_counter()
            decimate.resample_poly(ir, up, down, dev, "f64")
            e2e.append(time.perf_counter() - t0)
        row = {"ir": name, "from_sr": sr, "to_sr": base, "up": up, "down": down, "taps_per_phase": taps, "signals": s,
               "in_samples": n, "out_samples": n_out, "kernel_ms": k_ms, "wrapper_ms_median": 1e3 * float(np.median(e2e)),
               "fma_per_s": s * n_out * taps / (k_ms * 1e-3)}
        res["resample"].append(row)
        print(json.dumps(row), flush=True)

    c3 = dict(configs.canonical("C3"), _ir_audio=configs.synth_ir(5.0, 44100, 303))
    for label, p in (("with space_ir_sr=44100", dict(c3, space_ir_sr=44100)), ("without the key", c3)):
        engine.clear_render_cache()
        engine._IR_RATE_CACHE.clear()
        t0 = time.perf_counter()
        engine.render(p, device=dev)
        first = time.perf_counter() - t0
        cached = []
        for _ in range(5):
            t0 = time.perf_counter()
            engine.render(p, device=dev)
            cached.append(time.perf_counter() - t0)
        res["render_c3"][label] = {"first_ms": 1e3 * first, "cached_ms_median": 1e3 * float(np.median(cached))}
        print(label, res["render_c3"][label], flush=True)
    engine.clear_render_cache()

    arms = [("this tree, space_ir_sr=44100", ROOT, 44100), ("this tree, no key", ROOT, None)]
    if args.parent:
        arms.append(("parent commit, no key", os.path.abspath(args.parent), None))
    times = {a[0]: [] for a in arms}
    for _ in range(2):                                   # alternate the arms
        for label, root, key in arms:
            times[label] += sweep(root, key, args.sweep_reps)
    for label, ts in times.items():
        res["c5_sweep"][label] = {"render_batch_ms": [1e3 * t for t in ts], "median_ms": 1e3 * float(np.median(ts))}
        print(label, res["c5_sweep"][label]["median_ms"], flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
