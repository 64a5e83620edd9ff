"""Cost of true-stereo impulse responses (space_ir_stereo=True) on the GPU, against the same workloads in mono.

Workloads: the C5 sweep (4096 renders), C3, C4 with the default cap and C4 with its whole IR (space_ir_tap_cap=None); every
one of them has a two-channel IR.  Per workload and mode: ms_fir_run time and whole-step time (host clock around `reps`
runs that end in a device synchronise), the post stage's kernel time (PostMaxK + PostWriteK, plus the odd-length roll and
rotation, from torch.profiler in a separate pass) and the FIR kernels' times.  Beside each stereo FIR time: twice the mono
FIR time, the cost of running the two channels as independent rows.  Writes JSON (GPU name and power limit read in the
same run) to --out.

    python scripts/stereo_ir_time.py --out profiles/stereo_ir_time_b200.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def workloads():
    from audio_suite_b200 import configs
    return {"C5-sweep": [configs.c5_params(i) for i in range(4096)], "C3": [configs.canonical("C3")],
            "C4-capped": [configs.canonical("C4")], "C4-full-IR": [dict(configs.canonical("C4"), space_ir_tap_cap=None)]}


def _time(fn, reps):
    import torch
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        fn()
    torch.cuda.synchronize()
    return 1e3 * (time.perf_counter() - t0) / reps


def measure(dev, plist, reps):
    import torch
    from torch.profiler import ProfilerActivity, profile
    from audio_suite_b200 import engine
    br = engine.BatchRenderer(plist, device=dev, precision="f64")
    try:
        st = dev.stream_ptr()
        step_ms = _time(br.run, reps)
        fir_ms = _time(lambda: br.api.ms_fir_run(br.fir_handle, st), reps)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            br.run()
            torch.cuda.synchronize()
        kern = {}
        for e in prof.key_averages():
            t = getattr(e, "self_device_time_total", None) or getattr(e, "self_cuda_time_total", 0)
            if t:
                kern[e.key] = kern.get(e.key, 0.0) + t / 1e3
        post_ms = sum(v for k, v in kern.items() if "PostMaxK" in k or "PostWriteK" in k or "RollK" in k)
        fir_k = {k: v for k, v in kern.items() if "Fir" in k or "ErScatterK" in k}
        return dict(renders=len(plist), fir_rows=len(br.tables.fir), step_ms=step_ms, fir_ms=fir_ms, post_kernels_ms=post_ms,
                    fir_kernels_ms=dict(sorted(fir_k.items(), key=lambda kv: -kv[1])[:8]))
    finally:
        br.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "stereo_ir_time_b200.json"))
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--only", default="", help="comma-separated workload names (default: all)")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("stereo_ir_time.py measures on a CUDA device; none found")
    from audio_suite_b200 import engine
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    dev = engine.CudaDevice(0)
    res = {}
    for name, plist in workloads().items():
        if args.only and name not in args.only.split(","):
            continue
        mono = measure(dev, plist, args.reps)
        stereo = measure(dev, [dict(p, space_ir_stereo=True) for p in plist], args.reps)
        res[name] = dict(mono=mono, stereo=stereo, twice_mono_fir_ms=2 * mono["fir_ms"],
                         stereo_fir_over_twice_mono=stereo["fir_ms"] / (2 * mono["fir_ms"]))
        print(json.dumps({name: res[name]}))
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(dict(gpu=q.stdout.strip(), torch=torch.__version__, precision="f64", reps=args.reps, workloads=res), f, indent=1)


if __name__ == "__main__":
    main()
