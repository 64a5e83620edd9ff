"""FIR-stage time of the partitioned route for long impulse responses (space_ir_tap_cap=None) on the GPU.

Workloads: C4 with its whole 10 s IR (960000 taps, 57.6 M frames), C3 with its 5 s IR over a 60 s output, and the C5 sweep
(4096 x 96000 frames) with the shared 5 s IR uncapped (clipped per render to <= 96000 taps); C4 with the default cap beside
them.  For every partition length of the sweep (MS_FIR_PART, read once per process by the CUDA build: one child process
each) and for the library's own choice: ms_fir_run time (host clock around `reps` runs that end in a device synchronise),
the MAC kernel's own time (torch.profiler, a separate pass), algorithmic bytes / FLOPs from shapes, and GB/s against the
peak bench.py uses.  Writes JSON (GPU name and power limit read in the same run) to --out.

    python scripts/long_ir_time.py --out profiles/long_ir_time_b200.json
"""
import argparse
import json
import math
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

PARTS = (0, 4096, 8192, 16384, 32768, 65536)           # 0: the library's rule


def workloads():
    from audio_suite_b200 import configs
    c4 = dict(configs.canonical("C4"), space_ir_tap_cap=None)
    c3 = dict(configs.canonical("C3"), space_ir_tap_cap=None, out_dur_s=60.0)
    c5 = [dict(configs.c5_params(i), space_ir_tap_cap=None) for i in range(4096)]
    return {"C4-full-IR": [c4], "C3-60s": [c3], "C5-uncapped": c5, "C4-capped": [configs.canonical("C4")]}


def rule_part(h, out_n, w_mac=0.05):
    """ms_stage_api.inl fir_long_part, restated to report which P the rule picks."""
    best, best_cost = 0, 0.0
    for P in (4096, 8192, 16384, 32768, 65536):
        J = -(-out_n // P); Jh = (J + 1) // 2; K = -(-h // P); head = min(K - 1, Jh)
        cost = (2 * Jh + head) * 2.0 * P + w_mac * Jh * K * 2.0 * P
        if not best or cost < best_cost:
            best, best_cost = P, cost
    return best


def shapes(fir, part, real_bytes):
    """Algorithmic bytes and FLOPs of the long rows of a FIR table at partition `part` (0: the rule)."""
    cpx = 2 * real_bytes
    nbytes = flops = 0.0
    parts = set()
    for f in fir:
        ir_len, out_n, xb = int(f["ir_len"]), int(f["out_n"]), int(f["x_begin"])
        if ir_len <= 8192:
            continue
        h = max(1, min(ir_len, out_n - xb))
        P = part or rule_part(h, out_n)
        parts.add(P)
        N = 2 * P; J = -(-out_n // P); Jh = (J + 1) // 2; K = -(-h // P); head = min(K - 1, Jh)
        ent = Jh + head
        nbytes += 2 * out_n * real_bytes                 # input read, output written
        nbytes += 2 * ent * N * cpx + 2 * Jh * N * cpx   # Z written + read, Y written + read
        nbytes += K * N * cpx                            # partition spectra, once
        flops += 8.0 * Jh * K * N + 5.0 * N * math.log2(N) * (ent + Jh)
    return nbytes, flops, sorted(parts)


def child(reps):
    import torch
    from audio_suite_b200 import engine
    dev = engine.CudaDevice(0)
    part = int(os.environ.get("MS_FIR_PART", "0"))
    out = {}
    for name, plist in workloads().items():
        if name == "C4-capped" and part:
            continue
        br = engine.BatchRenderer(plist, device=dev, precision="f64")
        try:
            br.run()
            torch.cuda.synchronize()
            st = dev.stream_ptr()
            for _ in range(2):
                assert br.api.ms_fir_run(br.fir_handle, st) == 0
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(reps):
                br.api.ms_fir_run(br.fir_handle, st)
            torch.cuda.synchronize()
            stage_ms = 1e3 * (time.perf_counter() - t0) / reps
            from torch.profiler import ProfilerActivity, profile
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                br.api.ms_fir_run(br.fir_handle, st)
                torch.cuda.synchronize()
            kern = {}
            for e in prof.key_averages():
                if e.device_type.name == "CUDA" or getattr(e, "self_device_time_total", 0):
                    t = getattr(e, "self_device_time_total", None) or getattr(e, "self_cuda_time_total", 0)
                    kern[e.key] = kern.get(e.key, 0.0) + t / 1e3
            mac_ms = sum(v for k, v in kern.items() if "FirLongMacK" in k)
            nbytes, flops, parts = shapes(br.tables.fir, part, 8)
            out[name] = dict(renders=len(plist), frames=int(sum(int(f["out_n"]) for f in br.tables.fir)), fir_stage_ms=stage_ms,
                             mac_ms=mac_ms, kernels_ms={k: v for k, v in sorted(kern.items(), key=lambda kv: -kv[1])[:8]},
                             algorithmic_bytes=nbytes, algorithmic_flops=flops, parts=parts)
        finally:
            br.close()
    print(json.dumps(dict(part=part, results=out)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "long_ir_time.json"))
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--parts", default=",".join(str(p) for p in PARTS))
    ap.add_argument("--child", action="store_true")
    args = ap.parse_args()
    if args.child:
        return child(args.reps)
    import torch
    if not torch.cuda.is_available():
        sys.exit("long_ir_time.py measures on a CUDA device; none found")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        peaks = {}
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "MEASURED_PEAKS.json hbm_gbs" if "hbm_gbs" in peaks else "6650 GB/s fallback of bench.py"
    runs = []
    for part in [int(p) for p in args.parts.split(",")]:
        env = dict(os.environ)
        env.pop("MS_FIR_PART", None)
        if part:
            env["MS_FIR_PART"] = str(part)
        p = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", "--reps", str(args.reps)], env=env,
                           capture_output=True, text=True, cwd=ROOT)
        if p.returncode:
            runs.append(dict(part=part, error=p.stderr[-3000:]))
            continue
        r = json.loads(p.stdout.strip().splitlines()[-1])
        for w in r["results"].values():
            w["achieved_gbs"] = w["algorithmic_bytes"] / (w["fir_stage_ms"] * 1e-3) / 1e9
            w["share_of_peak"] = w["achieved_gbs"] / peak
        runs.append(r)
        print(json.dumps(r))
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(dict(gpu=q.stdout.strip(), torch=torch.__version__, peak_gbs=peak, peak_source=peak_src, precision="f64",
                       capped_c4_fir_stage_ms_r02=1.01, runs=runs), f, indent=1)


if __name__ == "__main__":
    main()
