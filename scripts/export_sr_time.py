"""Cost of the export sample rate (`export_sr`) on the GPU.

Workloads: the C5 sweep (4096 renders, 48 kHz) delivered at 48 kHz, 44.1 kHz and 16 kHz, and C4 (96 kHz) delivered at
96 kHz, 48 kHz and 44.1 kHz, all in f64.  Per workload:
  * the post stage alone (ms_post, or ms_post_export for an export rate), CUDA events around `reps` calls;
  * the kernels of one step from torch.profiler in a separate pass: PostMaxK, PostWriteK, PostExportK;
  * for the resampling pass (PostExportK) and the plain write pass (PostWriteK): bytes and FMAs from the shapes, and the
    rates those give.  Both read 16 bytes per input frame (two f64 channels); the write pass stores 8 bytes per input
    frame, the resampling pass 8 bytes per output frame and forms 2 * taps FMAs per output frame.
And render_batch end to end for the C5 sweep at 48 kHz against 16 kHz (alternating, host clock, each call ends with the
device->host copy complete), with the bytes that copy moves.  Writes JSON (GPU name and power limit read in the same run).

    python scripts/export_sr_time.py --out profiles/export_sr_time_b200.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM_BYTES_PER_S = 7.7e12            # HGX B200 data sheet, one GPU (a bound, not a measurement)


def workloads():
    from audio_suite_b200 import configs
    c5 = [configs.c5_params(i) for i in range(4096)]
    c4 = configs.canonical("C4")
    out = {}
    for ex in (None, 44100, 16000):
        out["C5-sweep@%s" % (ex or 48000)] = [dict(p, export_sr=ex) for p in c5]
    for ex in (None, 48000, 44100):
        out["C4@%s" % (ex or 96000)] = [dict(c4, export_sr=ex)]
    return out


def _events(fn, reps):
    import torch
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps


def measure(dev, plist, reps):
    import numpy as np
    import torch
    from torch.profiler import ProfilerActivity, profile
    from audio_suite_b200 import engine
    br = engine.BatchRenderer(plist, device=dev, precision="f64")
    try:
        t, st, api = br.tables, dev.stream_ptr(), br.api
        br.run()
        if br.n_export:
            assert br.n_plain == 0

            def post():
                return api.ms_post_export(dev.ptr(br.d_post_export), dev.ptr(br.d_export), br.n_export, br.max_n_export,
                                          br.max_out_export, dev.ptr(br.mono), dev.ptr(br.maxbits), dev.ptr(br.d_bank), dev.ptr(br.out), st)
        else:
            def post():
                return api.ms_post(dev.ptr(br.d_post), br.n_renders, br.max_out_n, dev.ptr(br.mono), dev.ptr(br.maxbits), dev.ptr(br.out), st)
        post_ms = _events(post, reps)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            br.run()
            torch.cuda.synchronize()
        kern = {}
        for e in prof.key_averages():
            tt = getattr(e, "self_device_time_total", None) or getattr(e, "self_cuda_time_total", 0)
            for k in ("PostMaxK", "PostWriteK", "PostExportK"):
                if k in e.key and tt:
                    kern[k] = kern.get(k, 0.0) + tt / 1e3
        n_in = int(t.post["n"].sum())
        n_out = int(t.out_n.sum())
        res = dict(renders=len(plist), input_frames=n_in, output_frames=n_out, post_stage_ms=post_ms, kernels_ms=kern)
        if "PostWriteK" in kern:
            b = 16 * n_in + 8 * n_in
            res["PostWriteK"] = dict(bytes=b, GB_per_s=b / kern["PostWriteK"] / 1e6, bytes_over_hbm_peak_ms=1e3 * b / HBM_BYTES_PER_S)
        if "PostExportK" in kern:
            taps = t.export["rate"][:, 3].astype(np.int64)
            outs = (t.export["out_end"] - t.export["out"]).astype(np.int64)
            fma = int(np.sum(2 * taps * outs))
            b = 16 * n_in + 8 * n_out
            ms = kern["PostExportK"]
            res["PostExportK"] = dict(bytes=b, fma=fma, taps_per_phase=sorted(set(taps.tolist())), GB_per_s=b / ms / 1e6,
                                      GFMA_per_s=fma / ms / 1e6, bytes_over_hbm_peak_ms=1e3 * b / HBM_BYTES_PER_S)
        return res
    finally:
        br.close()


def end_to_end(dev, reps):
    """render_batch of the C5 sweep at 48 kHz and at export 16 kHz, alternating; ms per sweep and device->host bytes."""
    import torch
    from audio_suite_b200 import configs, engine
    c5 = [configs.c5_params(i) for i in range(4096)]
    arms = {"48000": c5, "16000": [dict(p, export_sr=16000) for p in c5]}
    hosts, times = {}, {k: [] for k in arms}
    for k, plist in arms.items():                     # warm-up, and the pinned output buffers
        outs = engine.render_batch(plist, device=dev)
        frames = sum(o.shape[0] for o in outs)
        hosts[k] = (torch.empty(2 * frames, dtype=torch.float32).pin_memory(), frames)
    for _ in range(reps):
        for k, plist in arms.items():
            t0 = time.perf_counter()
            engine.render_batch(plist, device=dev, host_out=hosts[k][0])
            times[k].append(1e3 * (time.perf_counter() - t0))
    return {k: dict(frames=hosts[k][1], d2h_bytes=8 * hosts[k][1], ms=times[k], median_ms=sorted(times[k])[len(times[k]) // 2])
            for k in arms}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "export_sr_time_b200.json"))
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--e2e-reps", type=int, default=5)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("export_sr_time.py measures on a CUDA device; none found")
    from audio_suite_b200 import engine
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    dev = engine.CudaDevice(0)
    res = {}
    for name, plist in workloads().items():
        res[name] = measure(dev, plist, args.reps)
        print(json.dumps({name: res[name]}), flush=True)
    e2e = end_to_end(dev, args.e2e_reps)
    print(json.dumps({"render_batch": e2e}), flush=True)
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(dict(gpu=q.stdout.strip(), torch=torch.__version__, precision="f64", reps=args.reps, workloads=res,
                       render_batch_c5=e2e), f, indent=1)


if __name__ == "__main__":
    main()
