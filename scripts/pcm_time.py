"""Cost of integer PCM export (`export_format`, `export_dither`) on the GPU.

Workloads, all f64: the C5 sweep (4096 renders, 48 kHz) and C4 (one 96 kHz render), each as float32 (ms_post) and as pcm16
and pcm24 with dither off and on (ms_post_pcm).  Per workload:
  * the post stage alone, CUDA events around `reps` calls;
  * the kernels of one step from torch.profiler in a separate pass: PostMaxK, PostWriteK, PostWritePcmK;
  * for the write pass: bytes from the shapes.  It reads 16 bytes per frame (two f64 channels) and stores 8 (float32),
    4 (pcm16) or 6 (pcm24) bytes per frame.
And render_batch end to end on the C5 sweep as float32, pcm16 and pcm24 (dither on), alternating, host clock, each call
ending with its device->host copy complete, with the bytes each format copies.  Writes JSON (GPU name and power limit
read in the same run).

    python scripts/pcm_time.py --out profiles/pcm_time_b200.json
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
FORMATS = (("float32", None), ("pcm16", False), ("pcm16", True), ("pcm24", False), ("pcm24", True))
STORE_BYTES = {"float32": 8, "pcm16": 4, "pcm24": 6}


def workloads():
    from audio_suite_b200 import configs
    c5 = [configs.c5_params(i) for i in range(4096)]
    c4 = configs.canonical("C4")
    out = {}
    for fmt, dither in FORMATS:
        tag = fmt if dither is None else "%s-dither%d" % (fmt, dither)
        extra = dict(export_format=fmt) if dither is None else dict(export_format=fmt, export_dither=dither)
        out["C5-sweep/" + tag] = (fmt, [dict(p, **extra) for p in c5])
        out["C4/" + tag] = (fmt, [dict(c4, **extra)])
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


def measure(dev, fmt, plist, reps):
    import torch
    from torch.profiler import ProfilerActivity, profile
    from audio_suite_b200 import engine
    br = engine.BatchRenderer(plist, device=dev, precision="f64")
    try:
        t, st, api = br.tables, dev.stream_ptr(), br.api
        br.run()
        if br.n_pcm:
            [g] = br.pcm_groups
            assert br.n_plain == 0 and g["n"] == br.n_renders and g["d_export"] is None

            def post():
                return api.ms_post_pcm(dev.ptr(g["d_post"]), dev.ptr(g["d_pcm"]), None, g["n"], g["max_n"], 0, g["bits"], g["dither"],
                                       dev.ptr(br.mono), dev.ptr(br.maxbits), None, dev.ptr(br.out), st)
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
            k = next((k for k in ("PostWritePcmK", "PostWriteK", "PostMaxK") if k in e.key), None)
            if k and tt:
                kern[k] = kern.get(k, 0.0) + tt / 1e3
        n = int(t.post["n"].sum())
        res = dict(renders=len(plist), frames=n, out_bytes=8 * int(t.frames), post_stage_ms=post_ms, kernels_ms=kern)
        w = "PostWriteK" if fmt == "float32" else "PostWritePcmK"
        if w in kern:
            b = 16 * n + STORE_BYTES[fmt] * n
            res[w] = dict(bytes=b, GB_per_s=b / kern[w] / 1e6, bytes_over_hbm_peak_ms=1e3 * b / HBM_BYTES_PER_S)
        return res
    finally:
        br.close()


def end_to_end(dev, reps):
    """render_batch of the C5 sweep as float32, pcm16 and pcm24 (dither on), alternating; ms per sweep and device->host bytes."""
    import torch
    from audio_suite_b200 import configs, engine, plan as P
    c5 = [configs.c5_params(i) for i in range(4096)]
    arms = {fmt: [dict(p, export_format=fmt) for p in c5] for fmt in ("float32", "pcm16", "pcm24")}
    hosts, times, digest = {}, {k: [] for k in arms}, {}
    for k, plist in arms.items():                     # warm-up, and the pinned output buffers
        outs = engine.render_batch(plist, device=dev)
        bits = None if k == "float32" else int(k[3:])
        slots = sum(P.output_slots(o.shape[0], bits) for o in outs)
        hosts[k] = (torch.empty(2 * slots, dtype=torch.float32).pin_memory(), slots, sum(o.shape[0] for o in outs))
        digest[k] = [str(outs[0].dtype), list(outs[0].shape)]
    for _ in range(reps):
        for k, plist in arms.items():
            t0 = time.perf_counter()
            engine.render_batch(plist, device=dev, host_out=hosts[k][0])
            times[k].append(1e3 * (time.perf_counter() - t0))
    out = {}
    for k in arms:
        ms = sorted(times[k])
        out[k] = dict(frames=hosts[k][2], slots=hosts[k][1], d2h_bytes=8 * hosts[k][1], dtype_shape0=digest[k], ms=times[k],
                      median_ms=ms[len(ms) // 2], min_ms=ms[0], max_ms=ms[-1], spread_ms=ms[-1] - ms[0])
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "pcm_time_b200.json"))
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--e2e-reps", type=int, default=7)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("pcm_time.py measures on a CUDA device; none found")
    from audio_suite_b200 import engine
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    dev = engine.CudaDevice(0)
    res = {}
    for name, (fmt, plist) in workloads().items():
        res[name] = measure(dev, fmt, plist, args.reps)
        print(json.dumps({name: res[name]}), flush=True)
    e2e = end_to_end(dev, args.e2e_reps)
    print(json.dumps({"render_batch": e2e}), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(dict(gpu=q.stdout.strip(), torch=torch.__version__, precision="f64", reps=args.reps, workloads=res,
                       render_batch_c5=e2e), f, indent=1)


if __name__ == "__main__":
    main()
