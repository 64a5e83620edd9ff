#!/usr/bin/env python
"""bench.py -- Microsound batched preset sweep (BASELINE.json configs[4], "C5"): 4096 randomised-parameter
renders (2 s stereo @ 48 kHz each, design SR 1.2-9.6 MHz, five generator modes, band-limit, spectral
stretch, reflection cloud + 8192-tap IR, stereo diffusion, soft clip, normalise), partitioned by render
index over the GPUs of one box.

  python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
  python bench.py --impl reference --gpus N --steps K ...  # the reference algorithm on the host cores

One step = one pass of the whole render pipeline over the batch.  `value` = rendered stereo samples
per second (2 x output frames) with all plan tables resident in HBM; `e2e` = the same through the
public API from host parameter dicts to host float32 audio (planning, H2D, kernels, D2H all timed).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

FRAMES_PER_RENDER = 96000
METRIC = "microsound_rendered_samples_per_s"
UNIT = "samples/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--renders", type=int, default=4096, help="renders in the sweep (total, all GPUs)")
    ap.add_argument("--precision", default="auto", choices=["auto", "f32", "f64"])
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--cpu-sample", type=int, default=48, help="renders timed for cpu_baseline (rank 0, N=1)")
    ap.add_argument("--chunk", type=int, default=384, help="renders per streamed slice of the end-to-end run (measured on B200, 4096 renders: "
                                                           "256 -> 81.5 ms, 320 -> 74.5, 384 -> 74.8, 512 -> 78.5, 768 -> 79.0, 1024 -> 78.5)")
    ap.add_argument("--slices", type=int, default=0,
                    help="N>1: parts per rank whose gather overlaps the next part's rendering; each part replays a CUDA graph of "
                         "its launch sequence, so small parts are not launch-bound.  0 = auto (1 at N=1, 4 at N>1)")
    ap.add_argument("--no-graph", action="store_true", help="N>1: launch the parts eagerly instead of replaying CUDA graphs")
    ap.add_argument("--no-pipeline", action="store_true", help="N>1: wait for each pass's gather before the next pass starts")
    ap.add_argument("--collective", default="peer_copy", choices=["gather", "all_gather", "peer_copy"],
                    help="N>1: how the rendered buffers reach rank 0 (parallel.PipelinedGather): peer_copy = every rank stores its slab "
                         "into rank 0's symmetric-memory buffer over NVLink with the copy engines (falls back to the NCCL gather, and "
                         "says so in config, if symmetric memory cannot be set up); gather / all_gather = NCCL")
    ap.add_argument("--no-gather", action="store_true", help="skip the NCCL gather of rendered buffers (N>1)")
    ap.add_argument("--config", default="C5", choices=["C1", "C1b", "C2", "C3", "C4", "C5"],
                    help="C5 (default) is the metric's workload; C1..C4 time ONE render of that BASELINE.json config: the kernel "
                         "sequence with the plan resident (value), render() from the parameter dict to the float64 result (e2e) "
                         "and the numpy port on one host core (cpu_baseline) -- single GPU only")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the audio the last timed step rendered to DIR/*.npy (float32, at most "
                         "64 MB; see dump_outputs).  The same arguments give the same inputs, so two builds compare value for value")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes this project's renders; the reference arm keeps none")
    return args


def workload_config(args, extra=None):
    cfg = {"workload": "C5 batched preset sweep: %d renders x 2.0 s stereo @48 kHz (BASELINE.json configs[4])" % args.renders,
           "renders": args.renders, "frames_per_render": FRAMES_PER_RENDER, "taps": "8192 IR + 320-tap reflection cloud",
           "parallelism": "renders partitioned by index, %d rank(s)" % args.gpus,
           "l2": "working set (GBs) exceeds the 126 MB L2; no flush needed"}
    if extra:
        cfg.update(extra)
    return cfg


DUMP_RENDER_BYTES = 32 << 20        # whole renders, picked by a fixed seed
DUMP_SAMPLES = 1 << 22              # float32 values at seeded positions across every render's output (16 MB)


def dump_outputs(path, parts, sizes, dist=None):
    """Writes what a caller of the timed path receives -- float32 stereo audio [frames, 2] per render -- to `path`:
    render_<i>.npy for whole renders of the sweep picked by a fixed seed (until 32 MB are written) and samples.npy,
    the values at DUMP_SAMPLES seeded positions of all renders' outputs laid end to end in sweep order.  The picks
    depend only on `sizes` (float32 values of every render of the sweep, by sweep index), so runs with the same
    arguments write the same positions however the renders are partitioned.  `parts` = [(BatchRenderer, [sweep index
    of each of its renders])] for the renders this process holds.  With `dist` (N>1) every rank calls this with its
    own renders: each writes the picked renders it holds, and rank 0 collects the samples."""
    import torch
    os.makedirs(path, exist_ok=True)
    part_of, local = np.full(len(sizes), -1), np.zeros(len(sizes), dtype=np.int64)
    for j, (b, index) in enumerate(parts):
        assert np.array_equal(2 * b.tables.out_n.astype(np.int64), sizes[index]), "render lengths differ from `sizes`"
        part_of[index], local[index] = j, np.arange(len(index))
    rng = np.random.default_rng(20260)
    left = DUMP_RENDER_BYTES
    for i in rng.permutation(len(sizes)):
        if 4 * sizes[i] <= left:
            left -= 4 * sizes[i]
            if part_of[i] >= 0:
                np.save(os.path.join(path, "render_%05d.npy" % i), parts[part_of[i]][0].output(local[i]).astype(np.float32))
    ends = np.cumsum(sizes)
    pos = np.sort(rng.integers(0, int(ends[-1]), min(DUMP_SAMPLES, int(ends[-1]))))
    i_of = np.searchsorted(ends, pos, side="right")
    held = np.flatnonzero(part_of[i_of] >= 0)
    values = np.empty(held.size, dtype=np.float32)
    for j, (b, _) in enumerate(parts):
        sel = part_of[i_of[held]] == j
        i = i_of[held[sel]]
        at = pos[held[sel]] - (ends - sizes)[i] + 2 * b.tables.out_at[local[i]].astype(np.int64)
        out = b.outputs_device()
        values[sel] = out[torch.from_numpy(at).to(out.device)].cpu().numpy()
    pieces = [(held, values)]
    if dist is not None:
        pieces = [None] * dist.get_world_size() if dist.get_rank() == 0 else None
        dist.gather_object((held, values), pieces, dst=0)
        if dist.get_rank() != 0:
            return
    samples = np.full(pos.size, np.nan, dtype=np.float32)
    for h, v in pieces:
        samples[h] = v
    assert not np.isnan(samples).any(), "some renders of the sweep are held by no rank"
    np.save(os.path.join(path, "samples.npy"), samples)


# ----------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None
        self.nvml, self.polled, self.alive, self.mx = None, [], False, 0.0

    def start(self):
        """NVML polled every 5 ms from a thread (a 10 ms step at N=8 still gets samples); nvidia-smi -lms as fallback."""
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml, self.h = pynvml, pynvml.nvmlDeviceGetHandleByIndex(int(self.index))
            self.mx = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.alive = True
            threading.Thread(target=self._poll, daemon=True).start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _poll(self):
        n = self.nvml
        bits = (("hw_slowdown", getattr(n, "nvmlClocksThrottleReasonHwSlowdown", 0x8)),
                ("hw_thermal_slowdown", getattr(n, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40)),
                ("sw_thermal_slowdown", getattr(n, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20)),
                ("sw_power_cap", getattr(n, "nvmlClocksThrottleReasonSwPowerCap", 0x4)))
        while self.alive:
            try:
                sm = float(n.nvmlDeviceGetClockInfo(self.h, n.NVML_CLOCK_SM))
                mask = int(n.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                self.polled.append((time.time(), sm, [name for name, b in bits if mask & b]))
            except Exception:
                pass
            time.sleep(0.005)

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        self.alive = False
        if self.proc:
            self.proc.terminate()
        sm, mx, reasons = [], self.mx, set()
        for t, mhz, names in self.polled:
            if t0 <= t <= t1:
                sm.append(mhz)
                reasons.update(names)
        for t, line in self.rows:
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 9:
                continue
            try:
                mx = max(mx, float(parts[2]))
                if t0 <= t <= t1:
                    sm.append(float(parts[1]))
                    for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), parts[5:9]):
                        if v.lower().startswith("active"):
                            reasons.add(name)
            except ValueError:
                continue
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm), "source": "nvml 5 ms poll" if self.nvml else "nvidia-smi -lms 20"}


# ----------------------------------------------------------------------------------------------- reference arm
def _ref_worker(idx):
    from audio_suite_b200 import configs
    from oracle import microsound_np as O
    out, _ = O.render(configs.c5_params(idx))
    return out.shape[0]


def cpu_pool_throughput(indices, procs):
    """samples/s of the numpy restatement of the reference over `indices`, `procs` worker processes."""
    import multiprocessing as mp
    os.environ.setdefault("OMP_NUM_THREADS", "1")
    os.environ.setdefault("OPENBLAS_NUM_THREADS", "1")
    if procs <= 1:
        t = time.perf_counter()
        frames = sum(_ref_worker(i) for i in indices)
        return 2.0 * frames / (time.perf_counter() - t)
    ctx = mp.get_context("fork")
    with ctx.Pool(procs) as pool:
        pool.map(_ref_worker, list(indices[:procs]))          # spin the workers up (imports, IR synthesis)
        t = time.perf_counter()
        frames = sum(pool.map(_ref_worker, list(indices), chunksize=1))
        dt = time.perf_counter() - t
    return 2.0 * frames / dt


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = len(os.sched_getaffinity(0))
    per_step = max(cores, min(2 * cores, 256))
    vals = []
    for s in range(args.warmup + args.steps):
        idx = [(s * per_step + i) % args.renders for i in range(per_step)]
        v = cpu_pool_throughput(idx, cores)
        if s >= args.warmup:
            vals.append(v)
    value = float(np.mean(vals))
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": len(vals),
            "warmup": args.warmup, "ms_per_step": 1e3 * per_step * FRAMES_PER_RENDER * 2 / value, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(args, {"sample_renders_per_step": per_step}),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                             "sample": "%d renders of the sweep per step, one worker process per core "
                                       "(oracle/microsound_np.py, verified <=2e-13 against the reference)" % per_step},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ----------------------------------------------------------------------------------------------- our arm
def algorithmic_bytes(br):
    """Compulsory traffic per stage (SURVEY.md 8d), element size = the precision actually used.
    Element counts are accumulated while the job tables are packed (tables.pack_chunk)."""
    es = 4 if br.precision == "f32" else 8
    a = br.tables.alg
    return {"synth": es * a["synth"], "tilt_spectral": es * a["tilt_spectral"], "grain_spectral": es * a["grain_spectral"],
            "overlap_add": es * a["overlap_add"], "fir_overlap_save": es * (a["fir_in"] + a["fir_taps"]),
            "post": es * a["post"] + 2 * 4 * a["post"] + 6 * 4 * a["post"]}


def run_ours(args):
    import torch
    import torch.distributed as dist
    from audio_suite_b200 import configs, engine, parallel

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = engine.CudaDevice(local)
    ir = configs.synth_ir(5.0, 48000, 303)
    if world > 1:
        # equal counts per rank (equal-shape slabs for the gather), near-equal predicted cost: every rank derives the same
        # partition from the parameters alone (parallel.param_cost), no communication
        everything = [configs.c5_params(i, shared_ir=ir) for i in range(args.renders)]
        owners = parallel.balanced_equal_partition([parallel.param_cost(p) for p in everything], world)
        mine = owners[rank]
        frames_per_rank = [len(o) * FRAMES_PER_RENDER for o in owners]
        params = [everything[i] for i in mine]
        del everything
    else:
        mine = list(range(args.renders))
        frames_per_rank = [len(mine) * FRAMES_PER_RENDER]
        params = [configs.c5_params(i, shared_ir=ir) for i in mine]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident plan: kernels only.  With several ranks every rank renders its share in `--slices` parts
    #      and the NCCL gather of part k runs while part k+1 renders (parallel.SlicedGather).
    gather = world > 1 and not args.no_gather
    equal = len(set(frames_per_rank)) == 1
    want = args.slices if args.slices > 0 else 1
    slices = want if (gather and len(mine) % want == 0 and equal) else 1
    # default at N>1: ONE part per rank, eager launches, and the gather of pass k overlapping pass k+1 (two output buffers,
    # parallel.PipelinedGather).  --slices S > 1: S parts per rank, each a CUDA-graph replay, the gather of part k overlapping
    # part k+1 of the SAME pass (parallel.SlicedGather) -- measured slower: parts render less efficiently than the whole.
    pipelined = gather and slices == 1 and equal and not args.no_pipeline
    use_graph = world > 1 and slices > 1 and not args.no_graph
    per = len(mine) // slices
    brs = [engine.BatchRenderer(params[k * per:(k + 1) * per], device=dev, precision=args.precision) for k in range(slices)]
    br = brs[0]
    sg = pg = None
    if pipelined:
        collective = args.collective
        if collective == "peer_copy":
            # all ranks must take the same branch: agree on whether symmetric memory came up everywhere
            try:
                pg = parallel.PipelinedGather(len(mine) * FRAMES_PER_RENDER, dist, rank, world, dev.dev, collective="peer_copy")
                okflag = 1
            except Exception as exc:                       # noqa: BLE001 -- reported, not hidden: config.collective says "gather"
                print("rank %d: symmetric memory unavailable (%s); NCCL gather instead" % (rank, exc), file=sys.stderr)
                pg, okflag = None, 0
            t = torch.tensor([okflag], dtype=torch.int32, device=dev.dev)
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
            if int(t.item()) == 0:
                collective, pg = "gather", None
        if pg is None:
            pg = parallel.PipelinedGather(len(mine) * FRAMES_PER_RENDER, dist, rank, world, dev.dev, collective=collective)
        outs = [br.out, torch.empty_like(br.out)]
    elif gather:
        sg = parallel.SlicedGather([per * FRAMES_PER_RENDER] * slices, dist, rank, world, dev.dev)
    if use_graph:
        for b in brs:
            b.capture()

    def step(mark=None, with_gather=True):
        if pg is not None:
            if with_gather:
                br.out = outs[pg.slot()]            # the buffer whose previous gather has completed
            br.run(mark)
            if with_gather:
                pg.start(br.outputs_device())
            return
        for k, b in enumerate(brs):
            if use_graph and mark is None:
                b.replay()
            else:
                b.run(mark)
            if sg is not None and with_gather:
                sg.start(k, b.outputs_device())
        if sg is not None and with_gather:
            sg.finish()

    def drain():
        if pg is not None:
            pg.finish()

    for _ in range(max(3, args.warmup)):
        step()
    drain()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    stage_names, stage_ev = [], []
    launches0 = dev.lib.ms_launch_count()
    barrier()
    torch.cuda.profiler.start()          # ncu --profile-from-start off captures exactly the timed steps
    wall0 = time.time()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for s in range(args.steps):
        evs = [torch.cuda.Event(enable_timing=True)]
        evs[0].record()
        names = []

        def mark(name, evs=evs, names=names):
            ev = torch.cuda.Event(enable_timing=True)
            ev.record()
            evs.append(ev)
            names.append(name)
        if use_graph:
            step()                      # graph replays: no per-stage events inside the timed region (taken below, untimed)
        else:
            step(mark)
            stage_names, _ = names, stage_ev.append(evs)
    drain()                             # the last pass's gather completes inside the timed region
    e1.record()
    barrier()
    torch.cuda.profiler.stop()
    wall1 = time.time()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, [(b, mine[k * per:(k + 1) * per]) for k, b in enumerate(brs)],
                     np.full(args.renders, 2 * FRAMES_PER_RENDER, dtype=np.int64), dist if world > 1 else None)
    render_only_ms = None
    if use_graph or gather:
        # the same steps without the gather (render only), and one eager pass for the per-stage events: both untimed extras
        barrier()
        r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        r0.record()
        for s in range(args.steps):
            step(with_gather=False)
        r1.record()
        barrier()
        t = torch.tensor([r0.elapsed_time(r1) / args.steps], dtype=torch.float64, device=dev.dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        render_only_ms = float(t.item())
        if use_graph:
            evs = [torch.cuda.Event(enable_timing=True)]
            evs[0].record()
            names = []

            def mark(name, evs=evs, names=names):
                ev = torch.cuda.Event(enable_timing=True)
                ev.record()
                evs.append(ev)
                names.append(name)
            for b in brs:
                b.run(mark)
            torch.cuda.synchronize()
            stage_names, stage_ev = names, [evs]
    launches = (dev.lib.ms_launch_count() - launches0) // args.steps
    if use_graph:
        launches = sum(b.graph_launches for b in brs)          # kernel nodes replayed per step (the library counter only sees captures)
    ms = e0.elapsed_time(e1) / args.steps
    t = torch.tensor([ms], dtype=torch.float64, device=dev.dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    clocks = sampler.stop(wall0, wall1) if rank == 0 else None
    stage_ms = {}
    for evs in stage_ev:
        for name, a, b in zip(stage_names, evs[:-1], evs[1:]):
            stage_ms[name] = stage_ms.get(name, 0.0) + a.elapsed_time(b) / len(stage_ev)
    if os.environ.get("MS_RANK_TIMES"):                 # every rank's own stage table (rank 0's goes into the JSON line)
        print("rank %d: step %.3f ms own clock, stages %s, renders %d" % (
            rank, ms, {k: round(v, 3) for k, v in stage_ms.items()}, len(mine)), file=sys.stderr, flush=True)

    # ---- individual kernels of one step: the library calls a hook after every launch, a CUDA event is recorded
    #      there (on the launching stream), consecutive events bracket one kernel.  Separate untimed steps, so
    #      the headline timing above carries no hook overhead.
    kernel_ms = {}
    if rank == 0:
        import re
        from audio_suite_b200 import _abi
        rec = []

        def _hook(name, stream):
            ev = torch.cuda.Event(enable_timing=True)
            ev.record()
            rec.append((name.decode(), ev))
        cb = _abi.LAUNCH_HOOK(_hook)
        import ctypes
        reps = max(1, min(3, args.steps))
        order = []
        for s in range(reps):
            rec.clear()
            first = torch.cuda.Event(enable_timing=True)
            first.record()
            dev.lib.ms_set_launch_hook(ctypes.cast(cb, ctypes.c_void_p))
            br.run()
            dev.lib.ms_set_launch_hook(None)
            torch.cuda.synchronize()
            prev = first
            for i, (name, ev) in enumerate(rec):
                m = re.search(r"K = (?:ms[fd]::)?([^;\]]+)", name)
                key = "%02d %s" % (i, m.group(1).strip() if m else name[-40:])
                if s == 0:
                    order.append(key)
                kernel_ms[key] = kernel_ms.get(key, 0.0) + prev.elapsed_time(ev) / reps
                prev = ev
        kernel_ms = {k: round(kernel_ms[k], 4) for k in order}

    # ---- end to end through the public API: host dicts -> host float32 audio
    h2d = d2h = 0
    e2e_ms = []
    host_out = torch.empty(2 * len(mine) * FRAMES_PER_RENDER, dtype=torch.float32).pin_memory()
    E2E_WARM = 3      # untimed: the first call starts the planning workers, the second sizes the per-slot device arenas, the third settles the allocator
    for s in range(E2E_WARM + args.e2e_steps if args.e2e_steps > 0 else 0):
        barrier()
        t0 = time.perf_counter()
        # public API: host parameter dicts in, host float32 audio out; planning (worker processes), table
        # uploads, kernels and the device->host drain overlap slice by slice (engine.render_batch)
        outs = engine.render_batch(params, device=dev, precision=args.precision, host_out=host_out, chunk=args.chunk)
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) * 1e3
        assert len(outs) == len(mine)
        h2d, d2h = engine.render_batch.last_h2d_bytes, host_out.numel() * 4
        if s >= E2E_WARM:
            e2e_ms.append(dt)
    t = torch.tensor([float(np.mean(e2e_ms)) if e2e_ms else float('nan')], dtype=torch.float64, device=dev.dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_ms_max = float(t.item())

    if rank == 0:
        total_samples = 2.0 * args.renders * FRAMES_PER_RENDER
        value = total_samples / (ms_max * 1e-3)
        alg = {}
        for b in brs:
            for k, v in algorithmic_bytes(b).items():
                alg[k] = alg.get(k, 0) + v
        dom = max(stage_ms, key=stage_ms.get)
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "MEASURED_PEAKS.json hbm_gbs (of measured)" if "hbm_gbs" in peaks else "6650 GB/s (of fallback)"
        stages = {k: {"ms": round(v, 4), "algorithmic_GB": round(alg.get(k, 0) / 1e9, 4),
                      "GBps": round(alg.get(k, 0) / 1e9 / (v * 1e-3), 1) if v > 0 else None,
                      "frac_of_hbm": round(alg.get(k, 0) / 1e9 / (v * 1e-3) / peak, 4) if v > 0 else None}
                  for k, v in stage_ms.items()}
        ach = alg.get(dom, 0) / 1e9 / (stage_ms[dom] * 1e-3)
        traffic, traffic_note = None, "no ncu capture committed"
        try:
            nt = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
            traffic = float(nt["dram_bytes_per_render"][dom]) * args.renders / world
            traffic_note = ("dram__bytes_read.sum + dram__bytes_write.sum of the stage's launches from profiles/%s "
                            "(%d renders profiled), scaled to this rank's %d renders" % (nt["source"], nt["renders_profiled"], args.renders // world))
        except Exception:
            pass
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
                "ms_per_step": ms_max, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": br.precision, "data": "synthetic",
                "config": workload_config(args, {"precision_rule": "auto = f64 (engine.choose_precision)" if args.precision == "auto" else args.precision,
                                                 "collective": (collective if pipelined else "gather") if gather else None,
                                                 "gather": (("every rank stores its rendered buffer into rank 0's symmetric-memory receive slab over NVLink (copy engines, symmetric-memory "
                                                             "barriers on a side stream)" if collective == "peer_copy" else "NCCL %s of the rendered buffers to rank 0" % collective) +
                                                            " inside the timed region; pass k is gathered while pass k+1 "
                                                            "renders into a second output buffer, the last gather completes before the closing event" if pipelined else
                                                            ("NCCL gather of rendered buffers to rank 0 inside the step, %d slices per rank, "
                                                             "slice k gathered while slice k+1 renders; %s" % (
                                                                 slices, "each slice replays a CUDA graph of its launch sequence" if use_graph else "eager launches"))) if gather else "none",
                                                 "partition": "equal counts, cost-balanced by parameters (parallel.balanced_equal_partition)" if world > 1 else "single rank",
                                                 "e2e_note": "at N>1 every rank drains its own shard to its own pinned host buffer: the end-to-end result stays sharded on the host (no gather)" if world > 1 else "single rank"}),
                "ms_per_step_render_only": render_only_ms,
                "frames_per_s": value / 2.0,
                "gpu_launches": int(launches),
                "clocks": clocks,
                "e2e": {"value": total_samples / (e2e_ms_max * 1e-3), "unit": UNIT, "ms_per_step": e2e_ms_max,
                        "steps": len(e2e_ms), "warmup": E2E_WARM, "ms_each_rank0": [round(x, 2) for x in e2e_ms],
                        "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                        "includes": "host planning (numpy's RNG streams restated natively, job tables), pinned H2D of tables, all kernels, D2H of float32 audio "
                                    "into pinned host memory; streamed in slices of %d renders so the three overlap" % args.chunk},
                "roofline": {"bound": "hbm", "kernel": dom, "achieved": round(ach, 1), "peak": peak, "unit": "GB/s",
                             "frac": round(ach / peak, 4), "traffic": traffic, "traffic_note": traffic_note,
                             "algorithmic_bytes": alg.get(dom, 0), "launches": "see kernels_ms", "peak_source": peak_src,
                             "note": "stage = consecutive launches of one pipeline stage, CUDA events on the launch stream; "
                                     "see profiles/ for the per-kernel ncu launch list.  \"hbm\" is the tier's accounting; the "
                                     "resource that binds the FFT-type kernels of these stages is the SM's L1 / shared-memory data pipe "
                                     "(ncu l1tex__data_pipe_lsu_wavefronts at 70-93 % of peak, DRAM at 5-54 %: profiles/r02_ncu_key_metrics.md)"},
                "stages": stages,
                "kernels_ms": kernel_ms}
        if world == 1 and args.cpu_sample > 0:
            idx = list(range(args.cpu_sample))
            v = cpu_pool_throughput(idx, 1)
            line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": 1, "kind": "port",
                                    "sample": "first %d renders of the sweep, serial like the reference's batch loop "
                                              "(main_v2.py:1578-1593), oracle/microsound_np.py" % args.cpu_sample}
        print(json.dumps(line))
    for b in brs:
        b.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_single_config(args):
    """One render of C1 / C1b / C2 / C3 / C4 (launch-latency-bound except C4): same JSON contract, N = 1."""
    import torch
    from audio_suite_b200 import configs, engine
    from oracle import microsound_np as O
    torch.cuda.set_device(0)
    dev = engine.CudaDevice(0)
    p = configs.canonical(args.config)
    br = engine.BatchRenderer([p], device=dev, precision=args.precision)
    frames = int(br.tables.frames)
    for _ in range(max(3, args.warmup)):
        br.run()
    torch.cuda.synchronize()
    sampler = ClockSampler(0)
    sampler.start()
    time.sleep(0.2)
    launches0 = dev.lib.ms_launch_count()
    wall0 = time.time()
    names, per_step = [], []
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for s in range(args.steps):
        evs = [torch.cuda.Event(enable_timing=True)]
        evs[0].record()
        names = []

        def mark(name, evs=evs, names=names):
            ev = torch.cuda.Event(enable_timing=True)
            ev.record()
            evs.append(ev)
            names.append(name)
        br.run(mark)
        per_step.append((names, evs))
    e1.record()
    torch.cuda.synchronize()
    wall1 = time.time()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, [(br, [0])], np.array([2 * frames], dtype=np.int64))
    ms = e0.elapsed_time(e1) / args.steps
    launches = (dev.lib.ms_launch_count() - launches0) // args.steps
    clocks = sampler.stop(wall0, wall1)
    stage_ms = {}
    for names, evs in per_step:
        for name, a, b in zip(names, evs[:-1], evs[1:]):
            stage_ms[name] = stage_ms.get(name, 0.0) + a.elapsed_time(b) / args.steps
    alg = algorithmic_bytes(br)
    br.close()
    lat, lat_cached = [], []
    for s in range(3 + max(1, args.e2e_steps)):
        t0 = time.perf_counter()
        out, meta = engine.render(p, device=dev, precision=args.precision, cache=False)       # plans from scratch every time
        if s >= 3:
            lat.append((time.perf_counter() - t0) * 1e3)
    for s in range(4 + max(1, args.e2e_steps)):
        t0 = time.perf_counter()
        out, meta = engine.render(p, device=dev, precision=args.precision)                    # unchanged settings: plan cache + graph replay
        if s >= 4:
            lat_cached.append((time.perf_counter() - t0) * 1e3)
    engine.clear_render_cache()
    reps = 1 if args.config == "C4" else 5
    t0 = time.perf_counter()
    for _ in range(reps):
        ref, _ = O.render(p)
    cpu_ms = (time.perf_counter() - t0) * 1e3 / reps
    err = float(np.max(np.abs(out[::7] - ref[::7])))
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    dom = max(stage_ms, key=stage_ms.get)
    ach = alg.get(dom, 0) / 1e9 / (stage_ms[dom] * 1e-3)
    total = 2.0 * frames
    e2e_ms = float(np.mean(lat))
    line = {"metric": METRIC, "value": total / (ms * 1e-3), "unit": UNIT, "n_gpus": 1, "steps": args.steps, "warmup": max(3, args.warmup),
            "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": br.precision, "data": "synthetic",
            "config": {"workload": "%s: one render of BASELINE.json's config (SURVEY.md Appendix D), %d stereo frames" % (args.config, frames),
                       "l2": "working set %s the 126 MB L2" % ("exceeds" if args.config == "C4" else "fits: these single renders are launch-latency-bound, not bandwidth-bound")},
            "gpu_launches": int(launches), "clocks": clocks,
            "e2e": {"value": total / (e2e_ms * 1e-3), "unit": UNIT, "ms_per_step": e2e_ms, "steps": len(lat), "warmup": 3,
                    "h2d_bytes_per_step": int(br.h2d_bytes), "d2h_bytes_per_step": int(frames * 2 * 4),
                    "includes": "render(params): planning, table upload, kernels, device->host copy, float64 (out_n, 2) result + meta",
                    "ms_when_settings_unchanged": float(np.mean(lat_cached)),
                    "note_unchanged": "same call again on unchanged parameters: the planned renderer is reused (plan cache) and the kernel "
                                      "sequence replays as one CUDA graph; the audio is recomputed every time"},
            "roofline": {"bound": "hbm", "kernel": dom, "achieved": round(ach, 1), "peak": peak, "unit": "GB/s", "frac": round(ach / peak, 4),
                         "traffic": None, "algorithmic_bytes": alg.get(dom, 0), "peak_source": "MEASURED_PEAKS.json hbm_gbs (of measured)" if "hbm_gbs" in peaks else "6650 GB/s (of fallback)"},
            "stages": {k: {"ms": round(v, 4), "algorithmic_GB": round(alg.get(k, 0) / 1e9, 4)} for k, v in stage_ms.items()},
            "cpu_baseline": {"value": total / (cpu_ms * 1e-3), "unit": UNIT, "cores": 1, "kind": "port", "ms": cpu_ms,
                             "sample": "the same single render, oracle/microsound_np.py, one core"},
            "max_abs_vs_oracle": err}
    print(json.dumps(line))


def main():
    args = parse()
    # rank 0 prints ONE JSON line on stdout and nothing else: libraries that write to file descriptor 1 (NCCL's version
    # banner) are sent to stderr while the bench runs; the saved descriptor gets the JSON line at the end
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)
    real_stdout = os.fdopen(saved, "w")
    import builtins
    _print = builtins.print

    def _json_print(*a, **k):
        k.setdefault("file", real_stdout)
        _print(*a, **k)
        real_stdout.flush()
    builtins.print = _json_print
    try:
        if args.impl == "reference":
            run_reference(args)
        elif args.config != "C5":
            run_single_config(args)
        else:
            run_ours(args)
    finally:
        builtins.print = _print


if __name__ == "__main__":
    main()
