"""Regenerates profiles/README.md from the artefacts committed beside it (round 2)."""
import io
import json
import os

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
P = os.path.join(ROOT, "profiles")
load = lambda name: json.load(open(os.path.join(P, name)))
d, r = load("r02_bench_n1.json"), load("r02_bench_ref.json")
r1 = load("bench_r01i_n1.json")
o = io.StringIO()
w = lambda *a: print(*a, file=o)
w("# profiles/ — round 2 measurements (B200, sm_100a, CUDA 12.9, driver 580)\n")
w("All runs: `gpurun` on fresh B200 boxes; timed numbers come from `bench.py` (CUDA events, no profiler); ncu numbers are")
w("cold-cache / serialised and are used for *shares* and counters only.  Regenerate this file with `python scripts/profiles_readme.py`.")
w("Round-1 artefacts (`*_r01*`) are kept for the history; everything named `r02_*` is the final build of round 2.\n")
w("## 1. bench.py, C5 sweep (4096 renders x 96000 stereo frames, f64), N = 1 (`r02_bench_n1.json`, `r02_bench_ref.json`)\n")
e = d["e2e"]
w("* `value` (plan resident in HBM): **%.3e samples/s** (%.2f ms/step), %d kernel launches/step, SM clock %s MHz, throttle reasons %s" % (
    d["value"], d["ms_per_step"], d["gpu_launches"], d["clocks"]["sm_mhz"], d["clocks"]["reasons"]))
w("* `e2e` (host dicts -> pinned host float32 audio, `render_batch`): **%.3e samples/s** (%.1f ms/step, runs %s; H2D %.1f MB, D2H %.2f GB)" % (
    e["value"], e["ms_per_step"], e.get("ms_each_rank0"), e["h2d_bytes_per_step"] / 1e6, e["d2h_bytes_per_step"] / 1e9))
w("* `cpu_baseline` (oracle port, 1 core): %.3e samples/s;  `--impl reference` (oracle port, %d cores): %.3e samples/s" % (
    d["cpu_baseline"]["value"], r["cpu_baseline"]["cores"], r["value"]))
w("* e2e / reference-arm = **%.0fx**;  value / reference-arm = %.0fx  (same box, back to back)" % (e["value"] / r["value"], d["value"] / r["value"]))
w("* history of the same metric (ms/step, kernels | e2e): round 1 first run 84.9 | 252 -> round 1 final %.1f | %.0f -> round 2 final **%.2f | %.0f**\n" % (
    r1["ms_per_step"], r1["e2e"]["ms_per_step"], d["ms_per_step"], e["ms_per_step"]))
w("| stage | round 1 ms | round 2 ms | algorithmic GB | GB/s | fraction of measured HBM peak (%.1f GB/s) |" % d["roofline"]["peak"])
w("|---|---|---|---|---|---|")
for k, v in d["stages"].items():
    w("| %s | %.2f | **%.2f** | %.2f | %.1f | %.4f |" % (k, r1["stages"][k]["ms"], v["ms"], v["algorithmic_GB"], v["GBps"] or 0, v["frac_of_hbm"] or 0))
w("")
rf = d["roofline"]
w("`roofline` of the dominant stage (%s): achieved %.1f GB/s of %.1f (frac %.4f); algorithmic bytes %.2f GB, measured DRAM traffic %.2f GB (%s).  "
  "The HBM fraction is small because **no FFT-type kernel here is DRAM-bound: they run at 70-93 %% of the SM's L1 / shared-memory data pipe** "
  "(section 3) -- that pipe, not HBM or the FP64 units, is the roofline these kernels sit under.\n" % (
      rf["kernel"], rf["achieved"], rf["peak"], rf["frac"], rf["algorithmic_bytes"] / 1e9, (rf["traffic"] or 0) / 1e9, rf["traffic_note"]))
w("### Every launch of one step, timed live (CUDA event after each launch via `ms_set_launch_hook`; the length classes of a spectral stage run one after the other in this mode)\n")
w("`ColsWarpK / ColsWarp512K / ColsWarpPlainK<LD, ST, TWID>`: warp-local column transforms (in-tile Bluestein of 256 / 512, plain 256); "
  "`ColsK<LD, ST, TWID, SB>` / `RowsK<LD, MODE, ST>`: block-wide tiles; `SpecOpK`: the spectral operators, elementwise.\n")
w("| # kernel | ms |\n|---|---|")
for k, v in d["kernels_ms"].items():
    w("| %s | %.3f |" % (k, v))
w("")
w("### 1 / 2 / 4 / 8 GPUs (`torchrun`, one rank per GPU; strong scaling: 4096 renders in total; `r02_bench_n{1,2,4,8}.json`)\n")
w("Every rank stores its rendered float32 buffer into rank 0's symmetric-memory receive slab over NVLink (copy engines) inside the timed region; "
  "pass k is gathered while pass k+1 renders.\n")
w("| N | ms/step | render only ms | samples/s | speed-up | efficiency | round 1 ms/step | e2e ms/step |\n|---|---|---|---|---|---|---|---|")
base = None
for n in (1, 2, 4, 8):
    x = load("r02_bench_n%d.json" % n)
    y = load("bench_r01i_n%d.json" % n)
    base = base or x["value"]
    w("| %d | %.2f | %s | %.3e | %.2fx | %.3f | %.2f | %.1f |" % (
        n, x["ms_per_step"], ("%.2f" % x["ms_per_step_render_only"]) if x.get("ms_per_step_render_only") else "-", x["value"], x["value"] / base,
        x["value"] / base / n, y["ms_per_step"], x["e2e"]["ms_per_step"]))
w("")
w("Where the 8-GPU step goes (per-rank CUDA events, `MS_RANK_TIMES=1`): a rank renders its 512 renders in about 4.2-4.4 ms alone (the ideal share is 3.7 ms: "
  "sixty launches over an eighth of the batch leave partial waves); with the gather in flight every rank's kernels take 0.45-0.5 ms longer and the "
  "ranks are coupled pass by pass through the gather's barriers (4.9 ms).  NCCL's gather in place of the peer copies: 6.0 ms; without the overlap: 9.0 ms.  "
  "End to end the multi-GPU runs are bound by the host: eight GPUs draining to pinned host memory at once get about 12 GB/s each "
  "(~100 GB/s in total on these boxes, against 50 GB/s for one GPU alone), so 3.15 GB of audio cost ~32 ms whatever N >= 2 is.\n")
w("### The other BASELINE.json configs, one render each (`r02_bench_C*.json`, `bench.py --config`)\n")
w("| config | kernels ms (graph replay) | render() ms end to end | numpy oracle on one host core, samples/s | launches |\n|---|---|---|---|---|")
for c in ("C1b", "C1", "C2", "C3", "C4"):
    x = load("r02_bench_%s.json" % c)
    w("| %s | %.3f | %.2f | %.3e | %s |" % (c, x["ms_per_step"], x["e2e"]["ms_per_step"], x["cpu_baseline"]["value"], x.get("gpu_launches")))
w("")
w("C1-C3 are launch-latency-sized (a few hundred KB of data); `render()` is dominated by Python (plan cache lookup, one D2H, the float64 copy the reference returns).  "
  "C4 (57.6 M frames): 21 ms of kernels; `render()` spends the rest bringing the 922 MB float64 array the reference's signature promises to pageable host memory.\n")
w("## 2. ncu launch list of one step, 512-render slab (`launches_r02_512renders.csv`, table in `r02_launch_table.md`)\n")
w("`ncu --profile-from-start off --metrics gpu__time_duration.sum,dram__bytes_read.sum,dram__bytes_write.sum --clock-control none` around the timed step of "
  "`bench.py --renders 512` (after the same command had exited 0 without ncu).  Stage shares under ncu:\n")
nt = load("ncu_traffic.json")
w("| stage | ncu share | ncu ms | bench share (N = 1, 4096 renders) | DRAM MB per render |\n|---|---|---|---|---|")
tot = sum(v["ms"] for v in d["stages"].values())
for k in d["stages"]:
    w("| %s | %.3f | %.3f | %.3f | %.2f |" % (k, nt["ncu_share"][k], nt["ncu_ms"][k], d["stages"][k]["ms"] / tot, nt["dram_bytes_per_render"][k] / 1e6))
w("\n(`ncu_traffic.json` holds the per-stage DRAM bytes per render that `bench.py` scales into `roofline.traffic`.)\n")
w("## 3. `ncu --set full` of the kernels that carry the step, final build (`r02_ncu_key_metrics.md`, `r02_ncu_full_details.csv`)\n")
w(open(os.path.join(P, "r02_ncu_key_metrics.md")).read())
w("Reading (this is what drove the second half of round 2):\n")
w("* **The FFT-type kernels are bound by the L1 / shared-memory data pipe** (`l1tex__data_pipe_lsu_wavefronts`): 87-93 % of its peak in FirP1K / FirP3K / PostMaxK, "
  "70-77 % in ColsWarpK / FirP2K.  DRAM is at 5-54 %, the FP64 pipe at 4-23 %, issue slots at 33-52 %.  Shared-memory traffic is only about half of those wavefronts: "
  "the other half are GLOBAL accesses, which this pipe moves at half the width of a shared-memory access -- and a table lookup at a per-lane address costs up to 32 sectors a request.")
w("* Before that reading (capture `r2x`, same kernels): ColsWarpK 90 % of the pipe, FirP1K 91 %, FirP3K 93 %.  Cutting table lookups -- twiddle powers by squaring instead of "
  "three loads, column twiddles stepped from one `sincospi` instead of two scattered loads per element -- took FirP1K 1.73 -> 1.49 ms, FirP2K 5.02 -> 4.12, FirP3K 1.88 -> 1.61, "
  "ColsWarpK 1.22 -> 0.95 (C5 sweep, N = 1) without touching the arithmetic.")
w("* ColsWarp512K (16 values per lane, 128 registers, two CTAs per SM) sits at 24 % occupancy and ~50 % of the pipe: latency-bound, still 27 % faster than the block-wide tile it replaced.")
w("* OlaK waits on its chain of dependent global loads (long scoreboard 18.6 warps per issue at 64 registers / 44 % occupancy in this capture); "
  "capping it at 32 registers afterwards (eight CTAs per SM) took it 1.54 -> 1.27 ms, and the same cap took SynthTiltK 0.59 -> 0.39, SynthDustK 0.76 -> 0.54 and "
  "SpecOpK 1.98 -> 1.62 ms (the table above predates that change for these four kernels; `r02_bench_n1.json` has their final times).  PostWriteK is the one kernel near DRAM (66 %).")
w("* synth_normal_cluster_kernel: barrier stalls lead (4 cluster barriers per round) -- the price of spreading an event over four CTAs; it still cuts the small-batch synthesis from 0.59 to 0.40 ms.\n")
w("## 4. SASS (`sass_r02_census.md`)\n")
w("Opcode census + excerpts of the shipped library: `UCGABAR_ARV / UCGABAR_WAIT` + the `UPRMT` / `SR_SWINHI` / `LD.E` sequence of distributed-shared-memory loads in the cluster "
  "synthesis kernel (default path for small batches), `WARPSYNC` instead of `BAR` inside the warp-local transforms, `SHFL` scans / reductions, no `ATOM` in the scatter kernels, no `UTMA*` / `*MMA`.\n")
w("## 5. compute-sanitizer\n")
w("`r02_compute_sanitizer_closed.log`: the pool refuses compute-sanitizer (exit 86).  The race check is the schedule-shuffling block emulator "
  "(`tests/test_emul_kernels.py::test_results_do_not_depend_on_the_thread_schedule`) plus bitwise repeatability and the bit-identity of the cluster synthesis kernel against the one-CTA form on the GPU.\n")
w("## 6. Round-1 artefacts kept for the record\n")
w("`bench_r01*`, `launches_r01*`, `ncu_full_r01i_key_kernels.csv`, `ncu_full_raw_r01c_512renders.csv`, `small_configs_r01j.json`: see git history of this file for their description.")
open(os.path.join(P, "README.md"), "w").write(o.getvalue())
print(o.getvalue()[:3000])
