"""Turns an ncu launch list (csv: gpu__time_duration.sum, dram__bytes_read.sum, dram__bytes_write.sum, ... per launch of ONE
bench.py step) into a markdown table and profiles/ncu_traffic.json (DRAM bytes per render and per pipeline stage, which
bench.py reports as roofline.traffic).  usage: ncu_summarise.py launches.csv RENDERS [out.json]"""
import collections
import csv
import json
import sys

UNIT = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "ns": 1e-6, "us": 1e-3, "ms": 1.0, "s": 1e3}


def load(path):
    rows = [r for r in csv.reader(open(path)) if len(r) > 10 and r[0].isdigit()]
    launches = collections.OrderedDict()
    for r in rows:
        d = launches.setdefault(r[0], {"name": r[4], "grid": r[8], "block": r[7]})
        d[r[-3]] = float(r[-1].replace(",", "")) * UNIT.get(r[-2], 1.0)
    return list(launches.values())


def stage_of(launches):
    """Pipeline stage of every launch, from the fixed order of BatchRenderer.run()."""
    out, stage = [], "synth"
    seen_tilt_finish = any("SynthTiltK" in l["name"] for l in launches)
    fft_before_tilt = seen_tilt_finish
    for l in launches:
        n = l["name"]
        if "SynthNormalK" in n or "SynthDustK" in n or "synth_normal_cluster_kernel" in n:
            stage = "synth"
        elif "SynthTiltK" in n:
            out.append("tilt_spectral")
            fft_before_tilt = False
            continue
        elif "AdsrTableK" in n or "OlaK" in n:
            stage = "overlap_add"
        elif "ErScatterK" in n or "FirP1K" in n or "FirP2K" in n or "FirP3K" in n:
            stage = "fir_overlap_save"
        elif "PostMaxK" in n or "PostWriteK" in n or "RollK" in n:
            stage = "post"
        elif "ColsK" in n or "RowsK" in n or "ColsWarpK" in n or "SpecOpK" in n:
            if stage == "synth":
                stage = "tilt_spectral" if fft_before_tilt else "grain_spectral"
            elif stage == "tilt_spectral" and not fft_before_tilt:
                stage = "grain_spectral"
        out.append(stage)
    return out


def main():
    path, renders = sys.argv[1], int(sys.argv[2])
    L = load(path)
    st = stage_of(L)
    tot = sum(l["gpu__time_duration.sum"] for l in L)
    print("| # | kernel | stage | grid | ms | share | DRAM read MB | DRAM write MB | GB/s |")
    print("|---|---|---|---|---|---|---|---|---|")
    per_stage = collections.OrderedDict()
    for i, (l, s) in enumerate(zip(L, st)):
        t = l["gpu__time_duration.sum"]
        rd, wr = l.get("dram__bytes_read.sum", 0.0), l.get("dram__bytes_write.sum", 0.0)
        name = l["name"].replace("void ms_kernel<", "").split(", const")[0].replace("msd::", "").replace("msf::", "")
        if name.startswith("void "):                         # kernels launched outside ms_launch (cluster kernels)
            name = name[5:].split("(")[0]
        print("| %d | %s | %s | %s | %.3f | %.1f%% | %.1f | %.1f | %.0f |" % (i, name, s, l["grid"], t, 100 * t / tot, rd / 1e6, wr / 1e6,
                                                                       (rd + wr) / 1e9 / (t * 1e-3) if t else 0))
        d = per_stage.setdefault(s, {"ms": 0.0, "dram_bytes": 0.0, "launches": 0})
        d["ms"] += t
        d["dram_bytes"] += rd + wr
        d["launches"] += 1
    print("\ntotal %.3f ms under ncu for %d renders" % (tot, renders))
    out = {"renders_profiled": renders, "source": path.split("/")[-1],
           "dram_bytes_per_render": {s: d["dram_bytes"] / renders for s, d in per_stage.items()},
           "ncu_ms": {s: round(d["ms"], 4) for s, d in per_stage.items()},
           "ncu_share": {s: round(d["ms"] / tot, 4) for s, d in per_stage.items()}}
    if len(sys.argv) > 3:
        json.dump(out, open(sys.argv[3], "w"), indent=1)
    print(json.dumps(out["ncu_share"]))


if __name__ == "__main__":
    main()
