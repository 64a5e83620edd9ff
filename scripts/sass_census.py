"""Opcode census + excerpts of the shipped library's SASS (float64 build): writes profiles/sass_r02_census.md.
usage: python scripts/sass_census.py   (needs cuobjdump on PATH)"""
import collections
import os
import re
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "audio_suite_b200", "csrc", "libmicrosound_b200.so")
sass = subprocess.run(["cuobjdump", "-sass", LIB], capture_output=True, text=True).stdout
demangle = lambda s: subprocess.run(["c++filt", s], capture_output=True, text=True).stdout.strip()
funcs, cur = collections.OrderedDict(), None
for line in sass.splitlines():
    m = re.search(r"Function : (\S+)", line)
    if m:
        cur = funcs.setdefault(m.group(1), [])
        continue
    m = re.match(r"\s+/\*([0-9a-f]+)\*/\s+(.*?);", line)
    if m and cur is not None:
        cur.append((m.group(1), m.group(2).strip()))
KEEP = ("ColsWarpK<0", "ColsWarpK<2", "ColsWarp512K<0", "ColsWarp512K<2", "ColsWarpPlainK<0", "ColsWarpPlainK<2", "SpecOpK", "RowsK<0, 0, 2>",
        "RowsK<0, 0, 4>", "FirP1K", "FirP2K", "FirP3K", "FirSortK", "OlaK", "PostMaxK", "PostWriteK", "SynthNormalK", "SynthDustK",
        "synth_normal_cluster_kernel<4>", "PartialLockK", "ErScatterK", "DecimateK")
COLS = [("inst", None), ("FP64", r"^(@!?U?P\d+ )?D(FMA|ADD|MUL|SETP|MNMX)"), ("LDS", r"\bLDS"), ("STS", r"\bSTS"), ("LDG", r"\bLDG"), ("STG", r"\bSTG"),
        ("BAR", r"\bBAR\."), ("WARPSYNC", r"\bWARPSYNC"), ("SHFL", r"\bSHFL"), ("CGABAR", r"UCGABAR"), ("DSMEM (UPRMT / SR_SWINHI)", r"UPRMT|SR_SWINHI"),
        ("LDL", r"\bLDL"), ("STL", r"\bSTL"), ("ATOM", r"\bATOM|\bRED\."), ("UTMA / UBLKCP", r"UTMA|UBLKCP"), ("MMA", r"MMA")]
rows = []
names = {}
for f, ins in funcs.items():
    d = demangle(f)
    if "msd::" not in d:
        continue
    short = d.replace("void ms_kernel<", "").replace("msd::", "")
    short = re.sub(r"^void ", "", short).split("(")[0]
    short = short.split(", const")[0].split(", ms_")[0].split(", msd")[0].split(", double")[0]
    hit = [k for k in KEEP if k in short]
    if not hit or short in names:
        continue
    names[short] = f
    rows.append((short, [len(ins) if pat is None else sum(1 for _, t in ins if re.search(pat, t)) for _, pat in COLS]))
out = ["# SASS census of the shipped libmicrosound_b200.so (round 2, final build)\n",
       "`cuobjdump -sass audio_suite_b200/csrc/libmicrosound_b200.so`, float64 build (`msd::`), static opcode counts per kernel; regenerate with",
       "`python scripts/sass_census.py`.  What to look for: `WARPSYNC` instead of `BAR` inside the warp-local FFT phases (ColsWarpK, ColsWarp512K,",
       "ColsWarpPlainK, FirP1K/P2K/P3K); the hardware cluster barrier `UCGABAR_ARV` / `UCGABAR_WAIT` and the distributed-shared-memory accesses",
       "(PTX `mapa` + `ld.shared::cluster` become `UPRMT` of the CTA rank into the shared-window address, `S2UR SR_SWINHI` and a generic `LD.E`) in",
       "`synth_normal_cluster_kernel` -- the cluster form of the synthesis kernel that the DEFAULT path launches for small",
       "batches; `SHFL` in the reductions / scans; no `ATOM` / `RED` in ErScatterK and",
       "PartialLockK (deterministic gather forms; PostMaxK keeps one order-independent atomicMax per CTA); `LDL` / `STL` = register spills (FirP2K).",
       "There is no `UTMA*` / `UBLKCP`: tiles are staged through registers with all loads of a tile in flight before the first dependent store",
       "(DESIGN.md section 4) -- the two ends of the FIR pipeline read / write real samples at 8-byte granularity, which the 16-byte alignment",
       "rule of the bulk-async copies excludes, and the scratch side was not worth a second mechanism; and no `*MMA`: nothing here is a dense",
       "contraction.\n",
       "| kernel | " + " | ".join(c for c, _ in COLS) + " |", "|---|" + "---|" * len(COLS)]
for short, vals in sorted(rows):
    out.append("| %s | %s |" % (short, " | ".join(str(v) for v in vals)))


def excerpt(title, key, pats, n=6):
    f = next((names[s] for s in names if key in s), None)
    if f is None:
        return
    out.append("\n### %s\n`%s`\n```" % (title, demangle(f)[:110]))
    k = 0
    for addr, t in funcs[f]:
        if any(re.search(p, t) for p in pats):
            out.append("    /*%s*/  %s ;" % (addr, t))
            k += 1
            if k >= n:
                break
    out.append("```")


out.append("\n## Excerpts")
excerpt("cluster barrier + distributed shared memory -- synth_normal_cluster_kernel<4> (default path for small batches)", "synth_normal_cluster_kernel<4>",
        [r"UCGABAR", r"UPRMT", r"SR_SWINHI", r"LD\.E R\d+, \[RZ\.U32\+UR"], 12)
excerpt("warp-level barriers inside the transforms -- ColsWarp512K (two 512-point FFTs chained through registers)", "ColsWarp512K<2", [r"WARPSYNC", r"BAR\."], 8)
excerpt("warp-level barriers inside the FFT phases -- FirP2K", "FirP2K", [r"WARPSYNC", r"BAR\."], 8)
excerpt("block maximum by warp shuffles -- PostMaxK", "PostMaxK", [r"SHFL"], 5)
excerpt("prefix scan by warp shuffles -- SynthNormalK", "SynthNormalK", [r"SHFL"], 5)
open(os.path.join(ROOT, "profiles", "sass_r02_census.md"), "w").write("\n".join(out) + "\n")
print("\n".join(out[:40]))
