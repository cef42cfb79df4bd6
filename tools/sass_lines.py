#!/usr/bin/env python
"""Warp-instructions executed per SOURCE LINE of one kernel: joins the per-SASS-instruction counts of an .ncu-rep
(`ncu --set full --import-source on`, read here without a GPU) with the line table of the built library (nvdisasm -g).
usage: tools/sass_lines.py file.ncu-rep <kernel-substring of the mangled name, e.g. step_call_kernelILi4E> [n_envs] [top]"""
import csv, re, subprocess, sys, tempfile, os
from collections import defaultdict
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
rep, key = sys.argv[1], sys.argv[2]
n_envs = float(sys.argv[3]) if len(sys.argv) > 3 else 1048576.0
top = int(sys.argv[4]) if len(sys.argv) > 4 else 60
lib = ROOT / "3d-navigation-reinforcement-learning_b200" / "lib" / "libnav3d_b200.so"
tmp = tempfile.mkdtemp()
subprocess.run(["cuobjdump", "-xelf", "all", str(lib)], cwd=tmp, capture_output=True)
cubin = next(p for p in Path(tmp).glob("nav3d_engine.sm_100a.cubin"))
sass = subprocess.run(["nvdisasm", "-g", "-c", str(cubin)], capture_output=True, text=True).stdout.splitlines()
# line table of the function: offset -> (file, line)
table, cur, infn = {}, None, False
for ln in sass:
    if ln.startswith(".text.") and ln.rstrip().endswith(":"):
        infn = key in ln and "$" not in ln
        continue
    if not infn:
        continue
    m = re.search(r'//## File "([^"]+)", line (\d+)', ln)
    if m:
        cur = (os.path.basename(m.group(1)), int(m.group(2)))
        continue
    m = re.match(r"\s*/\*([0-9a-f]{4,})\*/\s+(.*);", ln)
    if m:
        table[int(m.group(1), 16)] = (cur, m.group(2).strip())
out = subprocess.run(["ncu", "-i", rep, "--page", "source", "--csv"], capture_output=True, text=True).stdout
rows = list(csv.reader(out.splitlines()))
h = next(i for i, r in enumerate(rows) if "Instructions Executed" in r)
hdr = rows[h]
# NAV3D_COL: sum another per-instruction column of the source page instead (e.g. "L2 Theoretical Sectors Global")
ia, iaddr, isamp = hdr.index(os.environ.get("NAV3D_COL", "Instructions Executed")), hdr.index("Address"), hdr.index("# Samples")
data = [r for r in rows[h + 1:] if len(r) > ia and r[ia].isdigit()]
base = int(data[0][iaddr], 16)
per_line, samples, total, missing = defaultdict(int), defaultdict(int), 0, 0
for r in data:
    off = int(r[iaddr], 16) - base
    n = int(r[ia]); total += n
    ent = table.get(off)
    if ent is None:
        missing += n
        continue
    per_line[ent[0]] += n
    samples[ent[0]] += int(r[isamp]) if r[isamp].isdigit() else 0
print(f"total warp-instructions {total} = {total / n_envs:.1f} per env-step; unmapped {missing / n_envs:.1f}")
srcs = {}
def text(f, l):
    if f not in srcs:
        for cand in (ROOT / "3d-navigation-reinforcement-learning_b200" / "csrc" / f,):
            srcs[f] = cand.read_text().splitlines() if cand.exists() else []
    s = srcs[f]
    return s[l - 1].strip()[:110] if 0 < l <= len(s) else ""
tot_s = sum(samples.values()) or 1
for (f, l), n in sorted(per_line.items(), key=(lambda kv: -samples[kv[0]]) if os.environ.get("NAV3D_SORT") == "samples" else (lambda kv: -kv[1]))[:top]:
    print(f"{n / n_envs:7.2f}  {100 * samples[(f, l)] / tot_s:5.1f}%smp  {f}:{l:<5} {text(f, l)}")
# optional: totals per named line range of nav3d_core.cuh (env NAV3D_RANGES="name:lo-hi,...")
rng = os.environ.get("NAV3D_RANGES")
if rng:
    print("-- by range (warp-instructions per env-step, share of stall samples)")
    for part in rng.split(","):
        name, lh = part.split(":"); lo, hi = (int(v) for v in lh.split("-"))
        n = sum(v for (f, l), v in per_line.items() if f == "nav3d_core.cuh" and lo <= l <= hi)
        sm = sum(v for (f, l), v in samples.items() if f == "nav3d_core.cuh" and lo <= l <= hi)
        print(f"{n / n_envs:7.2f}  {100 * sm / tot_s:5.1f}%smp  {name}")
    n = sum(v for (f, l), v in per_line.items() if f != "nav3d_core.cuh")
    sm = sum(v for (f, l), v in samples.items() if f != "nav3d_core.cuh")
    print(f"{n / n_envs:7.2f}  {100 * sm / tot_s:5.1f}%smp  (other files)")
