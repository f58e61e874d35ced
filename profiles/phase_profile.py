#!/usr/bin/env python
"""Attribute ncu per-SASS counters to kernel phases by source line ranges.

Usage: phase_profile.py <ncu source csv> <nvdisasm --print-line-info listing> <mangled kernel>
Phases are delimited by marker comments in rt_kernels.cu; inlined helpers (the fp64 primitives,
sqrt_rsqrt, div_seeded, layer_pair_ffp, div_unchecked) are reported by helper name."""
import csv, re, sys, collections
src_csv, listing, kern = sys.argv[1:4]
cu = open("/root/repo/raytracerfortran_b200/csrc/rt_kernels.cu").read().splitlines()
def find(pat, start=0):
    for i in range(start, len(cu)):
        if pat in cu[i]: return i + 1
    raise SystemExit(f"marker not found: {pat}")
kstart = find("rt_batch_kernel(const BatchArgs a")
v1 = find("constexpr bool kDeep = (VARIANT == 3);", kstart)
marks = [("kernel prologue", kstart), ("A stage+tables", find("// ---------------- A:", kstart)),
         ("B per-ray setup", find("// ---------------- B:", kstart)), ("sort", find("// ---------------- counting sort", kstart)),
         ("C setup", find("// ---------------- C: solve", kstart)),
         ("C refill", find("// ---- refill idle lanes", v1)),
         ("C eval loop ctl", find("// ---- f and f' at x", v1)), ("C transition", find("// ---- advance the ray", v1)),
         ("C' travel times", find("// ---- travel times at the final p", v1)), ("D outputs", find("// ---------------- D:", v1)),
         ("end", find("// \"next\" row N1: INTERPLAYER_novar", v1))]
helpers = [("fp64 prims (dmul..dsqrt builtins)", find("double dmul(double a"), find("double dsqrt(double a") + 1),
           ("sqrt_rsqrt", find("double sqrt_rsqrt("), find("double div_seeded(")),
           ("div_seeded", find("double div_seeded("), find("// a / b by exactly")),
           ("div_unchecked", find("// a / b by exactly"), find("// 32-bit shared-memory addressing")),
           ("lds/sts helpers", find("// 32-bit shared-memory addressing"), find("// One solver pass evaluates")),
           ("layer_pair_ffp", find("// One solver pass evaluates"), find("// variant 1: the solver"))]
def phase_of(ln):
    if ln is None: return "?"
    for name, a, b in helpers:
        if a <= ln < b: return name
    if ln < kstart: return "other helpers"
    for (name, a), (_, b) in zip(marks, marks[1:]):
        if a <= ln < b: return name
    return "?"
lines = open(listing).read().splitlines()
start = next(i for i, l in enumerate(lines) if l.startswith(f".text.{kern}:"))
cur = None; seq = []
for l in lines[start + 1:]:
    if l.startswith("//---"): break
    m = re.search(r'//## File "([^"]+)", line (\d+)', l)
    if m: cur = int(m.group(2)); continue
    m = re.match(r"\s*/\*([0-9a-f]{4,})\*/\s+(.*?);", l)
    if m: seq.append((cur, m.group(2)))
rows = list(csv.reader(open(src_csv))); hdr = rows[1]; idx = {h: i for i, h in enumerate(hdr)}
recs = [r for r in rows[2:] if len(r) >= len(hdr)]
assert len(recs) == len(seq), (len(recs), len(seq))
fp64 = ("DFMA", "DMUL", "DADD", "DSETP")
agg = collections.OrderedDict()
tot = totf = 0
for (ln, sass), r in zip(seq, recs):
    inst = int(r[idx["Instructions Executed"]] or 0); thr = int(r[idx["Predicated-On Thread Instructions Executed"]] or 0)
    op = (sass.split()[1] if sass.startswith("@") else sass.split()[0]).split(".")[0]
    a = agg.setdefault(phase_of(ln), [0, 0, 0, 0])
    a[0] += inst; a[1] += thr; a[2] += int(r[idx["# Samples"]] or 0)
    if op in fp64: a[3] += inst; totf += inst
    tot += inst
slots = tot + totf
print(f"total warp-inst {tot:.3e}  fp64 {totf:.3e}  issue slots (2*fp64+other) {slots:.3e}")
print(f"{'phase':36s} {'warp-inst':>10s} {'share':>6s} {'fp64':>6s} {'lane':>5s} {'slots%':>7s} {'samples':>8s}")
for name, (i, t, s, f) in sorted(agg.items(), key=lambda kv: -kv[1][0]):
    print(f"{name:36s} {i:10.3e} {i/tot:6.3f} {f/max(i,1):6.2f} {t/32/max(i,1):5.2f} {100*(i+f)/slots:7.2f} {s:8d}")
