#!/usr/bin/env python3
"""Per-kernel totals and the shares of one EM iteration from an ncu launch list
(`ncu --metrics gpu__time_duration.sum --clock-control none --csv --log-file X.csv python bench.py ...`); no GPU.
    python tools/launch_shares.py gpurun_out/X.csv > profiles/X_shares.txt"""
import collections
import csv
import re
import sys

rows = [r for r in csv.reader(l for l in open(sys.argv[1]) if l.startswith('"'))]
hdr, rows = rows[0], rows[1:]
ki, vi, ui = hdr.index("Kernel Name"), hdr.index("Metric Value"), hdr.index("Metric Unit")
tot, cnt = collections.Counter(), collections.Counter()
for r in rows:
    name = re.sub(r"\(.*", "", r[ki])[:64]
    ns = float(r[vi].replace(",", "")) * {"ns": 1.0, "us": 1e3, "ms": 1e6}[r[ui]]
    tot[name] += ns
    cnt[name] += 1
print("per-launch times under ncu are cold-cache and serialised: compare shares, not absolutes\n")
# the headline iteration (round 2): prep, pass A, pass B + C (Kuzmin: the gather-through-L1 instances "..., 1>"), finish, M-step;
# round-1 lists (em_fused / em_finalize / stage_p) still match their own names
seg3 = any("seg3_pass_kernel" in k for k in tot)
if seg3:
    l1 = any("seg3_pass_kernel" in k and k.rstrip().endswith(", 1>") for k in tot)
    step = {k: tot[k] / cnt[k] for k in tot
            if "seg3_prep" in k or "seg3_finish" in k or "normalise" in k
            or ("seg3_pass_kernel" in k and k.rstrip().endswith(", 1>" if l1 else ", 0>"))}
else:
    step = {k: tot[k] / cnt[k] for k in tot
            if "tip::" in k and (("em_fused" in k and "double, 0, 0>" in k) or "em_finalize" in k or "stage_p_kernel<double>" in k
                                 or "normalise" in k)}
s = sum(step.values())
print("one EM iteration (E-step + M-step), mean per launch:")
for k, v in sorted(step.items(), key=lambda kv: -kv[1]):
    print("  %-64s %8.1f us  %5.1f%% of the iteration" % (k, v / 1e3, 100 * v / s))
print("\nall launches of the command:")
g = sum(tot.values())
for k, v in tot.most_common():
    print("  %-64s n=%4d total %10.1f us %5.1f%%" % (k, cnt[k], v / 1e3, 100 * v / g))
