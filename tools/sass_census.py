#!/usr/bin/env python
"""SASS census of the shipped library (runs in the build container: cuobjdump needs no GPU).
Per kernel: counts of the instructions that prove which hardware paths the code uses --
DMMA (FP64 tensor pipe, mma.sync.m8n8k4.f64), UBLKCP (cp.async.bulk, TMA 1-D), UTMALDG (tensor-map TMA),
SYNCS (mbarrier), BAR (named barriers), USETMAXREG (register re-allocation), LDGSTS (cp.async), UTCMMA / tcgen05
(none expected: tcgen05 has no f64 kind)."""
import collections
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
lib = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "bipymc_b200", "lib", "libbipymc_b200.so")
out = subprocess.run(["cuobjdump", "-sass", lib], stdout=subprocess.PIPE, text=True).stdout
keys = ["DMMA", "UBLKCP", "UTMALDG", "SYNCS", "BAR", "USETMAXREG", "LDGSTS", "UTC", "DFMA", "DADD", "DMUL", "MUFU", "REDUX"]
cur, per, arch = None, collections.OrderedDict(), set()
for line in out.splitlines():
    m = re.search(r"Function : (\S+)", line)
    if m:
        cur = subprocess.run(["c++filt", m.group(1)], stdout=subprocess.PIPE, text=True).stdout.strip()
        cur = re.sub(r"\(.*", "", cur)
        per[cur] = collections.Counter()
        continue
    m = re.search(r"arch = (sm_\w+)", line)
    if m:
        arch.add(m.group(1))
    if cur is None:
        continue
    m = re.search(r"^\s+/\*[0-9a-f]+\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_.]+)", line)
    if m:
        op = m.group(1)
        per[cur]["_total"] += 1
        for k in keys:
            if op.startswith(k):
                per[cur][k] += 1
print("library:", os.path.relpath(lib, ROOT), " arch:", ",".join(sorted(arch)))
print("%-64s %7s " % ("kernel", "instr") + " ".join("%6s" % k for k in keys))
tot = collections.Counter()
for name, c in per.items():
    tot.update(c)
    if any(c[k] for k in keys[:8]) or "fused" in name:
        print("%-64s %7d " % (name[-64:], c["_total"]) + " ".join("%6d" % c[k] for k in keys))
print("%-64s %7d " % ("ALL KERNELS (%d)" % len(per), tot["_total"]) + " ".join("%6d" % tot[k] for k in keys))
