"""Per-kernel SASS evidence of the Blackwell paths: counts of the mnemonics that prove tcgen05 / TMEM / TMA use
(UTCHMMA = tcgen05.mma, LDTM / STTM = tcgen05.ld / st, UTMALDG / UTMASTG = TMA load / store, UTCBAR = tcgen05.commit,
SYNCS = mbarrier) next to the legacy tensor-core (HMMA) and special-function (MUFU) counts, from
    cuobjdump -sass wavjepa_b200/libwavjepa_b200.so
    python scripts/sass_summary.py [library] > profiles/r02_sass_summary.txt     (default: the in-tree library)"""
import collections
import os
import re
import subprocess
import sys

LIB = sys.argv[1] if len(sys.argv) > 1 else \
    os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "wavjepa_b200", "libwavjepa_b200.so")
KEYS = ["UTCHMMA", "UTCHMMA.2CTA", "LDTM", "STTM", "UTMALDG", "UTMASTG", "UTCBAR", "SYNCS", "HMMA", "MUFU", "HFMA2", "total"]
out = subprocess.run(["cuobjdump", "-sass", LIB], capture_output=True, text=True).stdout
kern, counts = None, collections.OrderedDict()
for line in out.splitlines():
    m = re.match(r"\s*Function : (\S+)", line)
    if m:
        kern = subprocess.run(["c++filt", m.group(1)], capture_output=True, text=True).stdout.strip()
        kern = re.sub(r"\(CUtensorMap_st.*|\(wj::.*|\(.*", "", kern).replace("void ", "").replace("wj::", "")
        counts[kern] = collections.Counter()
        continue
    m = re.match(r"\s*/\*[0-9a-f]{4}\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_.]+)", line)
    if m and kern:
        op = m.group(1)
        c = counts[kern]
        c["total"] += 1
        base = op.split(".")[0]
        if base in ("UTCHMMA", "LDTM", "STTM", "UTMALDG", "UTMASTG", "UTCBAR", "SYNCS", "HMMA", "MUFU", "HFMA2"):
            c[base] += 1
        if op.startswith("UTCHMMA") and ".2CTA" in op:
            c["UTCHMMA.2CTA"] += 1
print(f"{'kernel':64s} " + " ".join(f"{k:>12s}" for k in KEYS))
tot = collections.Counter()
for k, c in counts.items():
    print(f"{k[:64]:64s} " + " ".join(f"{c[x]:12d}" for x in KEYS))
    tot.update(c)
print(f"{'ALL KERNELS (' + str(len(counts)) + ')':64s} " + " ".join(f"{tot[x]:12d}" for x in KEYS))
