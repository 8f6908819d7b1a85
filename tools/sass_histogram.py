"""Instruction histogram of the shipped library:  python tools/sass_histogram.py [out.json]

Runs `cuobjdump -sass` on latent-space-normalizing-flow_b200/_lib/liblsnf_b200.so and counts, per kernel, the SASS
mnemonics that prove which hardware paths a kernel uses (B200_PROFILING.md): UTCHMMA (tcgen05.mma), UTCHMMA.2CTA
(cta_group::2), LDTM / STTM (tcgen05.ld / st: TMEM), UTMALDG / UTMASTG (TMA tensor loads / stores), UBLKCP (bulk
copies), SYNCS (mbarrier), ACQBULK / PREEXIT (griddepcontrol.wait / launch_dependents: programmatic dependent
launch), plus the classic HMMA / FFMA counts for contrast."""
import collections
import json
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "latent-space-normalizing-flow_b200", "_lib", "liblsnf_b200.so")
WATCH = ["UTCHMMA", "UTCHMMA.2CTA", "UTCQMMA", "UTCQMMA.2CTA", "UTCBAR", "LDTM", "STTM", "UTMALDG", "UTMASTG", "UTMAPF", "UBLKCP", "SYNCS", "ELECT",
         "ACQBULK", "PREEXIT", "HMMA", "FFMA", "MUFU", "BAR.SYNC", "LDG", "STG", "LDS", "STS", "RED", "ATOM"]


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r2_sass_histogram.json")
    txt = subprocess.run(["cuobjdump", "-sass", LIB], capture_output=True, text=True, check=True).stdout
    kernels, cur = collections.OrderedDict(), None
    for line in txt.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            name = subprocess.run(["c++filt", m.group(1)], capture_output=True, text=True).stdout.strip() or m.group(1)
            name = re.sub(r"\(.*", "", name).replace("void ", "").replace("lsnf::", "")
            cur = kernels.setdefault(name, collections.Counter())
            continue
        m = re.match(r"\s+/\*[0-9a-f]+\*/\s+(?:@!?U?P\d+\s+)?([A-Z][A-Z0-9_.]*)", line)
        if m and cur is not None:
            op = m.group(1)
            cur["instructions"] += 1
            for w in WATCH:
                if op == w or op.startswith(w + "."):
                    cur[w] += 1
    res = {k: {w: v[w] for w in ["instructions"] + WATCH if v[w]} for k, v in kernels.items()}
    total = collections.Counter()
    for v in res.values():
        total.update(v)
    json.dump({"library": os.path.relpath(LIB, ROOT), "arch": "sm_100a", "total": dict(total), "kernels": res},
              open(out, "w"), indent=1)
    for k, v in res.items():
        if any(w in v for w in ("UTCHMMA", "LDTM", "UTMALDG", "UTMASTG", "UBLKCP")):
            print(k, {w: c for w, c in v.items() if w in ("instructions", "UTCHMMA", "UTCHMMA.2CTA", "LDTM", "UTMALDG", "UTMASTG", "UBLKCP")})
    print("total", {w: total[w] for w in ("UTCHMMA", "UTCHMMA.2CTA", "LDTM", "UTMALDG", "UTMASTG", "UBLKCP")})


if __name__ == "__main__":
    main()
