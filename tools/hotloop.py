#!/usr/bin/env python
"""hotloop.py -- instruction mix of a kernel's vector tile loop, from the SASS of an object file (no GPU needed).

    python tools/hotloop.py build/lean/ek_ops_ept.o 'OpEptWbILi0ELi1ELi1E.*IdLi2'

The tile loop is taken as the span between the first LDG.E.EF.128 and the last backward branch after the last STG.E.EF.128
of the kernel; blocks that end in a CALL (the out-of-line exact recompute) are left out.  Counts are per loop iteration
(= kUnroll x VEC points); straight-line code only -- kernels with uniform branches inside the loop over-count.
"""
import collections
import re
import subprocess
import sys


def main():
    obj, pat = sys.argv[1], re.compile(sys.argv[2])
    names = [ln.split()[2] for ln in subprocess.run(["cuobjdump", "-sass", obj], capture_output=True, text=True).stdout.splitlines() if "Function :" in ln]
    for name in names:
        if not pat.search(name):
            continue
        out = subprocess.run(["cuobjdump", "-sass", "-fun", name, obj], capture_output=True, text=True).stdout
        ins = []
        for ln in out.splitlines():
            m = re.match(r"\s+/\*([0-9a-f]{4,5})\*/\s+(?:@!?U?P[0-9T]\s+)?([A-Z0-9_.]+)(.*?);", ln)
            if m:
                ins.append((int(m.group(1), 16), m.group(2), m.group(3)))
        lds = [a for a, o, _ in ins if o.startswith("LDG.E.EF.128")]
        sts = [a for a, o, _ in ins if o.startswith("STG.E.EF.128")]
        if not lds or not sts:
            print(name, "no vector loop found")
            continue
        lo, hi = lds[0], sts[-1]
        # the first vector loop only (kernels hold one per load flavour): it ends at the first backward branch to (or before) its first load
        for a, o, rest in ins:
            m = re.search(r"0x([0-9a-f]+)", rest)
            if a > lo and o == "BRA" and m and int(m.group(1), 16) <= lo and any(lo < x < a for x in sts):
                hi = a
                break
        # cold-call blocks: from the branch that skips them to the CALL's BSYNC: approximate as the 20 instructions before a CALL
        calls = [a for a, o, _ in ins if o.startswith("CALL") and lo <= a <= hi]
        skip = []
        for c in calls:
            # walk back to the guarding forward branch "@!P0 BRA target" whose target lies after the call
            for a, o, rest in reversed([x for x in ins if x[0] < c]):
                m = re.search(r"0x([0-9a-f]+)", rest)
                if o == "BRA" and m and int(m.group(1), 16) > c:
                    skip.append((a + 16, int(m.group(1), 16)))
                    break
        cnt = collections.Counter()
        for a, o, _ in ins:
            if lo <= a <= hi and not any(s <= a < e for s, e in skip):
                cnt[o.split(".")[0]] += 1
        tot = sum(cnt.values())
        fp64 = cnt["DFMA"] + cnt["DMUL"] + cnt["DADD"]
        print(f"{name[:110]}\n  loop span {lo:#x}-{hi:#x}: {tot} instructions per iteration, FP64 {fp64}, calls skipped {len(skip)}")
        print("  " + "  ".join(f"{k}:{v}" for k, v in cnt.most_common(18)))


if __name__ == "__main__":
    main()
