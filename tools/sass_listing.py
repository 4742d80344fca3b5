#!/usr/bin/env python3
"""SASS listing of the hot kernels for profiles/ (north star: "a committed SASS listing").

    python tools/sass_listing.py profiles/r1_sass

writes <prefix>_<kernel>.txt (instructions only, encodings stripped) for the instantiations the BASELINE configs
run -- 150 bp, one read group or a segmented batch: build_smem_kernel<3,true>, apply_smem_kernel<4,true>; 250 bp:
build<2,true>, apply<3,true>; the work-list walk of rows in read order with several read groups: build<1,true>,
apply<2,true>; build<4,true> is the plan round 1 ran at 150 bp -- plus <prefix>_summary.txt with a mnemonic histogram of each: the lines to
look for are UBLKCP (TMA bulk copy), SYNCS (mbarrier), ATOMS / REDS (shared-memory reductions), IDP
(4-way byte dot product), PRMT, LDS, STG.
"""
import collections
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SO = os.path.join(ROOT, "kbbq-py_b200", "kbbq", "libkbbq_b200.so")
WANT = {
    "_ZN4kbbq17build_smem_kernelILi3ELb1EEEvNS_9BuildArgsE": "build_smem_kernel_kps3",
    "_ZN4kbbq17build_smem_kernelILi4ELb1EEEvNS_9BuildArgsE": "build_smem_kernel_kps4",
    "_ZN4kbbq17apply_smem_kernelILi4ELb1EEEvNS_9ApplyArgsE": "apply_smem_kernel_kps4",
    "_ZN4kbbq17build_smem_kernelILi2ELb1EEEvNS_9BuildArgsE": "build_smem_kernel_kps2",
    "_ZN4kbbq17apply_smem_kernelILi3ELb1EEEvNS_9ApplyArgsE": "apply_smem_kernel_kps3",
    "_ZN4kbbq17build_smem_kernelILi1ELb1EEEvNS_9BuildArgsE": "build_smem_kernel_kps1",
    "_ZN4kbbq17apply_smem_kernelILi2ELb1EEEvNS_9ApplyArgsE": "apply_smem_kernel_kps2",
}


def main():
    prefix = sys.argv[1]
    txt = subprocess.run(["cuobjdump", "-sass", SO], capture_output=True, text=True, check=True).stdout
    cur, body = None, collections.defaultdict(list)
    for line in txt.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            cur = m.group(1)
            continue
        m = re.match(r"\s+/\*([0-9a-f]{4,})\*/\s+(.*?)\s*;?\s*/\* 0x[0-9a-f]+ \*/", line)
        if cur and m:
            body[cur].append("/*%s*/ %s" % (m.group(1), m.group(2).rstrip(" ;")))
    with open(prefix + "_summary.txt", "w") as summ:
        summ.write("SASS mnemonic histogram (cuobjdump -sass %s, sm_100a)\n" % os.path.relpath(SO, ROOT))
        for sym, name in WANT.items():
            ins = body.get(sym)
            if not ins:
                raise SystemExit("kernel not found: " + sym)
            with open("%s_%s.txt" % (prefix, name), "w") as fh:
                fh.write("// %s\n" % sym)
                fh.write("\n".join(ins) + "\n")
            hist = collections.Counter()
            for i in ins:
                op = re.sub(r"^/\*\w+\*/\s+(@!?U?P\d+\s+)?", "", i).split()[0]
                hist[op.split(".")[0] + ("." + op.split(".")[1] if op.startswith(("IDP", "UBLKCP", "SYNCS", "ATOMS", "REDS", "LDS", "STG", "LDG")) and "." in op else "")] += 1
            summ.write("\n%s  (%d instructions)\n" % (name, len(ins)))
            for op, n in hist.most_common():
                summ.write("  %-22s %5d\n" % (op, n))


if __name__ == "__main__":
    main()
