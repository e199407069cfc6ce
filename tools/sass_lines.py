#!/usr/bin/env python3
"""Executed warp instructions and stall samples per CUDA source line of one kernel.
Joins `ncu -i X.ncu-rep --page source --csv --kernel-name ... --launch-count 1` (SASS rows, in address order) with
`nvdisasm --print-line-info` of the matching cubin (same build), instruction by instruction.
usage: tools/sass_lines.py source_page.csv cubin mangled_name_fragment [top]"""
import collections
import csv
import os
import re
import subprocess
import sys


def main():
    page, cubin, frag = sys.argv[1:4]
    top = int(sys.argv[4]) if len(sys.argv) > 4 else 40
    dis = subprocess.run(["nvdisasm", "--print-line-info", cubin], capture_output=True, text=True).stdout.splitlines()
    lines, cur, infun = [], None, False
    for s in dis:
        m = re.match(r"\s*\.text\.(\S+):", s)
        if m:
            infun = frag in m.group(1)
            continue
        if s.startswith("\t.section") or s.strip().startswith(".section"):
            infun = False
        if not infun:
            continue
        m = re.search(r'//## File "([^"]+)", line (\d+)', s)
        if m:
            cur = int(m.group(2))
            continue
        if re.match(r"\s*/\*[0-9a-f]{4,}\*/\s+\S", s):
            lines.append(cur)
    rows = list(csv.reader(open(page)))
    hdr = None
    ex, st = [], []
    for r in rows:
        if "Instructions Executed" in r:
            hdr = r
            ie, iss = hdr.index("Instructions Executed"), hdr.index("Warp Stall Sampling (All Samples)")
            continue
        if hdr is None or len(r) <= ie or not r[ie].isdigit():
            continue
        ex.append(int(r[ie]))
        st.append(int(r[iss]) if r[iss].isdigit() else 0)
    print("sass instructions: nvdisasm %d, ncu %d" % (len(lines), len(ex)))
    n = min(len(lines), len(ex))
    per, pst = collections.Counter(), collections.Counter()
    for i in range(n):
        per[lines[i]] += ex[i]
        pst[lines[i]] += st[i]
    tot, tst = sum(per.values()) or 1, sum(pst.values()) or 1
    src = open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "peleanalysis_b200", "csrc", "stencil_tma.cu")).read().splitlines()
    for ln, c in per.most_common(top):
        text = src[ln - 1].strip()[:110] if ln and ln <= len(src) else "?"
        print("%5s %6.2f%% inst %6.2f%% stall | %s" % (ln, 100.0 * c / tot, 100.0 * pst[ln] / tst, text))


if __name__ == "__main__":
    main()
