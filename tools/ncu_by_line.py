#!/usr/bin/env python
"""Joins an `ncu --page source --csv` SASS dump with `nvdisasm -g` line info and prints the hottest source lines.
usage: tools/ncu_by_line.py <src.csv> <nvdisasm.txt> <mangled-name-substring> [top]"""
import collections
import csv
import re
import sys

ROOT = __import__("os").path.dirname(__import__("os").path.dirname(__import__("os").path.abspath(__file__)))


def main():
    srccsv, dis, key = sys.argv[1:4]
    top = int(sys.argv[4]) if len(sys.argv) > 4 else 40
    txt = open(dis).read().split("\n")
    start = [i for i, l in enumerate(txt) if l.startswith(".text.") and key in l][0]
    end = [i for i, l in enumerate(txt) if i > start and l.startswith("//---------------------")]
    end = end[0] if end else len(txt)
    cur, seq = None, []
    for l in txt[start:end]:
        m = re.search(r'//## File "([^"]+)", line (\d+)', l)
        if m:
            cur = (m.group(1).split("/")[-1], int(m.group(2)))
            continue
        m = re.match(r"\s+/\*([0-9a-f]{4,})\*/\s+(.*?);", l)
        if m:
            seq.append((int(m.group(1), 16), cur, m.group(2)))
    rows = list(csv.reader(open(srccsv)))
    h = [i for i, r in enumerate(rows) if r and r[0] == "Address"][0]
    hdr = rows[h]
    ii, ti, si = hdr.index("Instructions Executed"), hdr.index("Thread Instructions Executed"), hdr.index("# Samples")
    prof = [(r[1], int(r[ii]), int(r[ti]), int(r[si])) for r in rows[h + 1:] if len(r) > ti and r[ii].isdigit()]
    if len(prof) != len(seq):
        print("warning: %d profiled instructions vs %d disassembled" % (len(prof), len(seq)))
    byline = collections.defaultdict(lambda: [0, 0, 0])
    for (off, loc, ins), (src, ie, te, sm) in zip(seq, prof):
        byline[loc][0] += ie
        byline[loc][1] += te
        byline[loc][2] += sm
    tot = sum(v[0] for v in byline.values())
    tots = sum(v[2] for v in byline.values())
    src = {}
    for f in ("trace.cuh", "kernels_trace.cu", "shade.cuh", "kernels_shade.cu"):
        try:
            src[f] = open(ROOT + "/tweeker_raytracer_b200/csrc/" + f).read().split("\n")
        except OSError:
            pass
    try:
        src["rt_portable_math.h"] = open(ROOT + "/include/rt_portable_math.h").read().split("\n")
    except OSError:
        pass
    print("total warp instructions %d, thread instructions %d, samples %d" % (tot, sum(v[1] for v in byline.values()), tots))
    for loc, v in sorted(byline.items(), key=lambda x: -x[1][0])[:top]:
        f, l = loc if loc else ("?", 0)
        line = src[f][l - 1].strip()[:100] if f in src and 0 < l <= len(src[f]) else ""
        print("%5.1f%% inst %5.1f%% smp thr/inst %4.1f  %s:%d  %s" % (100 * v[0] / tot, 100 * v[2] / max(tots, 1), v[1] / max(v[0], 1), f, l, line))


if __name__ == "__main__":
    main()
