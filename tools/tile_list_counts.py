"""Candidates per 8x4 tile of a pinhole launch, from the host build of the tile lists (csrc/primary_lists.cuh through
tests/native/primary_lists_host.cpp): the histogram, and for list capacities K the share of tiles (= of primary rays) whose list
fits and the traversal work those rays would otherwise do.  Runs on the CPU.

  python tools/tile_list_counts.py [scene] [resolution]      (default: rtigo3_geometry "1920 1080", the benchmark's camera)"""
import os
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import tile_lists as T  # noqa: E402  (the loader of the host build, shared with tests/test_cpu_primary_lists.py)


def main():
    name = sys.argv[1] if len(sys.argv) > 1 else "rtigo3_geometry"
    res = sys.argv[2] if len(sys.argv) > 2 else "1920 1080"
    w, h = (int(v) for v in res.split())
    with tempfile.TemporaryDirectory() as tmp:
        app, export = T.load(tmp, name, res)
        got, want, counts, work = T.primary(app, export, w, h, k=4096)       # room for every tile's whole list
        app.close()
    assert (got == want).all()
    c = counts.astype(np.int64)
    edges = [0, 1, 2, 3, 4, 6, 8, 12, 16, 24, 32, 48, 64, 128, 256, 1 << 30]
    hist, _ = np.histogram(c, bins=edges)
    print("%s %s: %d tiles, mean %.2f candidates, median %d" % (name, res, len(c), c.mean(), int(np.median(c))))
    print("candidates  tiles")
    for i, n in enumerate(hist):
        print("%5d-%-5s %6d" % (edges[i], "" if edges[i + 1] > 4096 else str(edges[i + 1] - 1), n))
    total = work.sum(axis=0).astype(np.float64)
    print("all rays: traversal nodes %.2f, triangles %.2f, instance entries %.2f per ray" % tuple(total / (32.0 * len(c))))
    for k in (16, 24, 32, 48):
        sel = c <= k
        sub = work[sel].sum(axis=0).astype(np.float64)
        print("K=%2d: %.1f %% of tiles and rays listed, mean list %.2f; their traversal work: %.1f %% of nodes, %.1f %% of triangles, "
              "%.1f %% of instance entries" % (k, 100.0 * sel.mean(), c[sel].mean(), 100 * sub[0] / total[0], 100 * sub[1] / total[1], 100 * sub[2] / total[2]))


if __name__ == "__main__":
    main()
