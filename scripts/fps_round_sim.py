"""CPU simulation of the multi-pick round of fps_bucket.cu (DESIGN 4.1): mean picks accepted per round on the benchmark's
clouds, for a given record granularity and cap K.  numpy only, no GPU; nothing here is a timing.

The points are sorted like the kernel sorts them (15 Morton bits handed out greedily to the axis with the largest cell
extent) and cut into `records` equal groups of consecutive sorted points (32 = one record per warp, 64 = one per half of
a warp's chunks).  Every group posts its candidate and a runner-up that leaves out exact duplicates of the candidate; a
round accepts the sorted candidates while (i) no neighbour in the sorted order shares its key with the low
log2(records) bits cleared (the kernel's sort key), (ii) the key is above the runner-up of every group an earlier pick
came from, (iii) no earlier pick lowers it.

    python scripts/fps_round_sim.py --records 64 --K 16 --clouds 0 9
"""
import argparse
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def morton_order(x, bits=15):
    lo, hi = x.min(0), x.max(0)
    e = hi - lo
    nb, c, order = [0, 0, 0], e.copy(), []
    for _ in range(bits):
        ax = 0
        if c[1] > c[0] and c[1] >= c[2]:
            ax = 1
        if c[2] > c[0] and c[2] > c[1]:
            ax = 2
        order.append(ax)
        nb[ax] += 1
        c[ax] *= 0.5
    q = [np.clip(np.floor((x[:, a] - lo[a]) * ((1 << nb[a]) / e[a])).astype(np.int64), 0, (1 << nb[a]) - 1) for a in range(3)]
    r, key = nb[:], np.zeros(len(x), np.int64)
    for ax in order:
        r[ax] -= 1
        key = (key << 1) | ((q[ax] >> r[ax]) & 1)
    return np.argsort(key, kind="stable")


def picks_per_round(x, records, K, m=4096):
    p = morton_order(x)
    xs = x[p].astype(np.float32)
    n = len(xs)
    g = n // records
    shift = int(records - 1).bit_length()  # record-id bits of the sort key
    md = np.full(n, 1e10, np.float32)
    pending, picks, rounds = [int(np.nonzero(p == 0)[0][0])], 1, 0
    while picks < m:
        for c in pending:
            md = np.minimum(md, ((xs - xs[c]) ** 2).sum(1).astype(np.float32))
        rounds += 1
        M = md.reshape(records, g)
        am = M.argmax(1)
        top = M[np.arange(records), am]
        XS = xs.reshape(records, g, 3)
        same = (XS == XS[np.arange(records), am][:, None, :]).all(2)
        run = np.where(same, -1, M).max(1)
        bucket = top.view(np.uint32) >> shift
        o = np.argsort(-top, kind="stable")
        pending, run2, k = [o[0] * g + am[o[0]]], run[o[0]], 1
        while k < records and len(pending) < K and picks + len(pending) < m:
            w = o[k]
            key, q = top[w], w * g + am[w]
            near = bucket[w] == bucket[o[k - 1]] or (k + 1 < records and bucket[w] == bucket[o[k + 1]])
            if near or not key > run2 or any(np.float32(((xs[pp] - xs[q]) ** 2).sum()) < key for pp in pending):
                break
            pending.append(q)
            run2 = max(run2, run[w])
            k += 1
        picks += len(pending)
    return (m - 1) / rounds


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--records", type=int, nargs="+", default=[32, 64])
    ap.add_argument("--K", type=int, nargs="+", default=[8, 16])
    ap.add_argument("--clouds", type=int, nargs="+", default=[0, 9], help="bench.make_inputs(16, 0) clouds (0-7 ground + "
                    "objects, 8-15 duplicate-padded)")
    args = ap.parse_args()
    import bench

    xyz = bench.make_inputs(16, 0)[0]
    for ci in args.clouds:
        for r in args.records:
            for k in args.K:
                print(f"cloud {ci:2d}  records {r:3d}  K {k:2d}  picks/round {picks_per_round(xyz[ci].astype(np.float32), r, k):.2f}",
                      flush=True)


if __name__ == "__main__":
    main()
