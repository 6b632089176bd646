"""Times find_contribs_from_reads on a config-2-sized read matrix (138 569 x 5408 fp64,
6.0 GB, far larger than the 126 MB L2) on one GPU:

* ``vote_first``: the current path, mxb_matrix_vote_first (row argmax + votes and
  first rows per column; 2H numbers come back);
* ``vote_count_unique``: the path it replaced, mxb_matrix_vote_count with the N-long
  argmax copied back and ordered by numpy.unique on the host.

Each call ends in a stream synchronise inside the library, so a host clock around it
measures the call.  Both paths are warmed up, then timed alternately; the median is
reported with GB/s over the 6.0 GB the argmax reads, next to the card's name and
power limit.  Usage: python scripts/shard_consumers_time.py [--reps 7] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit",
                               "--format=csv,noheader"], capture_output=True, text=True,
                              timeout=30).stdout.strip().splitlines()[0]
    except Exception as exc:       # the numbers are still printed, without the card
        return "unknown (%s)" % exc


def old_path(dev, wts, min_reads):
    from mixemt_b200 import consumers
    votes, best = consumers.vote_count(dev, wts)
    seen, first = np.unique(best, return_index=True)
    order = seen[np.argsort(first, kind="stable")]
    return [int(con) for con in order if votes[con] >= min_reads]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=138569)
    ap.add_argument("--cols", type=int, default=5408)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default=None)
    opt = ap.parse_args()

    from mixemt_b200 import consumers
    from mixemt_b200._lib import lib, check, ptr
    from mixemt_b200.runtime import DeviceMatrix, get_context
    ctx = get_context()
    n, h = opt.rows, opt.cols
    dev = DeviceMatrix.empty(ctx, n, h)
    rs = np.random.RandomState(11)
    block = 4096
    base = -rs.gamma(2.0, 5.0, size=(block, h))
    base[rs.rand(block, h) < 0.2] = 0.0
    for r0 in range(0, n, block):          # the block's columns rotated differently per chunk
        k = min(block, n - r0)
        chunk = np.ascontiguousarray(np.roll(base, 37 * (r0 // block), axis=1)[:k])
        check(lib.mxb_matrix_upload_rows(ctx.handle, dev.handle, r0, k, ptr(chunk)))
    wts = rs.randint(1, 30, size=n).astype(np.int64)
    args = argparse.Namespace(min_reads=10)

    paths = {"vote_first": lambda: consumers.find_contribs_from_reads(dev, wts, args),
             "vote_count_unique": lambda: old_path(dev, wts, 10)}
    results = {name: fn() for name, fn in paths.items()}          # warm-up
    results = {name: fn() for name, fn in paths.items()}
    assert results["vote_first"] == results["vote_count_unique"], "the two paths differ"
    times = {name: [] for name in paths}
    for _ in range(opt.reps):
        for name, fn in paths.items():
            ctx.synchronize()
            t0 = time.perf_counter()
            fn()
            times[name].append(time.perf_counter() - t0)
    gbytes = n * h * 8 / 1e9
    report = {"card": card(), "rows": n, "cols": h, "matrix_gb": round(gbytes, 3),
              "reps": opt.reps, "contributors": len(results["vote_first"])}
    for name, ts in times.items():
        med = float(np.median(ts))
        report[name] = {"median_ms": round(med * 1e3, 3), "min_ms": round(min(ts) * 1e3, 3),
                        "max_ms": round(max(ts) * 1e3, 3), "gb_per_s": round(gbytes / med, 1)}
    line = json.dumps(report)
    print(line)
    if opt.out:
        with open(opt.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
