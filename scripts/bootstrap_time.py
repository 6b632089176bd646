"""Time the bootstrap against what a user would write without it.

Two seeded Build-17 matrices: config-1 size (H1 70 % / L3e 30 %, 10 000 fragments) and
config-2 size (bench.py's: H1 / L3e / U5a1 50 / 30 / 20, 1 000 000 fragments).  For each:
(a) bootstrap_props with n_boot = 4 R (R = the replicates the session iterates per launch),
(b) the same replicates as n_boot sequential run_em_device calls on the counts of
mxb_boot_counts.  (a) and (b) must agree (iteration counts equal, proportions within 1e-13).
One warm-up of each per shape, then --pairs alternated (a, b) pairs.  Prints and writes JSON
(--out) with replicates/s, mean iterations, R, launches per replicate-iteration, and the card's
name and power limit read in the same run."""
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
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except OSError as e:   # pragma: no cover
        return "unknown (%s)" % e


def build(fragments, mixture, seed):
    from mixemt_b200.phylo_tables import PhyloTables
    from mixemt_b200 import synth
    from mixemt_b200.preprocess import HapVarBaseMatrix, build_matrix_from_csr
    from mixemt_b200.runtime import get_context
    phylo = PhyloTables.load(os.path.join(ROOT, "tests", "golden", "phylotree17.npz"))
    haps = sorted(phylo.hap_var)
    mix = synth.make_mixture(phylo, phylo.refseq, mixture, fragments, seed=seed)
    tables = HapVarBaseMatrix(phylo.refseq, phylo, haps).pack()
    out = build_matrix_from_csr(tables, mix.csr(tables), ctx=get_context(), want_host=False,
                                keep_device=True)
    return out[2], mix.weights.astype(np.float64)


def measure(name, dev, wts, pairs, seed):
    from conftest import make_args
    from mixemt_b200 import bootstrap, em
    ctx = dev.ctx
    a = make_args(max_iter=1000, tolerance=1e-4)
    np.random.seed(seed)
    props, _ = em.run_em(dev, wts, a)
    with np.errstate(divide="ignore"):
        start = np.log(props) - np.log(props.sum())
    r = bootstrap.bootstrap_props(dev, wts, a, props, n_boot=1, seed=seed).slots
    n_boot = 4 * r

    def run_a():
        l0 = ctx.launch_count
        t0 = time.perf_counter()
        res = bootstrap.bootstrap_props(dev, wts, a, props, n_boot=n_boot, seed=seed)
        return time.perf_counter() - t0, res, ctx.launch_count - l0

    def run_b():
        l0 = ctx.launch_count
        t0 = time.perf_counter()
        counts = bootstrap.boot_counts(wts, seed, 0, n_boot).astype(np.float64)
        lin, iters = np.empty((n_boot, len(props))), []
        for b in range(n_boot):
            lin[b], _, info, _ = em.run_em_device(dev, counts[b], a, want_host=False,
                                                  inits=start.reshape(1, -1))
            iters.append(info["iterations"][0])
        return time.perf_counter() - t0, (lin, np.array(iters)), ctx.launch_count - l0

    run_a(), run_b()                  # warm-up of both shapes
    ta, tb = [], []
    for _ in range(pairs):
        t, res, la = run_a()
        ta.append(t)
        t, (lin, iters), lb = run_b()
        tb.append(t)
    assert np.array_equal(res.iterations, iters), (res.iterations, iters)
    diff = float(np.abs(res.props - lin).max())
    assert diff <= 1e-13, diff
    it_sum = int(res.iterations.sum())
    out = {
        "matrix": name, "rows": dev.shape[0], "haplotypes": dev.shape[1], "slots_R": r,
        "n_boot": n_boot, "mean_iterations": float(res.iterations.mean()),
        "max_prop_diff": diff,
        "bootstrap_s": ta, "sequential_s": tb,
        "bootstrap_replicates_per_s": n_boot / float(np.median(ta)),
        "sequential_replicates_per_s": n_boot / float(np.median(tb)),
        "speedup_median": float(np.median(tb) / np.median(ta)),
        "bootstrap_launches_per_replicate_iteration": la / it_sum,
        "sequential_launches_per_replicate_iteration": lb / it_sum,
    }
    print(json.dumps(out), flush=True)
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--pairs", type=int, default=3)
    ap.add_argument("--skip-config2", action="store_true")
    ap.add_argument("--out", default=None)
    opts = ap.parse_args()
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    results = {"card": card()}
    dev, wts = build(10000, [("H1", 0.7), ("L3e", 0.3)], seed=1)
    results["config1"] = measure("config-1 size", dev, wts, opts.pairs, seed=11)
    dev.free()
    if not opts.skip_config2:
        dev, wts = build(1000000, [("H1", 0.5), ("L3e", 0.3), ("U5a1", 0.2)], seed=2)
        results["config2"] = measure("config-2 size", dev, wts, opts.pairs, seed=12)
        dev.free()
    results["card_after"] = card()
    print(json.dumps({"card": results["card"], "card_after": results["card_after"]}))
    if opts.out:
        os.makedirs(os.path.dirname(os.path.abspath(opts.out)), exist_ok=True)
        with open(opts.out, "w") as f:
            json.dump(results, f, indent=1)


if __name__ == "__main__":
    main()
