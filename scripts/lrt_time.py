"""Time the contributor likelihood-ratio test against what a user would write without it.

The two seeded Build-17 matrices of scripts/bootstrap_time.py (config-1 and config-2 size).  For
each: the fit, then K = the contributors plus the next highest-proportion columns up to 16;
(a) contributor_lrt (1 + K refits side by side on class tiles, one log_likelihood call),
(b) 1 + K sequential one-restart run_em_device calls from the same starts, then log_likelihood
of the 1 + K results.  (a) and (b) must agree (iteration counts equal, proportions within 1e-13,
log-likelihoods within 1e-12 of sum_i w_i |l_i|).  One warm-up of each, then --pairs alternated
(a, b) pairs.  Then log_likelihood alone at K = 1, 4 and 16 on the config-2 matrix (CUDA events
around --reps calls, warm), with GB/s over the 8 N H bytes of the matrix it reads once per call.
Prints and writes JSON (--out), with the card's name and power limit read in the same run."""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

from bootstrap_time import build, card   # noqa: E402


def columns(props, contribs, k_max=16):
    cols = list(contribs)
    for c in np.argsort(props)[::-1]:
        if len(cols) >= k_max:
            break
        if int(c) not in cols and props[c] > 0:
            cols.append(int(c))
    return cols


def measure(name, dev, wts, pairs, seed):
    from conftest import make_args
    from mixemt_b200 import consumers, em, likelihood
    a = make_args(max_iter=1000, tolerance=1e-4, min_reads=10)
    np.random.seed(seed)
    props, _, _, mix_dev = em.run_em_device(dev, wts, a, keep_device=True, want_host=False)
    contribs = consumers.find_contribs_from_reads(mix_dev, wts.astype(np.int64), a)
    mix_dev.free()
    cols = columns(props, contribs)
    starts = np.vstack([np.log(props) - np.log(props.sum())] +
                       [likelihood.null_start(props, c) for c in cols])

    def run_a():
        t0 = time.perf_counter()
        res = likelihood.contributor_lrt(dev, wts, a, props, cols)
        return time.perf_counter() - t0, res

    def run_b():
        t0 = time.perf_counter()
        lnp, iters = np.empty_like(starts), []
        for k, s in enumerate(starts):
            lin, _, info, _ = em.run_em_device(dev, wts, a, want_host=False,
                                               inits=s.reshape(1, -1))
            with np.errstate(divide="ignore"):
                lnp[k] = np.log(lin)
            iters.append(info["iterations"][0])
        ll = likelihood.log_likelihood(dev, wts, np.exp(lnp))
        return time.perf_counter() - t0, (lnp, np.array(iters), ll)

    run_a(), run_b()
    ta, tb = [], []
    for _ in range(pairs):
        t, res = run_a()
        ta.append(t)
        t, (lnp, iters, ll) = run_b()
        tb.append(t)
    assert np.array_equal(res.iterations, iters), (res.iterations, iters)
    fits = np.vstack([res.lnprops_full, res.lnprops_null])
    diff = float(np.abs(np.exp(fits) - np.exp(lnp)).max())
    assert diff <= 1e-13, diff
    lls = np.concatenate([[res.loglik_full], res.loglik_null])
    ll_diff = float(np.abs(lls - ll).max())
    assert ll_diff <= 1e-12 * abs(res.loglik_full), ll_diff     # = sum_i w_i |l_i| (M <= 0)
    out = {
        "matrix": name, "rows": dev.shape[0], "haplotypes": dev.shape[1],
        "contributors": len(contribs), "K": len(cols), "slots_R": res.slots,
        "mean_iterations": float(res.iterations.mean()), "max_prop_diff": diff,
        "max_loglik_diff": ll_diff, "loglik_full": res.loglik_full,
        "statistic": res.statistic.tolist(), "pvalue": res.pvalue.tolist(),
        "lrt_s": ta, "sequential_s": tb,
        "speedup_median": float(np.median(tb) / np.median(ta)),
    }
    print(json.dumps(out), flush=True)
    return out, props


def loglik_rate(dev, wts, props, reps):
    import torch
    from mixemt_b200 import likelihood
    n, h = dev.shape
    rs = np.random.RandomState(0)
    out = []
    for k in (1, 4, 16):
        vecs = np.tile(props, (k, 1)) * rs.uniform(0.5, 1.5, size=(k, h))
        likelihood.log_likelihood(dev, wts, vecs)          # warm-up
        start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        start.record()
        t0 = time.perf_counter()
        for _ in range(reps):
            likelihood.log_likelihood(dev, wts, vecs)
        end.record()
        end.synchronize()
        wall = (time.perf_counter() - t0) / reps
        ms = start.elapsed_time(end) / reps
        res = {"K": k, "call_ms": ms, "wall_ms": wall * 1e3,
               "GB_per_s": 8.0 * n * h / (ms * 1e-3) / 1e9, "matrix_GB": 8.0 * n * h / 1e9}
        print(json.dumps(res), flush=True)
        out.append(res)
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--pairs", type=int, default=3)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--skip-config2", action="store_true")
    ap.add_argument("--out", default=None)
    opts = ap.parse_args()
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    results = {"card": card()}
    dev, wts = build(10000, [("H1", 0.7), ("L3e", 0.3)], seed=1)
    results["config1"], _ = measure("config-1 size", dev, wts, opts.pairs, seed=11)
    dev.free()
    if not opts.skip_config2:
        dev, wts = build(1000000, [("H1", 0.5), ("L3e", 0.3), ("U5a1", 0.2)], seed=2)
        results["config2"], props = measure("config-2 size", dev, wts, opts.pairs, seed=12)
        results["loglik_config2"] = loglik_rate(dev, wts, props, opts.reps)
        dev.free()
    results["card_after"] = card()
    print(json.dumps({"card": results["card"], "card_after": results["card_after"]}))
    if opts.out:
        os.makedirs(os.path.dirname(os.path.abspath(opts.out)), exist_ok=True)
        with open(opts.out, "w") as f:
            json.dump(results, f, indent=1)


if __name__ == "__main__":
    main()
