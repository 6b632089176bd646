"""Outputs of the EM driver on fixed seeds, for comparing two builds bit for bit.

    python scripts/em_driver_parity.py --out DIR [--tree PATH]
    python scripts/em_driver_parity.py --compare DIR_A DIR_B

The first form runs run_em / em_step through the Python API of the package in PATH (default:
this repository) and writes one .npz per case: proportions, read matrix, iterations, converged
flags and the kernel launches the call issued (ctx.launch_count).  Cases: the toy and Build-17
matrices with 1 and 3 restarts; the 2500 x 5408 noise matrix with 2 and 5 restarts, two per pass
and one at a time (MXB_EM_NO_BATCH=1); starts whose row likelihoods underflow (one restart on
fp64 rows and on class tiles, the "UFU" restarts two per pass and one at a time); max_iter 0
and 1; the split tail (MXB_EM_SPLIT_TAIL=1) and the general path (MXB_EM_FORCE_GENERAL=1);
sessions driven by mxb_em_iterate (mxb_em_get_lnprops and mxb_em_read_mix read back), by
mxb_em_iterate_fixed (20 iterations) and by mxb_em_profile (launch count only: its times are
not compared); em_step on the toy and the noise matrix; bootstraps on the Build-17 tiles with
fewer replicates than slots and with more (refilled slots), over fp64 rows, from a start whose
row likelihoods underflow, at max_iter 0, and on the toy matrix with more replicates than one
output window (4096); constrained refits (mxb_em_refit) on the Build-17 tiles with one start and
with more starts than slots, over fp64 rows, from the underflowing starts, from starts with a
-inf column (likelihood.null_start) and at max_iter 0.  The second form compares two such
directories: every array and every launch count must be equal; launch counts are printed side
by side.
"""
import argparse
import glob
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")


def _args(**kw):
    base = dict(verbose=False, init_alpha=1.0, tolerance=1e-4, max_iter=1000, n_multi=1)
    base.update(kw)
    return argparse.Namespace(**base)


def _inputs():
    """name -> (matrix, weights, inits with 5 rows) on fixed seeds."""
    from mixemt_b200 import synth
    from mixemt_b200.phylo_tables import PhyloTables
    from mixemt_b200.preprocess import HapVarBaseMatrix, build_matrix_from_csr
    out = {}
    toy = np.load(os.path.join(GOLDEN, "golden_toy.npz"))["em_mat"]
    out["toy"] = (toy, np.arange(1, toy.shape[0] + 1, dtype=np.float64))

    phylo = PhyloTables.load(os.path.join(GOLDEN, "phylotree17.npz"))
    haps = sorted(phylo.hap_var)
    mix = synth.make_mixture(phylo, phylo.refseq, [("H1", 0.5), ("L3e", 0.3), ("U5a1", 0.2)],
                             4000, seed=4)
    tables = HapVarBaseMatrix(phylo.refseq, phylo, haps).pack()
    b17, _, _, _ = build_matrix_from_csr(tables, mix.csr(tables))
    out["b17"] = (b17, mix.weights.astype(np.float64))

    rs = np.random.RandomState(11)      # test_batched_restarts_equal_sequential's matrix
    noise = -rs.gamma(2.0, 8.0, size=(2500, 5408))
    noise[rs.rand(2500, 5408) < 0.4] = 0.0
    noise[:, :40] += 3.0
    out["noise"] = (noise, rs.randint(1, 50, size=2500).astype(np.float64))

    for layout in ("fp64", "tiles"):    # test_logspace_rescue_gpu.py's underflowing matrices
        rs = np.random.RandomState(5)
        if layout == "fp64":
            n, h = 300, 1100
            m = -rs.gamma(2.0, 3.0, size=(n, h))
        else:
            n, h = 1280, 5408
            m = np.repeat(-rs.gamma(2.0, 3.0, size=(n, h // 64 + 1)), 64, axis=1)[:, :h].copy()
        m[:, 0] = 0.0
        m[: n // 4, 1:] -= 800.0
        out["under_" + layout] = (m, rs.randint(1, 5, size=n).astype(np.float64))

    res = {}
    for name, (m, w) in out.items():
        h = m.shape[1]
        if name.startswith("under_"):
            under = np.full(h, -np.log(h - 1.0))
            under[0] = -760.0
            fine = np.full(h, -np.log(float(h)))
            inits = np.array([under, fine, under, fine, under])
        else:
            inits = np.log(np.random.RandomState(h).dirichlet([1.0] * h, size=5))
        res[name] = (np.ascontiguousarray(m), w, inits)
    return res


def _cases():
    """(case name, matrix, n_multi, max_iter, tol, environment, kind)."""
    c = []
    for mat, it, tol in (("toy", 1000, 1e-6), ("b17", 400, 1e-5)):
        for k in (1, 3):
            c.append(("%s_n%d" % (mat, k), mat, k, it, tol, {}, "run"))
    for k in (2, 5):
        c.append(("noise_n%d" % k, "noise", k, 90, 3e-3, {}, "run"))
        c.append(("noise_n%d_nobatch" % k, "noise", k, 90, 3e-3, {"MXB_EM_NO_BATCH": "1"}, "run"))
    c.append(("under_fp64_n1", "under_fp64", 1, 60, 1e-6, {}, "run"))
    c.append(("under_tiles_n1", "under_tiles", 1, 60, 1e-6, {}, "run"))
    c.append(("under_fp64_UFU", "under_fp64", 3, 60, 1e-6, {}, "run"))
    c.append(("under_fp64_UFU_nobatch", "under_fp64", 3, 60, 1e-6, {"MXB_EM_NO_BATCH": "1"},
              "run"))
    for it in (0, 1):
        for mat, env in (("toy", {}), ("b17", {}), ("b17", {"MXB_EM_NO_PACK": "1"}),
                         ("noise", {})):
            for k in (1, 3):
                tag = "_rows" if env else ""
                c.append(("%s%s_n%d_iter%d" % (mat, tag, k, it), mat, k, it, 1e-4, env, "run"))
    for mat, it, tol in (("toy", 1000, 1e-6), ("noise", 90, 3e-3), ("under_fp64", 60, 1e-6),
                         ("under_tiles", 60, 1e-6), ("b17", 0, 1e-4), ("b17", 1, 1e-4)):
        c.append(("%s_session_iter%d" % (mat, it), mat, 1, it, tol, {}, "session"))
    split, general = {"MXB_EM_SPLIT_TAIL": "1"}, {"MXB_EM_FORCE_GENERAL": "1"}
    for mat, it, tol in (("b17", 400, 1e-5), ("noise", 90, 3e-3)):
        for tag, env in (("split", split), ("general", general)):
            for k in (1, 3):
                c.append(("%s_%s_n%d" % (mat, tag, k), mat, k, it, tol, env, "run"))
            c.append(("%s_%s_session" % (mat, tag), mat, 1, it, tol, env, "session"))
    for kind in ("fixed", "profile"):
        c.append(("b17_%s20" % kind, "b17", 1, 20, 0.0, {}, kind))
        c.append(("b17_rows_%s20" % kind, "b17", 1, 20, 0.0, {"MXB_EM_NO_PACK": "1"}, kind))
    c.append(("b17_boot1", "b17", 1, 400, 1e-5, {}, "boot"))
    c.append(("b17_boot40", "b17", 40, 400, 1e-5, {}, "boot"))
    c.append(("b17_rows_boot5", "b17", 5, 400, 1e-5, {"MXB_EM_NO_PACK": "1"}, "boot"))
    c.append(("under_tiles_boot3", "under_tiles", 3, 60, 1e-6, {}, "boot"))
    c.append(("b17_boot5_iter0", "b17", 5, 0, 1e-5, {}, "boot"))
    c.append(("toy_boot4100", "toy", 4100, 30, 1e-4, {}, "boot"))
    c.append(("b17_refit1", "b17", 1, 400, 1e-5, {}, "refit"))
    c.append(("b17_refit40", "b17", 40, 400, 1e-5, {}, "refit"))
    c.append(("b17_rows_refit5", "b17", 5, 400, 1e-5, {"MXB_EM_NO_PACK": "1"}, "refit"))
    c.append(("under_tiles_refit3", "under_tiles", 3, 60, 1e-6, {}, "refit"))
    c.append(("b17_refit_null4", "b17", 4, 400, 1e-5, {}, "refit_null"))
    c.append(("b17_refit5_iter0", "b17", 5, 0, 1e-5, {}, "refit"))
    c.append(("toy_em_step", "toy", 1, 1, 0.0, {}, "step"))
    c.append(("noise_em_step", "noise", 1, 1, 0.0, {}, "step"))
    return c


def _session(ctx, m, w, init, max_iter, tol):
    """mxb_em_set_lnprops + mxb_em_iterate on a session, then both log-proportions
    (mxb_em_get_lnprops 0 and 1, concatenated) and the read matrix (mxb_em_read_mix)."""
    import ctypes
    from mixemt_b200._lib import check, lib, ptr
    from mixemt_b200.runtime import DeviceMatrix
    n, h = m.shape
    dev = DeviceMatrix.from_host(ctx, m)
    sess, mix_h = ctypes.c_void_p(), ctypes.c_void_p()
    check(lib.mxb_em_create(ctx.handle, dev.handle, ptr(w), 0, ctypes.byref(sess)))
    check(lib.mxb_matrix_alloc(ctx.handle, n, h, ctypes.byref(mix_h)))
    l0 = ctx.launch_count
    check(lib.mxb_em_set_lnprops(sess, ptr(np.ascontiguousarray(init))))
    it, cv = ctypes.c_int64(), ctypes.c_int32()
    check(lib.mxb_em_iterate(sess, max_iter, tol, ctypes.byref(it), ctypes.byref(cv)))
    props = np.empty(2 * h)
    check(lib.mxb_em_get_lnprops(sess, 0, ptr(props[:h])))
    check(lib.mxb_em_get_lnprops(sess, 1, ptr(props[h:])))
    check(lib.mxb_em_read_mix(sess, mix_h, 0, 0.0))
    launches = ctx.launch_count - l0
    mix_dev = DeviceMatrix(ctx, mix_h)
    mix = mix_dev.to_host()
    mix_dev.free()
    lib.mxb_em_destroy(sess)
    dev.free()
    return props, mix, [it.value], [cv.value], launches


def _fixed(ctx, m, w, init, n_iter, profile):
    """mxb_em_iterate_fixed (or mxb_em_profile) for n_iter iterations on a session, then both
    log-proportions (mxb_em_get_lnprops 0 and 1, concatenated)."""
    import ctypes
    from mixemt_b200._lib import check, lib, ptr
    from mixemt_b200.runtime import DeviceMatrix
    h = m.shape[1]
    dev = DeviceMatrix.from_host(ctx, m)
    sess = ctypes.c_void_p()
    check(lib.mxb_em_create(ctx.handle, dev.handle, ptr(w), 0, ctypes.byref(sess)))
    l0 = ctx.launch_count
    check(lib.mxb_em_set_lnprops(sess, ptr(np.ascontiguousarray(init))))
    if profile:
        check(lib.mxb_em_profile(sess, n_iter, (ctypes.c_float * 4)()))
    else:
        check(lib.mxb_em_iterate_fixed(sess, n_iter, ctypes.byref(ctypes.c_float()), None))
    launches = ctx.launch_count - l0
    props = np.empty(2 * h)
    check(lib.mxb_em_get_lnprops(sess, 0, ptr(props[:h])))
    check(lib.mxb_em_get_lnprops(sess, 1, ptr(props[h:])))
    lib.mxb_em_destroy(sess)
    dev.free()
    return props, np.zeros(0), [n_iter], [0], launches


def _boot(ctx, m, w, start, n_boot, max_iter, tol):
    """mxb_em_bootstrap of replicates 0 .. n_boot - 1 from `start` on seed 7: their final
    log-proportions, iterations and converged flags; the slot count goes with the read matrix."""
    from mixemt_b200 import bootstrap
    from mixemt_b200.runtime import DeviceMatrix
    dev = DeviceMatrix.from_host(ctx, m)
    l0 = ctx.launch_count
    lnp, iters, conv, slots = bootstrap._run(dev, w, np.ascontiguousarray(start), 0, n_boot, 7,
                                             _args(max_iter=max_iter, tolerance=tol))
    launches = ctx.launch_count - l0
    dev.free()
    return lnp, np.array([slots]), iters, conv, launches


def _refit_starts(m, inits, k, null):
    """The first k starts of a refit case: the case's inits, more Dirichlet draws past 5, or
    (null) the normalised first init and likelihood.null_start of it for k - 1 columns."""
    from mixemt_b200 import likelihood
    h = m.shape[1]
    if null:
        p = np.exp(inits[0])
        cols = [0, 5, h // 2, h - 1][:k - 1]
        return np.array([np.log(p / p.sum())] + [likelihood.null_start(p, c) for c in cols])
    if k <= len(inits):
        return inits[:k]
    return np.log(np.random.RandomState(h + 1).dirichlet([1.0] * h, size=k))


def _refit(ctx, m, w, starts, max_iter, tol):
    """mxb_em_refit from `starts`: their final log-proportions, iterations and converged flags;
    the slot count goes with the read matrix."""
    from mixemt_b200 import likelihood
    from mixemt_b200.runtime import DeviceMatrix
    dev = DeviceMatrix.from_host(ctx, m)
    l0 = ctx.launch_count
    lnp, iters, conv, slots = likelihood._refit(dev, w, np.ascontiguousarray(starts), max_iter,
                                                tol)
    launches = ctx.launch_count - l0
    dev.free()
    return lnp, np.array([slots]), iters, conv, launches


def run(out_dir):
    from mixemt_b200 import em
    from mixemt_b200.runtime import DeviceMatrix, get_context
    os.makedirs(out_dir, exist_ok=True)
    ctx = get_context()
    data = _inputs()
    for name, mat, k, it, tol, env, kind in _cases():
        m, w, inits = data[mat]
        saved = {v: os.environ.get(v) for v in env}
        os.environ.update(env)
        try:
            if kind == "session":
                props, mix, iters, conv, launches = _session(ctx, m, w, inits[0], it, tol)
            elif kind in ("fixed", "profile"):
                props, mix, iters, conv, launches = _fixed(ctx, m, w, inits[0], it,
                                                           kind == "profile")
            elif kind == "boot":
                props, mix, iters, conv, launches = _boot(ctx, m, w, inits[0], k, it, tol)
            elif kind in ("refit", "refit_null"):
                starts = _refit_starts(m, inits, k, kind == "refit_null")
                props, mix, iters, conv, launches = _refit(ctx, m, w, starts, it, tol)
            elif kind == "step":
                mix = np.empty_like(m)
                l0 = ctx.launch_count
                _, props = em.em_step(m, w, inits[0], mix)
                launches = ctx.launch_count - l0
                iters, conv = [1], [0]
            else:
                dev = DeviceMatrix.from_host(ctx, m)
                l0 = ctx.launch_count
                props, mix, info, _ = em.run_em_device(dev, w, _args(n_multi=k, max_iter=it,
                                                                    tolerance=tol),
                                                       inits=inits[:k])
                launches = ctx.launch_count - l0
                dev.free()
                iters, conv = info["iterations"], info["converged"]
        finally:
            for v, old in saved.items():
                if old is None:
                    del os.environ[v]
                else:
                    os.environ[v] = old
        np.savez(os.path.join(out_dir, name + ".npz"), props=props, mix=mix,
                 iters=np.asarray(iters), conv=np.asarray(conv), launches=np.int64(launches))
        print("%-28s iters %s launches %d" % (name, list(iters), launches), flush=True)


def compare(a, b):
    bad = 0
    for pa in sorted(glob.glob(os.path.join(a, "*.npz"))):
        name = os.path.basename(pa)[:-4]
        pb = os.path.join(b, name + ".npz")
        if not os.path.exists(pb):
            print("%-28s missing in %s" % (name, b))
            bad += 1
            continue
        x, y = np.load(pa), np.load(pb)
        diff = [f for f in ("props", "mix", "iters", "conv", "launches")
                if not np.array_equal(x[f], y[f])]
        bad += bool(diff)
        print("%-28s %-10s launches %6d %6d (%+d)" % (name, "DIFF " + ",".join(diff) if diff
                                                      else "equal", int(x["launches"]),
                                                      int(y["launches"]),
                                                      int(y["launches"]) - int(x["launches"])))
    print("PARITY %s" % ("OK" if bad == 0 else "FAILED (%d cases differ)" % bad))
    return bad == 0


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", help="write the outputs of every case here")
    ap.add_argument("--tree", default=ROOT, help="repository whose mixemt_b200 package runs")
    ap.add_argument("--compare", nargs=2, metavar=("DIR_A", "DIR_B"))
    o = ap.parse_args()
    if o.compare:
        sys.exit(0 if compare(*o.compare) else 1)
    if not o.out:
        ap.error("--out or --compare is required")
    sys.path.insert(0, os.path.abspath(o.tree))
    run(o.out)


if __name__ == "__main__":
    main()
