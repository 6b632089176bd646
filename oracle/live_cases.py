#!/usr/bin/env python
"""Seeded cases of the tests that compare with the unmodified reference, and the
reference's outputs on them (tests/golden/golden_live.npz).

TEST INFRASTRUCTURE ONLY.  The tests rebuild the inputs with the functions below
(the Build-17 reads of the first case are stored with the outputs) and compare
the code under test with the stored outputs, so the comparisons also run where
the reference is not installed.  Where it is installed (oracle/refload.py) they
check the stored outputs against the reference as well.

    python oracle/live_cases.py

writes the file.  It takes the outputs from the reference when refload finds it,
and otherwise from the restatements in oracle/oracle_np.py that these same tests
hold bit-identical to the reference (build_em_matrix, run_em, em_step,
reduce_reads, and the consumers of the EM result).  The ``source`` entry of the
file says which.
"""
import argparse
import collections
import os
import sys
import types
import warnings

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import oracle_np, refload  # noqa: E402

GOLDEN_PATH = os.path.join(ROOT, "tests", "golden", "golden_live.npz")


def load_golden():
    return dict(np.load(GOLDEN_PATH))


def make_args(**kw):
    base = dict(verbose=False, init_alpha=1.0, tolerance=1e-4, max_iter=1000, n_multi=1)
    base.update(kw)
    return argparse.Namespace(**base)


def seeded_inits(seed, n_multi, h):
    """The Dirichlet starts the reference's run_em draws after np.random.seed(seed)."""
    np.random.seed(seed)
    return np.array([np.log(np.random.dirichlet([1.0] * h)) for _ in range(n_multi)])


# ---- Build-17: 12 reads of an H1/M7 mixture, matrix and a 2-restart run_em ------------------
def build17_reads(phylo17):
    from mixemt_b200 import synth
    mix = synth.make_mixture(phylo17, phylo17.refseq, [("H1", 0.6), ("M7", 0.4)], 300, seed=9)
    return mix.signatures[:12], mix.weights[:12]


def build17_sub(mat):
    """Every 11th haplogroup column: the run_em sub-problem."""
    return mat[:, ::11].copy()


RUN_EM_SEED, RUN_EM_MULTI, RUN_EM_MAX_ITER = 77, 2, 200


# ---- consumers of the EM result on a 150 x 40 stand-in ---------------------------------------
def consumers_case():
    props, mix, wts = oracle_np.synthetic_em_result(99, n=150, h=40)
    haps = ["hg%d" % j for j in range(40)]
    top = np.argsort(props)[::-1][:3].tolist()
    contribs = [["hap%d" % (k + 1), haps[j], props[j]] for k, j in enumerate(top)]
    return props, mix, wts, haps, contribs


CONSUMERS_MIN_READS, CONSUMERS_FOLD = 25, 2.0


def decode_assign(res, n):
    """assign_read_indexes' {name: rows} as one code per row (-1 unassigned, k for hap<k+1>)."""
    out = np.full(n, -2, dtype=np.int32)
    for name, rows in res.items():
        out[sorted(rows)] = -1 if name == 'unassigned' else int(name[3:]) - 1
    return out


# ---- em_step on 200 small inputs with the domain's edge values -------------------------------
def em_step_cases():
    """-inf cells, ties among row and column maxima, a row that fits no haplotype,
    zero weights, components with zero proportion."""
    rs = np.random.RandomState(0)
    for it in range(200):
        n, h = rs.randint(1, 14), rs.randint(1, 10)
        mat = -rs.gamma(2.0, 4.0, size=(n, h))
        mode = it % 5
        if mode >= 1:
            mat[rs.rand(n, h) < 0.2] = -np.inf
        if mode >= 2:
            mat = np.round(mat)
        if mode == 3:
            mat[rs.randint(n)] = -np.inf
        wts = rs.randint(0 if mode >= 2 else 1, 50, size=n)
        lp = np.log(rs.dirichlet([1.0] * h))
        if mode == 4:
            lp[rs.rand(h) < 0.3] = -np.inf
        yield mat, wts, lp


# ---- reduce_reads on 1500 seeded fragments ---------------------------------------------------
def reduce_case():
    return oracle_np.synthetic_read_obs(5, n_frag=1500)


def encode_read_sigs(read_sigs):
    """{signature: [read ids]} in dict order as two strings (signatures, ids per row)."""
    return ("\n".join(read_sigs), "\n".join(",".join(ids) for ids in read_sigs.values()))


# ---- build_em_matrix on 60 random small trees ------------------------------------------------
def packing_cases():
    """Trees with the variant spellings Phylotree has -- '(A73G)', 'T152C!', 'C150T!!',
    lower-case derived bases, back mutations onto the reference base, several variants of
    one haplogroup at one position, markers at positions that are not variant sites,
    mutation counts past the 0.5 cap -- and signatures with repeated and unsorted positions
    and 'N' observations."""
    rs = np.random.RandomState(1)
    for _ in range(60):
        ref_len = rs.randint(30, 200)
        refseq = "".join("ACGT"[i] for i in rs.randint(0, 4, size=ref_len))
        n_pos = rs.randint(1, min(25, ref_len))
        positions = np.sort(rs.choice(ref_len, size=n_pos, replace=False)).tolist()
        variants = {}
        for p in positions:
            cnt = collections.Counter()
            for _ in range(rs.randint(1, 4)):
                cnt[rs.choice(list("ACGT"))] += int(rs.randint(1, 80))
            variants[p] = cnt
        hap_var = {}
        for j in range(rs.randint(1, 12)):
            vs = []
            for _ in range(rs.randint(0, 8)):
                p = int(rs.choice(positions)) if rs.rand() < 0.85 else int(rs.randint(ref_len))
                v = "%s%d%s" % (refseq[p], p + 1, rs.choice(list("ACGTacgt")))
                r = rs.rand()
                v = ("(" + v + ")" if r < 0.15 else v + "!" if r < 0.3 else v + "!!" if r < 0.35
                     else "(" + v + "!)" if r < 0.4 else v)
                vs.append(v)
            hap_var["h%d" % j] = vs
        phylo = types.SimpleNamespace(variants=variants, hap_var=hap_var, refseq=refseq)
        haps = sorted(hap_var)
        reads = []
        for _ in range(rs.randint(1, 10)):
            ps = rs.choice(positions, size=rs.randint(1, n_pos + 1), replace=rs.rand() < 0.2)
            reads.append(",".join("%d:%s" % (p, rs.choice(list("ACGTN"))) for p in ps))
        yield refseq, phylo, haps, reads


# ---- the expected outputs ---------------------------------------------------------------------
def expected_outputs(phylo17, ref=True):
    """Every stored output, from the reference (``ref``, needs refload.available()) or
    from the oracle_np restatements."""
    if ref:
        _, ref_pre, ref_em = refload.load()
        from mixemt import assemble
    out = {"source": np.array("unmodified reference (mixemt)" if ref else
                              "oracle_np restatements, bit-identical to the reference "
                              "in the tests that use this file")}

    reads, wts = build17_reads(phylo17)
    haps = sorted(phylo17.hap_var)
    if ref:
        mat = ref_pre.build_em_matrix(phylo17.refseq, phylo17, reads, haps, make_args())
    else:
        mat = oracle_np.build_matrix_fast(phylo17.refseq, phylo17, reads, haps)[0]
    sub = build17_sub(mat)
    if ref:
        np.random.seed(RUN_EM_SEED)
        props, mix = ref_em.run_em(sub, wts, make_args(n_multi=RUN_EM_MULTI,
                                                       max_iter=RUN_EM_MAX_ITER))
    else:
        props, mix, _ = oracle_np.run_em(sub, wts, seeded_inits(RUN_EM_SEED, RUN_EM_MULTI,
                                                                sub.shape[1]),
                                         RUN_EM_MAX_ITER, 1e-4)
    out.update(b17_reads=np.array("\n".join(reads)), b17_weights=np.asarray(wts),
               b17_mat=mat, b17_props=props, b17_mix=mix)

    props, mix, cwts, chaps, contribs = consumers_case()
    if ref:
        found = assemble._find_contribs_from_reads(mix, cwts, make_args(min_reads=CONSUMERS_MIN_READS))
        res = assemble.assign_read_indexes(contribs, (props, mix), chaps, list(range(len(mix))),
                                           CONSUMERS_FOLD)
        red, cols = ref_pre.reduce_em_matrix(mix, chaps, contribs)
    else:
        found = oracle_np.find_contribs_from_reads(mix, cwts, CONSUMERS_MIN_READS)
        res = oracle_np.assign_read_indexes(contribs, (props, mix), chaps, len(mix), CONSUMERS_FOLD)
        red, cols = oracle_np.reduce_em_matrix(mix, chaps, contribs)
    out.update(c_contribs=np.asarray(found, dtype=np.int64), c_assign=decode_assign(res, len(mix)),
               c_reduced=red, c_reduced_cols=np.asarray([chaps.index(x) for x in cols]))

    zs, ps = [], []
    with warnings.catch_warnings(), np.errstate(all="ignore"):
        warnings.simplefilter("ignore")
        for mat, wts_, lp in em_step_cases():
            if ref:
                z, p = ref_em.em_step(mat, wts_, lp, np.empty_like(mat))
            else:
                z, p = oracle_np.em_step(mat, wts_, lp)
            zs.append(np.asarray(z, dtype=np.float64).ravel())
            ps.append(np.asarray(p, dtype=np.float64).ravel())
    out.update(step_z=np.concatenate(zs), step_p=np.concatenate(ps))

    read_obs = reduce_case()
    sigs = ref_pre.reduce_reads(read_obs) if ref else oracle_np.reduce_reads(read_obs)
    out["r_sigs"], out["r_ids"] = (np.array(s) for s in encode_read_sigs(sigs))

    mats = []
    for refseq, phylo, phaps, preads in packing_cases():
        if ref:
            m = ref_pre.build_em_matrix(refseq, phylo, preads, phaps, argparse.Namespace(verbose=False))
        else:
            m = oracle_np.build_matrix_loops(refseq, phylo, preads, phaps)[0]
        mats.append(np.asarray(m, dtype=np.float64).ravel())
    out["pack_mats"] = np.concatenate(mats)
    return out


if __name__ == "__main__":
    from mixemt_b200.phylo_tables import PhyloTables
    phylo = PhyloTables.load(os.path.join(ROOT, "tests", "golden", "phylotree17.npz"))
    out = expected_outputs(phylo, ref=refload.available())
    np.savez_compressed(GOLDEN_PATH, **out)
    print("%s written (%s), %.1f KB" % (GOLDEN_PATH, out["source"],
                                        os.path.getsize(GOLDEN_PATH) / 1024.0))
