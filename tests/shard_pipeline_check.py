"""The pipeline after the fit in rows mode, launched by torchrun (see
test_shard_pipeline.py):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 \
        --master-addr 127.0.0.1 --master-port 29527 tests/shard_pipeline_check.py OUTDIR

sharded build_em_input_arrays -> rows run_em -> find_contribs_from_reads ->
reduce_em_matrix -> refinement rows run_em (H = 2-3) -> assign_read_indexes ->
save_npy / load_npy, against the same chain on one GPU over the whole matrix: the same
contributors, proportions within 1e-12, identical assignments, a byte-identical file.
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def build17_fragments():
    """Fragments made by repeating each row of a Build-17 mixture weights[r] times."""
    from mixemt_b200 import synth
    from mixemt_b200.phylo_tables import PhyloTables
    phylo = PhyloTables.load(os.path.join(ROOT, "tests", "golden", "phylotree17.npz"))
    mix = synth.make_mixture(phylo, phylo.refseq, [("H1", 0.5), ("L3e", 0.3), ("U5a1", 0.2)],
                             1500, seed=7, strings=False)
    positions = np.asarray(sorted(phylo.variants), dtype=np.int32)
    rows = np.repeat(np.arange(mix.n_rows), mix.weights)
    obs = [np.arange(mix.row_ptr[r], mix.row_ptr[r + 1]) for r in rows.tolist()]
    frag_ptr = np.zeros(len(rows) + 1, dtype=np.int64)
    np.cumsum([len(o) for o in obs], out=frag_ptr[1:])
    idx = np.concatenate(obs)
    return phylo, frag_ptr, positions[mix.pos_idx[idx]], mix.base_ascii[idx]


def chain(frags, args, out_dir, tag):
    """Build, fit, contributors, reduce, refine, assign, save; returns what is compared."""
    from mixemt_b200 import consumers, em
    from mixemt_b200.preprocess import build_em_input_arrays
    phylo, frag_ptr, pos, base = frags
    dmat, w, haps, red = build_em_input_arrays(frag_ptr, pos, base, phylo.refseq, phylo, args,
                                               keep_device=True)
    inits = np.log(np.random.RandomState(8).dirichlet([1.0] * len(haps)))[None, :]
    props, _, _, mix = em.run_em_device(dmat, w, args, keep_device=True, want_host=False,
                                        inits=inits)
    contribs = consumers.find_contribs_from_reads(mix, w, args)
    cons = [["hap%d" % (k + 1), haps[j], props[j]] for k, j in enumerate(contribs[:3])]
    small, new_haps = consumers.reduce_em_matrix(dmat, haps, cons)
    inits2 = np.log(np.random.RandomState(9).dirichlet([1.0] * len(new_haps)))[None, :]
    props2, _, _, mix2 = em.run_em_device(small, w, args, keep_device=True, want_host=False,
                                          inits=inits2)
    cons2 = [[name, group, props2[new_haps.index(group)]] for name, group, _ in cons]
    assign = consumers.assign_read_indexes(cons2, (props2, mix2), new_haps,
                                           list(range(mix2.shape[0])), 2.0)
    path = consumers.save_npy(dmat, os.path.join(out_dir, "em_input_%s" % tag))
    path2 = consumers.save_npy(mix2, os.path.join(out_dir, "refined_%s" % tag))
    back = consumers.load_npy(path2, sharded=mix2.row_shard is not None)
    assert np.array_equal(back.to_host(), mix2.to_host()), "load_npy did not return the rows"
    return {"contribs": contribs, "props": props, "new_haps": new_haps, "props2": props2,
            "assign": {k: set(v) for k, v in assign.items()}, "path": path,
            "h2": len(new_haps)}


def main():
    import torch
    import torch.distributed as dist
    from conftest import make_args
    from mixemt_b200.runtime import get_context

    out_dir = sys.argv[1]
    local = int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    rank, world = dist.get_rank(), dist.get_world_size()
    ctx = get_context()
    ctx.init_comm_from_torch()
    frags = build17_fragments()

    rows = chain(frags, make_args(b200_shard="rows", max_iter=300, tolerance=1e-7, min_reads=10),
                 out_dir, "rows")
    assert 2 <= rows["h2"] <= 3, rows["new_haps"]
    gathered = [None] * world
    dist.all_gather_object(gathered, (rows["contribs"], rows["assign"]))
    assert all(g[0] == rows["contribs"] for g in gathered), "ranks disagree on the contributors"
    union = {}
    for _, part in gathered:
        for name, rows_ in part.items():
            assert not rows_ & union.get(name, set())
            union.setdefault(name, set()).update(rows_)
    if rank == 0:
        one = chain(frags, make_args(max_iter=300, tolerance=1e-7, min_reads=10), out_dir, "one")
        assert one["contribs"] == rows["contribs"], (one["contribs"], rows["contribs"])
        dp = np.abs(one["props"] - rows["props"]).max()
        dp2 = np.abs(one["props2"] - rows["props2"]).max()
        assert dp < 1e-12 and dp2 < 1e-12, (dp, dp2)
        assert one["assign"] == union, "assignments differ"
        assert open(one["path"], "rb").read() == open(rows["path"], "rb").read(), "files differ"
        from mixemt_b200._lib import lib
        how = "p2p" if lib.mxb_comm_p2p_enabled(ctx.handle) else "nccl"
        print("SHARD_PIPELINE_OK world=%d contribs=%s h2=%d dprops=%.2e dprops2=%.2e exchange=%s"
              % (world, rows["contribs"][:3], rows["h2"], dp, dp2, how))
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
