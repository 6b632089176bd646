"""Host rules of the bootstrap (mixemt_b200.bootstrap, csrc/bootstrap.cu, tile_plan.h), no GPU:
the numpy Philox4x32-10 against the Random123 known-answer vectors, the properties of a
replicate's fragment counts, argument validation, the replicate-slot rule and the restart
fan-out merge over 2- and 3-rank gloo groups."""
import ctypes
import math
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from mixemt_b200 import bootstrap, sharding
from mixemt_b200._lib import lib, check
from bootstrap_oracle import philox4x32_10, boot_counts
from conftest import make_args
from test_tile_plan import check_plan


@pytest.mark.parametrize("ctr,key,want", [
    ((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
    ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
    ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
     (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1)),
])
def test_philox_known_answers(ctr, key, want):
    assert tuple(int(x) for x in philox4x32_10(ctr, key)) == want


def _weights():
    w = np.random.RandomState(5).randint(0, 9, size=40).astype(np.float64)
    w[[0, 7, 39]] = 0
    return w


def test_counts_sum_to_w_and_skip_empty_rows():
    w = _weights()
    for seed, b in [(0, 0), (1, 3), (2 ** 53 - 1, 1000)]:
        c = boot_counts(w, seed, b)
        assert c.sum() == w.sum()
        assert (c[w == 0] == 0).all()


def test_replicate_counts_do_not_depend_on_the_batch():
    """Replicate b is a function of (w, seed, b): drawing 0..9 one by one or b alone agrees,
    and different b or seeds give different draws."""
    w = _weights()
    each = [boot_counts(w, 11, b) for b in range(10)]
    assert np.array_equal(each[6], boot_counts(w, 11, 6))
    assert not np.array_equal(each[0], each[1])
    assert not np.array_equal(each[0], boot_counts(w, 12, 0))


def test_counts_are_unbiased():
    """2000 replicates: the mean count of every row is within 4 sigma of its weight
    (multinomial: var = W p (1 - p))."""
    w = _weights()
    total = w.sum()
    mean = np.mean([boot_counts(w, 2024, b) for b in range(2000)], axis=0)
    p = w / total
    sd = np.sqrt(total * p * (1 - p) / 2000)
    assert (np.abs(mean - w) <= 4 * sd + 1e-12).all()


@pytest.mark.parametrize("weights,props,n_boot", [
    ([1, 2, np.nan], [0.5, 0.5], 3),
    ([1, 2, np.inf], [0.5, 0.5], 3),
    ([1, -1, 2], [0.5, 0.5], 3),
    ([1, 1.5, 2], [0.5, 0.5], 3),
    ([0, 0, 0], [0.5, 0.5], 3),
    ([2 ** 31, 2 ** 31, 0], [0.5, 0.5], 3),
    ([1, 2, 3], [0.5, 0.2, 0.3], 3),
    ([1, 2, 3], [0.5, np.nan], 3),
    ([1, 2, 3], [0.0, 0.0], 3),
    ([1, 2, 3], [0.5, 0.5], 0),
])
def test_validation_errors(weights, props, n_boot):
    mat = np.log(np.full((3, 2), 0.5))
    with pytest.raises(ValueError):
        bootstrap.bootstrap_props(mat, np.asarray(weights, dtype=np.float64), make_args(),
                                  np.asarray(props), n_boot=n_boot, seed=1)


def test_rows_mode_is_rejected():
    mat = np.log(np.full((3, 2), 0.5))
    with pytest.raises(ValueError):
        bootstrap.bootstrap_props(mat, np.ones(3), make_args(b200_shard="rows"),
                                  np.array([0.5, 0.5]), n_boot=2, seed=1)


def boot_slots(n_cls, n_rows, num_sms=148, per_slot=7e6, free=170e9):
    n_cls = np.ascontiguousarray(n_cls, dtype=np.int32)
    r = ctypes.c_int32()
    check(lib.mxb_boot_slots(ctypes.c_void_p(n_cls.ctypes.data), len(n_cls), n_rows, num_sms,
                             per_slot, free, ctypes.byref(r)))
    return r.value


@pytest.mark.parametrize("n_rows,median", [(5787, 135), (1250000, 135)])
def test_slot_rule_plans(n_rows, median):
    """Config-1 size (5787 signature rows) and a config-3 shard: R is a power of two up to 16,
    and the plan for 148 / R CTAs passes the plan checks of test_tile_plan."""
    rs = np.random.RandomState(3)
    nb = (n_rows + 127) // 128
    n_cls = np.minimum(5408, np.maximum(20, rs.lognormal(np.log(median), 0.9, size=nb))).astype(int)
    r = boot_slots(n_cls, n_rows)
    assert r in (1, 2, 4, 8, 16)
    check_plan(n_cls, n_rows, num_sms=148 // r)
    # the slot buffers take at most an eighth of the free memory
    assert boot_slots(n_cls, n_rows, per_slot=7e6, free=8 * 7e6 * 2) <= 2
    assert boot_slots(n_cls, n_rows, per_slot=7e6, free=1e6) == 1


def test_slot_rule_prefers_slots_on_a_small_matrix():
    """46 batches cannot fill 148 CTAs of the pass: the slots share the SMs at no cost."""
    n_cls = np.full(46, 135)
    assert boot_slots(n_cls, 46 * 128 - 5) == 16


def free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def gloo_allreduce(arr, op):
    t = torch.from_numpy(arr)
    dist.all_reduce(t, op=dist.ReduceOp.MAX if op == "max" else dist.ReduceOp.SUM)
    return arr


def _replicates(n_boot, h=7):
    """What one rank running all replicates holds: log-proportions with -inf cells."""
    rs = np.random.RandomState(n_boot)
    lnp = np.log(rs.dirichlet(np.ones(h), size=n_boot))
    lnp[:, 2] = -np.inf
    lnp[::3, 4] = -np.inf
    return lnp, rs.randint(1, 1000, size=n_boot), rs.randint(0, 2, size=n_boot)


N_BOOTS = (1, 2, 5, 40)


def _worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        res = {}
        for n_boot in N_BOOTS:
            lnp, iters, conv = _replicates(n_boot)
            mine = sharding.restart_shard(n_boot, rank, world)
            boot0 = mine[0] if mine else 0
            res[n_boot] = sharding.merge_bootstrap(lnp[mine], iters[mine], conv[mine], boot0,
                                                   n_boot, gloo_allreduce)
        out[rank] = res
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_fan_out_merge_equals_one_rank(world):
    mgr = mp.get_context("spawn").Manager()
    out = mgr.dict()
    mp.spawn(_worker, args=(world, free_port(), out), nprocs=world, join=True)
    res = dict(out)
    mgr.shutdown()
    for n_boot in N_BOOTS:
        lnp, iters, conv = _replicates(n_boot)
        for rank in range(world):
            got_lnp, got_it, got_cv = res[rank][n_boot]
            assert np.array_equal(got_lnp, lnp)
            assert np.array_equal(got_it, iters) and np.array_equal(got_cv, conv)
