"""The best-fit block pool behind a context's device memory and the pinned result pool
(csrc/block_pool.h), compiled with g++ against a counting fake allocator: reuse within the
slack and not beyond it, the cache limit and minimum size, take-only-from-cache, unknown
pointers, trim, a failing allocator, and the live / cached byte counts after every step."""
import ctypes
import os
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

HARNESS = r"""
#include <stdint.h>
#include <stdlib.h>
#include "block_pool.h"

static int64_t g_allocs = 0, g_releases = 0, g_fail = 0, g_synced = 0;
static mxb::BlockPool *g_pool = nullptr;

extern "C" {
void pool_new(size_t slack_div, size_t min_cached, size_t limit) {
    delete g_pool;
    g_allocs = g_releases = g_fail = g_synced = 0;
    g_pool = new mxb::BlockPool(
        [](size_t bytes) -> void * {
            if (g_fail) return nullptr;
            ++g_allocs;
            return malloc(bytes);
        },
        [](void *p) { ++g_releases; free(p); }, slack_div, min_cached, limit);
}
void *pool_take(size_t bytes, int only_cached) { return g_pool->take(bytes, only_cached != 0); }
int pool_give(void *p) { return g_pool->give(p, []() { ++g_synced; }) ? 1 : 0; }
void pool_trim(void) { g_pool->trim(); }
void pool_stats(int64_t *out) {
    size_t live = 0, cached = 0;
    g_pool->stats(&live, &cached);
    out[0] = (int64_t)live; out[1] = (int64_t)cached;
    out[2] = g_allocs; out[3] = g_releases; out[4] = g_synced;
}
void pool_fail(int on) { g_fail = on; }
}
"""


@pytest.fixture(scope="module")
def pool(tmp_path_factory):
    gxx = shutil.which("g++")
    if gxx is None:
        pytest.skip("g++ not available")
    d = tmp_path_factory.mktemp("block_pool")
    src, so = d / "harness.cpp", d / "libpool.so"
    src.write_text(HARNESS)
    subprocess.check_call([gxx, "-std=c++17", "-O1", "-Wall", "-Werror", "-fPIC", "-shared",
                           "-I" + os.path.join(ROOT, "mixemt_b200", "csrc"), str(src), "-o", str(so)])
    lib = ctypes.CDLL(str(so))
    lib.pool_new.argtypes = [ctypes.c_size_t] * 3
    lib.pool_take.restype = ctypes.c_void_p
    lib.pool_take.argtypes = [ctypes.c_size_t, ctypes.c_int]
    lib.pool_give.argtypes = [ctypes.c_void_p]
    lib.pool_stats.argtypes = [ctypes.POINTER(ctypes.c_int64)]
    return lib


def stats(lib):
    """(live bytes, cached bytes, underlying allocations, releases, syncs before caching)"""
    out = (ctypes.c_int64 * 5)()
    lib.pool_stats(out)
    return tuple(out)


MiB = 1 << 20


def test_best_fit_within_slack(pool):
    pool.pool_new(8, MiB, 1 << 40)
    blocks = {sz: pool.pool_take(sz, 0) for sz in (8 * MiB, 9 * MiB, 16 * MiB)}
    assert stats(pool) == (33 * MiB, 0, 3, 0, 0)
    for p in blocks.values():
        assert pool.pool_give(p) == 1
    assert stats(pool) == (0, 33 * MiB, 3, 0, 3)
    # 8.5 MiB: 9 MiB wastes 0.5 <= 8.5/8, 16 MiB would waste too much; the smallest fit wins
    p = pool.pool_take(8 * MiB + MiB // 2, 0)
    assert p == blocks[9 * MiB]
    assert stats(pool) == (9 * MiB, 24 * MiB, 3, 0, 3)
    # 8 MiB exactly: the 8 MiB block, not the (also fitting) larger ones
    q = pool.pool_take(8 * MiB, 0)
    assert q == blocks[8 * MiB]
    # 14 MiB: 16 MiB wastes 2 > 14/8 = 1.75: no reuse, a new block
    r = pool.pool_take(14 * MiB, 0)
    assert r not in blocks.values()
    assert stats(pool) == (31 * MiB, 16 * MiB, 4, 0, 3)
    # the same request with slack 1/4 (the pinned pool) reuses the 16 MiB block
    pool.pool_new(4, 0, 1 << 40)
    a = pool.pool_take(16 * MiB, 0)
    pool.pool_give(a)
    assert pool.pool_take(14 * MiB, 0) == a
    assert stats(pool)[:3] == (16 * MiB, 0, 1)


def test_limit_and_minimum_size(pool):
    pool.pool_new(8, MiB, 3 * MiB)
    small = pool.pool_take(MiB - 1, 0)
    a, b = pool.pool_take(2 * MiB, 0), pool.pool_take(2 * MiB, 0)
    assert stats(pool) == (5 * MiB - 1, 0, 3, 0, 0)
    pool.pool_give(small)          # below the minimum: released, no sync
    assert stats(pool) == (4 * MiB, 0, 3, 1, 0)
    pool.pool_give(a)              # cached (sync first)
    assert stats(pool) == (2 * MiB, 2 * MiB, 3, 1, 1)
    pool.pool_give(b)              # 4 MiB would pass the 3 MiB limit: released, no sync
    assert stats(pool) == (0, 2 * MiB, 3, 2, 1)
    # a request below the minimum never takes a cached block
    pool.pool_new(8, MiB, 1 << 40)
    big = pool.pool_take(MiB, 0)
    pool.pool_give(big)
    c = pool.pool_take(MiB - 8, 0)
    assert c != big and stats(pool) == (MiB - 8, MiB, 2, 0, 1)
    # limit 0 caches nothing
    pool.pool_new(8, MiB, 0)
    pool.pool_give(pool.pool_take(4 * MiB, 0))
    assert stats(pool) == (0, 0, 1, 1, 0)


def test_only_cached_unknown_pointers_and_trim(pool):
    pool.pool_new(4, 0, 1 << 40)
    assert pool.pool_take(4096, 1) is None           # nothing cached: no allocation either
    assert stats(pool) == (0, 0, 0, 0, 0)
    a = pool.pool_take(4096, 0)
    pool.pool_give(a)
    assert pool.pool_take(4000, 1) == a
    assert stats(pool) == (4096, 0, 1, 0, 1)
    assert pool.pool_give(ctypes.c_void_p(a + 16)) == 0   # not a block of the pool
    assert stats(pool) == (4096, 0, 1, 0, 1)
    assert pool.pool_give(a) == 1
    assert pool.pool_give(a) == 0                          # given back twice
    assert pool.pool_take(0, 0) is None
    b = pool.pool_take(100, 0)
    pool.pool_give(b)
    assert stats(pool) == (0, 4196, 2, 0, 3)
    pool.pool_trim()
    assert stats(pool) == (0, 0, 2, 2, 3)
    assert pool.pool_take(4096, 1) is None


def test_failing_allocator_leaves_no_record(pool):
    pool.pool_new(8, MiB, 1 << 40)
    a = pool.pool_take(2 * MiB, 0)
    pool.pool_give(a)
    pool.pool_fail(1)
    assert pool.pool_take(8 * MiB, 0) is None              # no fit in the cache, allocator fails
    assert stats(pool) == (0, 2 * MiB, 1, 0, 1)
    assert pool.pool_take(2 * MiB, 0) == a                 # the cache still serves
    pool.pool_fail(0)
    pool.pool_give(a)
    pool.pool_trim()
    assert stats(pool) == (0, 0, 1, 1, 2)
