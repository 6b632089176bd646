"""Fragment -> signature reduction (csrc/reduce.cpp, SURVEY.md 8f N1) against the
reference's reduce_reads / build_em_input ordering.  Host code: runs without a GPU."""
import numpy as np
import pytest

from mixemt_b200 import preprocess as pre
from oracle import live_cases, oracle_np, refload
from conftest import load_golden


@pytest.mark.parametrize("seed", [81, 82])
def test_reduce_reads_golden(seed):
    g = load_golden("golden_reduce.npz")
    read_obs = oracle_np.synthetic_read_obs(seed)
    want_first = str(g["s%d_first_order" % seed]).split("\n")
    want_sorted = str(g["s%d_sorted" % seed]).split("\n")
    # the oracle restatement is pinned to the reference's output ...
    ora = oracle_np.reduce_reads(read_obs)
    assert list(ora) == want_first and sorted(ora) == want_sorted
    # ... and so are the drop-in and the array form
    got = pre.reduce_reads(read_obs)
    assert list(got) == want_first
    assert all(got[s] == ora[s] for s in ora)
    assert got[want_sorted[5]] == str(g["s%d_ids_of_row5" % seed]).split("\n")
    ids, frag_ptr, pos, base = pre.flatten_read_obs(read_obs)
    red = pre.reduce_reads_arrays(frag_ptr, pos, base)
    assert red.signatures == want_sorted
    assert np.array_equal(red.weights, g["s%d_weights" % seed])
    assert "" in want_sorted and want_sorted[0] == ""          # empty fragments sort first
    # rows map back to their fragments
    for row, frags in enumerate(red.fragments_of_rows()):
        assert [ids[f] for f in frags.tolist()] == ora[want_sorted[row]]
        assert (red.sig_of_frag[frags] == row).all()
    assert np.array_equal(np.sort(red.frag_order), np.arange(len(ids)))


def test_string_order_is_not_numeric_order():
    # SURVEY.md F9: '100:C,200:T' < '10:A' < '9:A'
    frag_ptr = np.array([0, 1, 2, 4, 5])
    pos = np.array([9, 10, 100, 200, 9], dtype=np.int32)
    red = pre.reduce_reads_arrays(frag_ptr, pos, b"AACTA")
    assert red.signatures == ["100:C,200:T", "10:A", "9:A"]
    assert red.weights.tolist() == [1, 1, 2]
    assert red.sig_of_frag.tolist() == [2, 1, 0, 2]
    assert red.first_frag.tolist() == [2, 1, 0]


def test_edge_inputs():
    red = pre.reduce_reads_arrays(np.zeros(1, dtype=np.int64), np.zeros(0, dtype=np.int32), b"")
    assert red.n_rows == 0 and red.signatures == []
    red = pre.reduce_reads_arrays(np.zeros(4, dtype=np.int64), np.zeros(0, dtype=np.int32), b"")
    assert red.signatures == [""] and red.weights.tolist() == [3]
    with pytest.raises(ValueError):
        pre.reduce_reads_arrays(np.array([0, 2]), np.array([1], dtype=np.int32), b"A")
    assert pre.reduce_reads({}) == {}
    # multi-character observations keep the reference's formatting
    odd = {"a": {5: "AC", 3: "g"}, "b": {3: "g", 5: "AC"}}
    assert pre.reduce_reads(odd) == {"3:g,5:AC": ["a", "b"]}


def test_million_fragments_are_reduced_in_seconds():
    rs = np.random.RandomState(3)
    n = 1000000
    start = rs.randint(0, 4000, size=n)
    length = rs.randint(1, 60, size=n)
    frag_ptr = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(length, out=frag_ptr[1:])
    pos = (np.repeat(start - frag_ptr[:-1], length) + np.arange(frag_ptr[-1])).astype(np.int32) * 4
    base = np.frombuffer(b"ACGT", dtype=np.uint8)[(pos // 4 + (rs.rand(len(pos)) < 0.001)) % 4]
    import time
    t0 = time.perf_counter()
    red = pre.reduce_reads_arrays(frag_ptr, pos, base)
    dt = time.perf_counter() - t0
    assert red.weights.sum() == n and red.n_rows < n
    key = {}
    for f in rs.choice(n, size=2000, replace=False).tolist():      # spot check the grouping
        sig = (pos[frag_ptr[f]:frag_ptr[f + 1]].tobytes(), base[frag_ptr[f]:frag_ptr[f + 1]].tobytes())
        assert key.setdefault(sig, red.sig_of_frag[f]) == red.sig_of_frag[f]
    sigs = red.signatures
    assert all(sigs[i] < sigs[i + 1] for i in range(0, len(sigs) - 1, 97))
    assert dt < 60.0, dt


def test_reduce_reads_live_reference():
    """The drop-in reduce_reads against the reference's on 1500 seeded fragments
    (tests/golden/golden_live.npz); where the reference is installed, the stored
    output against the reference itself."""
    g = live_cases.load_golden()
    read_obs = live_cases.reduce_case()
    want = (str(g["r_sigs"]), str(g["r_ids"]))
    if refload.available():
        _, ref_pre, _ = refload.load()
        assert live_cases.encode_read_sigs(ref_pre.reduce_reads(read_obs)) == want
    assert live_cases.encode_read_sigs(pre.reduce_reads(read_obs)) == want


def test_fuzz_against_python_restatement():
    """Random small fragment sets (shared positions, empty fragments, multi-digit positions that
    sort differently as strings): the drop-in dict and the array form agree with the reference's
    loop (preprocess.py:163-174) and its sorted() order (:219-220)."""
    import random
    from mixemt_b200.preprocess import flatten_read_obs, reduce_reads, reduce_reads_arrays
    rnd = random.Random(3)
    for _ in range(400):
        pool = [rnd.randint(0, 16568) for _ in range(rnd.randint(1, 8))]
        read_obs = {}
        for f in range(rnd.randint(0, 60)):
            obs = {}
            for _ in range(rnd.randint(0, 6)):
                obs[rnd.choice(pool)] = rnd.choice("ACGTN")
            read_obs["r%d" % f] = obs
        want = {}
        for rid, obs in read_obs.items():
            sig = ','.join("%d:%s" % (p, obs[p]) for p in sorted(obs))
            want.setdefault(sig, []).append(rid)
        assert list(reduce_reads(read_obs).items()) == list(want.items())
        ids, frag_ptr, pos, base = flatten_read_obs(read_obs)
        red = reduce_reads_arrays(frag_ptr, pos, base)
        order = sorted(want)
        assert red.signatures == order
        assert red.weights.tolist() == [len(want[s]) for s in order]
