"""The matrix-build kernels (csrc/build.cu) on every case of build_cases.py: cells bit for bit and
match counts equal to the C oracle, and the route each row took equal to the restated routing,
with and without counts (another instantiation of the class kernel) and under the three
cross-check settings of mxb_build_matrix."""
import numpy as np
import pytest

import build_cases as bc
from mixemt_b200 import synth
from mixemt_b200.preprocess import HapVarBaseMatrix, build_matrix_from_csr
from oracle import oracle_c

pytestmark = pytest.mark.gpu

_ORACLE = {}


def _oracle(c):
    if c.name not in _ORACLE:
        _ORACLE[c.name] = oracle_c.build_matrix(c.tables, c.csr)
    return _ORACLE[c.name]


def _build(tables, csr, counts):
    routes = np.full(csr.n_rows, -1, dtype=np.int32)
    mat, cnt, _, _ = build_matrix_from_csr(tables, csr, want_counts=counts, routes_out=routes)
    return mat, cnt, routes


def _check(tables, csr, counts, want_routes, o_mat, o_cnt, what):
    mat, cnt, routes = _build(tables, csr, counts)
    assert np.array_equal(mat.view(np.uint64), o_mat.view(np.uint64)), \
        (what, np.argwhere(mat.view(np.uint64) != o_mat.view(np.uint64))[:5])
    if counts:
        assert np.array_equal(cnt, o_cnt), what
    assert np.array_equal(routes, want_routes), (what, routes, want_routes)


@pytest.mark.parametrize("counts", [True, False])
@pytest.mark.parametrize("name", bc.CASE_NAMES)
def test_case_bit_exact_on_every_route(name, counts, monkeypatch):
    c = bc.case(name)
    o_mat, o_cnt = _oracle(c)
    _check(c.tables, c.csr, counts, bc.predict_routes(c.tables, c.csr), o_mat, o_cnt, "default")
    # every row through the large-pool launch
    monkeypatch.setenv("MXB_BUILD_TIERS", "2")
    _check(c.tables, c.csr, counts, bc.predict_routes(c.tables, c.csr, two_tiers=False),
           o_mat, o_cnt, "MXB_BUILD_TIERS=2")
    monkeypatch.delenv("MXB_BUILD_TIERS")
    # deviation lists against the marker-free baseline (read when the tables are packed)
    monkeypatch.setenv("MXB_BUILD_BASE_REF", "1")
    ref_tables = bc.repacked(c.tables)
    ref_tables.to_device()
    monkeypatch.delenv("MXB_BUILD_BASE_REF")
    _check(ref_tables, c.csr, counts, bc.predict_routes(c.tables, c.csr, base_ref=True),
           o_mat, o_cnt, "MXB_BUILD_BASE_REF=1")
    # the plain dense kernel
    monkeypatch.setenv("MXB_BUILD_DENSE", "1")
    _check(c.tables, c.csr, counts, np.full(c.csr.n_rows, bc.DENSE_KERNEL, np.int32),
           o_mat, o_cnt, "MXB_BUILD_DENSE=1")


def test_routes_out_is_optional_and_checked():
    c = bc.case("pool_146_147_warp0")
    o_mat, _ = _oracle(c)
    mat, _, _, _ = build_matrix_from_csr(c.tables, c.csr)
    assert np.array_equal(mat.view(np.uint64), o_mat.view(np.uint64))
    with pytest.raises(ValueError):
        build_matrix_from_csr(c.tables, c.csr, routes_out=np.zeros(c.csr.n_rows, np.int64))


def test_build17_mixture_routes(phylo17):
    """Four sources, 4 % sequencing errors: every row takes the route the restated routing
    predicts, and the real rows reach both tiers of the class kernel."""
    haps = sorted(phylo17.hap_var)
    mix = synth.make_mixture(phylo17, phylo17.refseq,
                             [("H1", 0.4), ("L3e", 0.3), ("U5a1", 0.2), ("M7", 0.1)], 2000,
                             err=0.04, seed=21)
    tables = HapVarBaseMatrix(phylo17.refseq, phylo17, haps).pack()
    csr = mix.csr(tables)
    want = bc.predict_routes(tables, csr)
    o_mat, o_cnt = oracle_c.build_matrix(tables, csr)
    for counts in (True, False):
        _check(tables, csr, counts, want, o_mat, o_cnt, "build 17")
    paths = np.bincount(want % 4, minlength=4)
    assert paths[0] > 0 and paths[1] > 0, paths
