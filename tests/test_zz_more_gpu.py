"""Further GPU tests: accum path, edge-share hand-back, advisor regressions
(bitmap tail bits of fill(), storage of w on a hand-back), and the hub-cached
pull SpMV forced onto the small graphs of the parity suite."""
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle_binding as orc
from test_parity_gpu import make_matrix, ragged_graph

pytestmark = [pytest.mark.gpu]

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def gb():
    import graphblast_b200 as g
    g.init(0)
    return g


@pytest.mark.parametrize("name", ["PlusMultiplies", "MinimumPlus", "MaximumMultiplies"])
def test_pull_accum_combines_with_the_semiring_add(gb, name):
    """reference spmv.hpp:213-219: with an accumulator the pull result is combined
    into the old w with the SEMIRING's add (the accum functor itself is ignored)."""
    rp, ci = ragged_graph()
    n = len(rp) - 1
    rng = np.random.RandomState(5)
    val = (2.0 ** rng.randint(0, 3, len(ci))).astype(np.float32)
    A = make_matrix(gb, rp, ci, val, symmetric=False)
    sem = getattr(gb.Semiring, name)
    u_h = (2.0 ** rng.randint(0, 2, n)).astype(np.float32)
    w_old = (2.0 ** rng.randint(0, 4, n)).astype(np.float32)
    desc = gb.Descriptor(mxvmode=2)
    u = gb.Vector(n)
    u.build(u_h)
    w = gb.Vector(n)
    w.build(w_old)
    gb.vxm(w, None, "accum", sem, u, A, desc)
    res, _ = orc.vxm(int(sem), rp, ci, val, u_h)
    add = {"PlusMultiplies": np.add, "MinimumPlus": np.minimum,
           "MaximumMultiplies": np.maximum}[name]
    assert np.array_equal(w.extractTuples(), add(w_old, res))


def test_edge_share_check_does_not_change_results(gb):
    """GrB_PUSHPULL may hand a push back to the pull direction when the frontier
    owns more than a third of the stored entries (spmspv.hpp); a star graph whose
    hub is in a 4096+-entry frontier forces exactly that, and the result must equal
    the oracle's (and the forced-push result)."""
    n = 20000
    hub = 0
    src = np.zeros(n - 1, dtype=np.int32) + hub
    dst = np.arange(1, n, dtype=np.int32)
    rp, ci = orc.build_csr(n, src, dst, True)
    A = make_matrix(gb, rp, ci)
    sem = gb.Semiring.LogicalOrAnd
    f_ind = np.arange(0, 5000, dtype=np.int32)            # contains the hub
    f_val = np.ones(len(f_ind), dtype=np.float32)
    out = {}
    for mode in (0, 1):                                   # automatic, forced push
        desc = gb.Descriptor(mxvmode=mode, switchpoint=0.9)
        u = gb.Vector(n)
        u.build(f_ind, f_val)
        w = gb.Vector(n)
        gb.vxm(w, None, None, sem, u, A, desc)
        out[mode] = (w.extractTuples() != 0)
        if mode == 0:
            assert desc.lastmxv == gb.Desc_value.GrB_PULLONLY
        else:
            assert desc.lastmxv == gb.Desc_value.GrB_PUSHONLY
    up = np.zeros(n, np.uint8)
    uu = np.zeros(n, np.float32)
    up[f_ind] = 1
    uu[f_ind] = 1
    val = np.ones(len(ci), dtype=np.float32)
    want, wp = orc.vxm(int(sem), rp, ci, val, uu, u_present=up)
    assert np.array_equal(out[0], want != 0)
    assert np.array_equal(out[1], want != 0)


@pytest.mark.parametrize("name", ["PlusMultiplies", "MinimumPlus"])
def test_generic_pull_spmv_is_bit_reproducible(gb, name):
    """The generic pull SpMV on fresh matrices built from the same entries gives
    the same result to the bit (random float values on purpose): the products and
    the order they are added in depend on the structure only."""
    rp, ci = orc.rmat_csr(12)
    n = len(rp) - 1
    rng = np.random.RandomState(9)
    val = rng.rand(len(ci)).astype(np.float32) + 0.5
    u_h = rng.rand(n).astype(np.float32) + 0.5
    sem = getattr(gb.Semiring, name)
    out = []
    for _ in range(3):
        A = make_matrix(gb, rp, ci, val, symmetric=False)
        desc = gb.Descriptor(mxvmode=2)
        u = gb.Vector(n)
        u.build(u_h)
        w = gb.Vector(n)
        gb.vxm(w, None, None, sem, u, A, desc)
        gb.vxm(w, None, None, sem, u, A, desc)
        out.append(w.extractTuples().copy())
    assert np.array_equal(out[0].view(np.uint32), out[1].view(np.uint32))
    assert np.array_equal(out[0].view(np.uint32), out[2].view(np.uint32))


@pytest.mark.parametrize("n", [11, 33, 64, 1000])
def test_fill_then_push_when_size_is_not_a_multiple_of_32(gb, n):
    """fill(1) builds the bitmap shadow; the bits past n in the last word must stay
    clear, otherwise dense2sparse emits indices >= n (r01 advisor finding)."""
    rng = np.random.RandomState(n)
    src = rng.randint(0, n, 4*n).astype(np.int32)
    dst = rng.randint(0, n, 4*n).astype(np.int32)
    rp, ci = orc.build_csr(n, src, dst, True)
    A = make_matrix(gb, rp, ci)
    for sem in (gb.Semiring.PlusMultiplies, gb.Semiring.LogicalOrAnd):
        u = gb.Vector(n)
        u.fill(1.0)
        w = gb.Vector(n)
        gb.vxm(w, None, None, sem, u, A, gb.Descriptor(mxvmode=1))   # push only
        want, _ = orc.vxm(int(sem), rp, ci, np.ones(len(ci), np.float32),
                          np.ones(n, np.float32))
        got = w.extractTuples()
        assert got.shape[0] == n
        assert np.array_equal(got, want)
    u = gb.Vector(n)
    u.fill(1.0)
    import ctypes as C
    import torch
    from graphblast_b200 import _lib
    d_bits = torch.zeros((n + 31)//32 + 1, dtype=torch.int32, device="cuda")
    count = C.c_longlong(-1)
    assert _lib.load().gb200_vector_export_bits(
        u._h, C.c_void_p(d_bits.data_ptr()), C.byref(count)) == 0
    assert count.value == n
    words = d_bits.cpu().numpy().view(np.uint32)[:(n + 31)//32]
    assert int(np.unpackbits(words.view(np.uint8)).sum()) == n


def _run_parity_subset_with_hub_forced(kexpr):
    env = dict(os.environ)
    env.update(GB200_SPMV_HUB="1", GB200_SPMV_HUB_MIN_NNZ="0",
               GB200_SPMV_HUB_MIN_PCT="0")
    cmd = [sys.executable, "-m", "pytest", "-x", "-q", "-m", "gpu",
           os.path.join(ROOT, "tests", "test_parity_gpu.py"), "-k", kexpr]
    r = subprocess.run(cmd, env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT,
                       text=True, timeout=1500)
    assert r.returncode == 0, r.stdout[-4000:]
    assert " passed" in r.stdout


def test_hub_spmv_on_the_parity_suite_semirings():
    """Every generic pull of the semiring sweep / gvxm cases through the hub-cached
    kernel (kernels/spmv_hub.cuh): thresholds lowered so the small graphs take it."""
    _run_parity_subset_with_hub_forced("semiring_sweep or gvxm or mxv_matches")


def test_hub_spmv_on_the_parity_suite_algorithms():
    _run_parity_subset_with_hub_forced("sssp or pagerank")


@pytest.mark.parametrize("scale", [14, 16, 18, 20])
def test_triangle_count_matches_the_committed_reference_counts(gb, scale):
    """tests/golden/tc_golden.json holds the counts the reference's own CPU code
    (SimpleReferenceTc, reference test_tc.hpp:15-85) produced for the R-MAT bench
    graphs; the masked mxm must reproduce them exactly, through the library's own
    tril (reference gtc.cu:76-82)."""
    import json
    import torch
    from graphblast_b200 import algorithm, graphs
    table = json.load(open(os.path.join(ROOT, "tests", "golden", "tc_golden.json")))
    g = table["rmat%d" % scale]
    n = 1 << scale
    src, dst = graphs.rmat_edges(scale, 16, seed=1)
    rowptr, colind = graphs.build_csr(n, src, dst, undirected=True)
    assert int(colind.numel()) == g["nnz"]
    h_ci = colind.cpu().numpy()
    check = int(np.sum(h_ci.astype(np.int64) *
                       (np.arange(len(h_ci), dtype=np.int64) % 97 + 1)))
    assert check == g["colind_checksum"]
    desc = gb.Descriptor(mxvmode=0)
    A = graphs.matrix_from_csr(n, rowptr, colind, dtype=gb.api.INT32, symmetric=True)
    A.tril(desc)
    assert A.nvals() == g["nnz_tril"]
    B = gb.Matrix(n, n, dtype=gb.api.INT32)
    ntris, _ = algorithm.tc(A, B, desc)
    assert int(ntris) == g["triangles_tril"]
    del A, B
    torch.cuda.empty_cache()


def test_scatter_assign_scatter_extract_gather(gb):
    """The index-driven operations of the label-propagation consumers (reference
    graphblas/operations.hpp:771-860, kernels/scatter.hpp:8-50, kernels/gather.hpp:9-35)
    through the C ABI, against their definitions."""
    from graphblast_b200 import _lib
    lib = _lib.load()
    n = 1000
    rng = np.random.RandomState(3)
    desc = gb.Descriptor(mxvmode=0)
    perm = rng.permutation(n).astype(np.float32)
    vals = rng.randint(1, 100, n).astype(np.float32)
    u = gb.Vector(n); u.build(vals)
    ind = gb.Vector(n); ind.build(perm)
    # assignScatter: w[ind[i]] = u[i]
    w = gb.Vector(n); w.fill(-1.0)
    assert lib.gb200_assign_scatter(w._h, u._h, ind._h, desc._h) == 0
    want = np.full(n, -1.0, np.float32)
    want[perm.astype(np.int64)] = vals
    assert np.array_equal(w.extractTuples(), want)
    # extractGather: w[i] = u[ind[i]]
    g = gb.Vector(n); g.fill(-1.0)
    assert lib.gb200_extract_gather(g._h, u._h, ind._h, desc._h) == 0
    assert np.array_equal(g.extractTuples(), vals[perm.astype(np.int64)])
    # the two are inverse to each other on a permutation
    back = gb.Vector(n); back.fill(-1.0)
    assert lib.gb200_assign_scatter(back._h, g._h, ind._h, desc._h) == 0
    assert np.array_equal(back.extractTuples(), vals)
    # scatter: w[(int)u[i]] = val for targets in (0, len(u)); target 0 is skipped
    targets = np.array([0, 5, 5, 17, n - 1, n + 3, 250], dtype=np.float32)
    t = gb.Vector(len(targets)); t.build(targets)
    s = gb.Vector(n); s.fill(0.0)
    assert lib.gb200_scatter(s._h, t._h, 7.0, desc._h) == 0
    want = np.zeros(n, np.float32)
    # the dense form bounds targets by the length of u (reference scatter.hpp:44)
    for x in targets:
        if 0 < int(x) < len(targets):
            want[int(x)] = 7.0
    assert np.array_equal(s.extractTuples(), want)
