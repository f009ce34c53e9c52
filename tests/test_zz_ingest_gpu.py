"""Device ingest (SURVEY.md §8 f1): the library's own radix sort, tuples -> CSR with
the reference loader's semantics, CSR -> CSC, and the Matrix Market path, against
numpy, the oracle and the reference's own loader (oracle/_ref, stored results)."""
import ctypes as C
import os

import numpy as np
import pytest

import oracle_binding as orc

pytestmark = [pytest.mark.gpu]

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")


@pytest.fixture(scope="module")
def gb():
    import graphblast_b200 as g
    g.init(0)
    return g


@pytest.mark.parametrize("n,bits", [(1, 8), (2, 16), (100, 24), (2048, 8), (2049, 40),
                                    (5000, 48), (300000, 33), (1 << 20, 48)])
def test_radix_sort_is_a_stable_sort_of_the_low_bits(gb, n, bits):
    import torch
    from graphblast_b200 import _lib
    rng = np.random.RandomState(n + bits)
    keys = rng.randint(0, 1 << 62, n, dtype=np.int64).astype(np.uint64)
    if n > 10:
        keys[rng.randint(0, n, n // 3)] = keys[0]          # plenty of duplicates
    low = keys & np.uint64((1 << bits) - 1)
    pay = np.arange(n, dtype=np.uint32)
    d_k = torch.from_numpy(keys.view(np.int64)).cuda()
    d_p = torch.from_numpy(pay.view(np.int32)).cuda()
    rc = _lib.load().gb200_sort_pairs_u64(C.c_void_p(d_k.data_ptr()),
                                          C.c_void_p(d_p.data_ptr()), n, bits)
    assert rc == 0
    order = np.argsort(low, kind="stable")
    got_k = d_k.cpu().numpy().view(np.uint64)
    got_p = d_p.cpu().numpy().view(np.uint32)
    assert np.array_equal(got_p, pay[order])
    assert np.array_equal(got_k, keys[order])


@pytest.mark.parametrize("scale", [6, 12, 16])
def test_ingest_matches_the_oracle_loader(gb, scale):
    from graphblast_b200 import graphs
    src, dst = graphs.rmat_edges(scale, 16, seed=1)
    osrc, odst = orc.rmat_edges(scale, 16, 1)
    for undirected in (True, False):
        rp, ci = graphs.build_csr(1 << scale, src, dst, undirected=undirected)
        orp, oci = orc.build_csr(1 << scale, osrc, odst, undirected)
        assert np.array_equal(rp.cpu().numpy(), orp)
        assert np.array_equal(ci.cpu().numpy(), oci)


def test_ingest_edge_cases(gb):
    import torch
    from graphblast_b200 import graphs
    n = 9
    # duplicates with different values: the first tuple in input order wins, and a
    # forward tuple beats a reverse copy of an earlier tuple (reference appends the
    # reverse copies after all forward tuples, util.hpp:271-279)
    src = torch.tensor([3, 5, 3, 7, 7, 2], dtype=torch.int32, device="cuda")
    dst = torch.tensor([5, 3, 5, 7, 1, 8], dtype=torch.int32, device="cuda")
    val = torch.tensor([10., 20., 30., 40., 50., 60.], device="cuda")
    rp, ci, v = graphs.build_csr(n, src, dst, undirected=True, val=val,
                                 return_values=True)
    rp, ci, v = rp.cpu().numpy(), ci.cpu().numpy(), v.cpu().numpy()
    dense = np.zeros((n, n), dtype=np.float32)
    for r in range(n):
        dense[r, ci[rp[r]:rp[r + 1]]] = v[rp[r]:rp[r + 1]]
    want = np.zeros((n, n), dtype=np.float32)
    want[3, 5] = 10.      # forward (3,5)=10 first; reverse of (5,3)=20 comes later
    want[5, 3] = 20.      # forward (5,3)=20 beats reverse of (3,5)
    want[7, 1] = 50.; want[1, 7] = 50.
    want[2, 8] = 60.; want[8, 2] = 60.
    assert np.array_equal(dense, want)          # (7,7) self-loop dropped
    for r in range(n):
        assert np.all(np.diff(ci[rp[r]:rp[r + 1]]) > 0)
    # no tuples at all
    e = torch.zeros(0, dtype=torch.int32, device="cuda")
    rp, ci = graphs.build_csr(4, e, e, undirected=True)
    assert rp.cpu().tolist() == [0, 0, 0, 0, 0] and ci.numel() == 0
    # everything dropped
    s = torch.tensor([1, 2], dtype=torch.int32, device="cuda")
    rp, ci = graphs.build_csr(4, s, s, undirected=True)
    assert rp.cpu().tolist() == [0, 0, 0, 0, 0] and ci.numel() == 0


def test_csr_transpose_values(gb):
    import torch
    from graphblast_b200 import graphs
    scale = 10
    src, dst = graphs.rmat_edges(scale, 16, seed=1)
    n = 1 << scale
    rp, ci = graphs.build_csr(n, src, dst, undirected=True)
    nnz = ci.numel()
    val = torch.arange(1, nnz + 1, dtype=torch.float32, device="cuda")
    got = graphs.transpose_values(n, rp, ci, val).cpu().numpy()
    h_rp, h_ci = rp.cpu().numpy(), ci.cpu().numpy()
    rows = np.repeat(np.arange(n), np.diff(h_rp))
    order = np.lexsort((rows, h_ci))             # by (col, row): the CSC order
    assert np.array_equal(got, val.cpu().numpy()[order])


@pytest.mark.parametrize("name,directed", [("chesapeake.mtx", 0), ("chesapeake.mtx", 2),
                                           ("test_cc.mtx", 0), ("test_cc.mtx", 2),
                                           ("test_bc.mtx", 0), ("test_bc.mtx", 1),
                                           ("test_bc.mtx", 2)])
def test_matrix_market_path_matches_the_reference_loader(gb, name, directed):
    """gb200_matrix_load_mtx parses on the host and orders / symmetrises / dedups on
    the device; the CSR must be the reference readMtx + coo2csr's (oracle/_ref, as
    stored in tests/golden/ref_cpu.npz by tests/golden/make_golden_ref.py).
    test_sgm.mtx (nothing but self-loops) is left out: the reference's removeSelfloop
    (util.hpp:310-322) reads past the end of its vectors when every tuple is dropped,
    and depending on what the heap holds it returns or dies in vector::resize(-1); the
    all-loops case is covered in test_ingest_edge_cases."""
    path = os.path.join(GOLDEN, name)
    A = gb.Matrix.from_mtx(path, directed=directed)
    rp, ci, val = A.extract_csr()
    key = "mtx_%s_d%d_" % (os.path.splitext(name)[0], directed)
    with np.load(os.path.join(GOLDEN, "ref_cpu.npz")) as ref:
        want_rp, want_ci, want_val = (ref[key + "rowptr"], ref[key + "colind"],
                                      ref[key + "val"])
    assert np.array_equal(rp, want_rp)
    assert np.array_equal(ci, want_ci)
    assert np.array_equal(val, want_val)
