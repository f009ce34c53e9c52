"""CPU tests that PIN the oracle: oracle/gb_oracle.c against
  (1) the committed golden vectors generated from the reference's own CPU code
      (tests/golden/golden.json, tests/golden/make_golden.py),
  (2) the known answers pinned by the reference's tests/fixtures (BASELINE.md §2),
  (3) what the reference's own CPU code (oracle/_ref/libgbref.so) returns on the
      same inputs, stored in tests/golden/ref_cpu.npz
      (tests/golden/make_golden_ref.py).
"""
import json
import os

import numpy as np
import pytest

import oracle_binding as orc

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = json.load(open(os.path.join(HERE, "golden", "golden.json")))
REF_CPU = np.load(os.path.join(HERE, "golden", "ref_cpu.npz"))

CHESAPEAKE_LEVELS = [1, 3, 3, 3, 3, 3, 2, 2, 3, 3, 2, 2, 2, 3, 3, 3, 3, 3, 3, 3,
                     3, 2, 2, 3, 3, 3, 3, 3, 3, 3, 3, 3, 3, 2, 2, 3, 2, 3, 2]


def chesapeake_csr():
    n, src, dst, _ = orc.read_mtx_edges(os.path.join(HERE, "golden",
                                                     "chesapeake.mtx"))
    return orc.build_csr(n, src, dst, True)


def test_loader_matches_reference_csr():
    rp, ci = chesapeake_csr()
    g = GOLDEN["chesapeake"]
    assert len(rp) - 1 == g["n"] == 39 and len(ci) == g["nnz"] == 340
    assert rp.tolist() == g["rowptr"]
    assert ci.tolist() == g["colind"]


def test_loader_directed_and_duplicates():
    # duplicates, a self-loop and an unsorted order; directed keeps orientation
    src = np.array([2, 0, 0, 1, 1, 2, 0], dtype=np.int32)
    dst = np.array([0, 1, 1, 1, 2, 0, 2], dtype=np.int32)
    rp, ci = orc.build_csr(3, src, dst, undirected=False)
    assert rp.tolist() == [0, 2, 3, 4] and ci.tolist() == [1, 2, 2, 0]
    rp, ci = orc.build_csr(3, src, dst, undirected=True)
    assert rp.tolist() == [0, 2, 4, 6] and ci.tolist() == [1, 2, 0, 2, 0, 1]


def test_bfs_known_answer_chesapeake():
    rp, ci = chesapeake_csr()
    lv = orc.bfs(rp, ci, 0)
    assert lv.tolist() == CHESAPEAKE_LEVELS          # BASELINE.md §2
    assert lv.tolist() == GOLDEN["chesapeake"]["bfs_levels_src0"]
    assert lv.max() == 3 and lv.sum() == 104


def test_bfs_stop_depth_and_unreachable():
    # path 0-1-2, isolated 3
    rp = np.array([0, 1, 3, 4, 4], dtype=np.int32)
    ci = np.array([1, 0, 2, 1], dtype=np.int32)
    assert orc.bfs(rp, ci, 0).tolist() == [1, 2, 3, 0]
    assert orc.bfs(rp, ci, 0, stop=2).tolist() == [1, 2, 0, 0]
    assert orc.bfs(rp, ci, 3).tolist() == [0, 0, 0, 1]


def test_sssp_golden_chesapeake():
    g = GOLDEN["chesapeake"]
    rp, ci = chesapeake_csr()
    w = np.array(g["sssp_weights_seed1"], dtype=np.float32)
    d = orc.sssp(rp, ci, w, 0)
    assert d.tolist() == g["sssp_dist_src0"]


def test_sssp_unreachable_is_flt_max():
    rp = np.array([0, 1, 2, 2], dtype=np.int32)
    ci = np.array([1, 0], dtype=np.int32)
    d = orc.sssp(rp, ci, np.array([5, 5], dtype=np.float32), 0)
    assert d[0] == 0 and d[1] == 5 and d[2] == orc.FLT_MAX


def test_pagerank_golden_chesapeake():
    rp, ci = chesapeake_csr()
    p = orc.pr(rp, ci, 0.85, 1e-8, 10)
    want = np.array(GOLDEN["chesapeake"]["pagerank_a085_it10"], dtype=np.float32)
    assert np.array_equal(p, want)
    assert abs(float(p.sum()) - 1.0) < 1e-3


def test_triangles_known_answer_chesapeake():
    rp, ci = chesapeake_csr()
    lr, lc = orc.tril(rp, ci)
    assert orc.tc(lr, lc) == 194 == GOLDEN["chesapeake"]["triangles_tril"]
    assert orc.tc(rp, ci) == 6 * 194                 # SURVEY.md §8c


def test_reduce_rows_known_answer_test_cc():
    g = GOLDEN["test_cc"]
    rp = np.array(g["rowptr"], dtype=np.int32)
    sums = orc.reduce_rows(rp, np.ones(g["nnz"], dtype=np.float32))
    assert sums.tolist() == [1, 1, 3, 2, 2, 3, 3, 0, 1, 2, 2]   # test/greduce.cu:65
    assert sums.tolist() == g["row_sums"]


def test_vxm_plus_multiplies_matches_inline_loop():
    """test/gvxm.cu:41-55: correct[col] += val*vec[row]."""
    g = GOLDEN["test_cc"]
    rp = np.array(g["rowptr"], dtype=np.int32)
    ci = np.array(g["colind"], dtype=np.int32)
    val = np.ones(len(ci), dtype=np.float32)
    u = np.arange(1, g["n"] + 1, dtype=np.float32)
    want = np.zeros(g["n"], dtype=np.float32)
    for r in range(g["n"]):
        for k in range(rp[r], rp[r + 1]):
            want[ci[k]] += val[k] * u[r]
    got, _ = orc.vxm(orc_id("PLUS_MULTIPLIES"), rp, ci, val, u)
    assert np.array_equal(got, want)
    mask = (np.arange(g["n"]) % 3 == 0).astype(np.float32)
    got_m, _ = orc.vxm(orc_id("PLUS_MULTIPLIES"), rp, ci, val, u, mask=mask)
    assert np.array_equal(got_m, np.where(mask != 0, want, 0))
    got_c, _ = orc.vxm(orc_id("PLUS_MULTIPLIES"), rp, ci, val, u, mask=mask,
                       scmp=True)
    assert np.array_equal(got_c, np.where(mask == 0, want, 0))


SEMIRING_IDS = ["LOGICAL_OR_AND", "PLUS_MULTIPLIES", "MINIMUM_PLUS",
                "MAXIMUM_MULTIPLIES", "PLUS_DIVIDES", "PLUS_GREATER",
                "GREATER_PLUS", "PLUS_MINUS", "PLUS_LESS", "CUSTOM_LESS_PLUS",
                "MINIMUM_MULTIPLIES", "MULTIPLIES_MULTIPLIES",
                "NOT_EQUAL_TO_PLUS", "MINIMUM_SELECT_SECOND",
                "PLUS_NOT_EQUAL_TO", "CUSTOM_LESS_LESS", "MINIMUM_NOT_EQUAL_TO"]


def orc_id(name):
    return SEMIRING_IDS.index(name)


def test_semiring_identities():
    """reference graphblas/stddef.hpp:160-173, 194-213."""
    fmax = float(np.finfo(np.float32).max)
    fmin = float(np.finfo(np.float32).tiny)
    want = {"LOGICAL_OR_AND": 0.0, "PLUS_MULTIPLIES": 0.0, "MINIMUM_PLUS": fmax,
            "MAXIMUM_MULTIPLIES": 0.0, "GREATER_PLUS": fmin,
            "CUSTOM_LESS_PLUS": fmax, "MULTIPLIES_MULTIPLIES": 1.0,
            "NOT_EQUAL_TO_PLUS": fmax, "MINIMUM_SELECT_SECOND": fmax}
    for name, ident in want.items():
        assert orc.identity(orc_id(name)) == pytest.approx(ident, rel=0, abs=0)


def test_rmat_generator_golden_and_shape():
    g = GOLDEN["rmat10"]
    rp, ci = orc.rmat_csr(10)
    assert len(rp) - 1 == g["n"] and len(ci) == g["nnz"]
    chk = int(np.sum(ci.astype(np.int64) * (np.arange(len(ci)) % 97 + 1)))
    assert chk == g["colind_checksum"]
    # symmetric, sorted rows, no self loops
    rows = np.repeat(np.arange(g["n"]), np.diff(rp))
    assert not np.any(rows == ci)
    fwd = set(zip(rows.tolist(), ci.tolist()))
    assert all((c, r) in fwd for r, c in list(fwd)[:2000])
    for r in range(0, g["n"], 37):
        seg = ci[rp[r]:rp[r + 1]]
        assert np.all(np.diff(seg) > 0)
    lv = orc.bfs(rp, ci, 0)
    assert np.bincount(lv).tolist() == g["bfs_level_hist_src0"]
    lr, lc = orc.tril(rp, ci)
    assert orc.tc(lr, lc) == g["triangles_tril"]


def test_weight_stream_golden():
    """The reference's SSSP weights come from std::default_random_engine +
    uniform_int_distribution (algorithm/common.hpp:22-42); the product draws the
    same stream in gb200_host_uniform_weights — pinned here without a GPU."""
    import graphblast_b200 as gb
    got = gb.api.host_uniform_weights(1, 1, 64, 64)
    assert got.tolist() == GOLDEN["weights"]["seed1_first64"]
    got7 = gb.api.host_uniform_weights(7, 1, 64, 64)
    assert got7.tolist() == GOLDEN["weights"]["seed7_first64"]
    assert got.min() >= 1 and got.max() <= 64


def colind_checksum(ci):
    return int(np.sum(ci.astype(np.int64) * (np.arange(len(ci), dtype=np.int64) % 97 + 1)))


@pytest.mark.parametrize("scale", [8, 12])
def test_oracle_equals_reference_cpu_on_rmat(scale):
    ref = {k[len("rmat%d_" % scale):]: REF_CPU[k] for k in REF_CPU.files
           if k.startswith("rmat%d_" % scale)}
    rp, ci = orc.rmat_csr(scale)
    assert len(ci) == ref["nnz"] and colind_checksum(ci) == ref["colind_checksum"]
    src = int(np.argmax(np.diff(rp)))
    assert src == ref["source"]
    assert np.array_equal(orc.bfs(rp, ci, src), ref["bfs_source"])
    assert np.array_equal(orc.bfs(rp, ci, 0), ref["bfs_0"])
    w = ref["weights"].astype(np.float32)
    assert np.array_equal(orc.sssp(rp, ci, w, src), ref["sssp_source"])
    assert np.array_equal(orc.pr(rp, ci), ref["pr"])
    lr, lc = orc.tril(rp, ci)
    assert orc.tc(lr, lc) == ref["tc"]


@pytest.mark.parametrize("name,directed", [("chesapeake.mtx", 2),
                                           ("chesapeake.mtx", 0),
                                           ("test_cc.mtx", 0),
                                           ("test_cc.mtx", 2),
                                           ("test_bc.mtx", 0),
                                           ("test_bc.mtx", 2)])
def test_loader_equals_reference_readmtx(name, directed):
    # test_sgm.mtx holds only self-loops; the reference loader itself throws
    # std::length_error on it with the default GRB_UTIL_REMOVE_SELFLOOP=1
    # (util.hpp:307-329), so it is not part of this comparison.
    path = os.path.join(HERE, "golden", name)
    n, src, dst, symmetric = orc.read_mtx_edges(path)
    undirected = (symmetric or directed == 2) and directed != 1
    rp, ci = orc.build_csr(n, src, dst, undirected)
    key = "mtx_%s_d%d_" % (os.path.splitext(name)[0], directed)
    assert np.array_equal(rp, REF_CPU[key + "rowptr"])
    assert np.array_equal(ci, REF_CPU[key + "colind"])


def test_oracle_equals_reference_cpu_on_random_graphs():
    """Property test of the oracle pin: on 100 random undirected graphs of assorted
    shapes (isolated vertices, multi-edges in the input, tiny and ragged degrees;
    fixed draws, edge cases first) the restatement agrees bit for bit with the
    reference's own CPU code on BFS, SSSP, PageRank and the triangle count."""
    cases = REF_CPU["rand_cases"]
    assert len(cases) == 100
    n_all, nnz_all = cases[:, 0], REF_CPU["rand_nnz"]

    def per_case(key, sizes):
        return np.split(REF_CPU["rand_" + key], np.cumsum(sizes)[:-1])
    bfs_0, bfs_last, pr = (per_case(k, n_all) for k in ("bfs_0", "bfs_last", "pr"))
    weights = per_case("weights", nnz_all)
    sssp_0 = per_case("sssp_0", np.where(nnz_all > 0, n_all, 0))
    for i, (n, m, seed) in enumerate(cases.tolist()):
        rng = np.random.RandomState(seed)
        src = rng.randint(0, n, m).astype(np.int32)
        dst = rng.randint(0, n, m).astype(np.int32)
        rp, ci = orc.build_csr(n, src, dst, True)          # drops loops/duplicates
        assert len(ci) == nnz_all[i]
        assert np.array_equal(orc.bfs(rp, ci, 0), bfs_0[i])
        assert np.array_equal(orc.bfs(rp, ci, n - 1), bfs_last[i])
        if len(ci):
            w = weights[i].astype(np.float32)
            assert np.array_equal(orc.sssp(rp, ci, w, 0), sssp_0[i])
        assert np.array_equal(orc.pr(rp, ci), pr[i])
        lr, lc = orc.tril(rp, ci)
        assert orc.tc(lr, lc) == REF_CPU["rand_tc"][i]


@pytest.mark.parametrize("scale", [14, 16])
def test_tc_goldens_match_the_oracle_port(scale):
    """tests/golden/tc_golden.json (counted by the reference's CPU code) against
    the C restatement on the same generated graph."""
    import json
    table = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)),
                                        "golden", "tc_golden.json")))
    g = table["rmat%d" % scale]
    rp, ci = orc.rmat_csr(scale)
    assert len(ci) == g["nnz"]
    check = int(np.sum(ci.astype(np.int64) *
                       (np.arange(len(ci), dtype=np.int64) % 97 + 1)))
    assert check == g["colind_checksum"]
    lr, lc = orc.tril(rp, ci)
    assert len(lc) == g["nnz_tril"]
    assert int(orc.tc(lr, lc)) == g["triangles_tril"]
