#!/usr/bin/env python
"""Generates tests/golden/ref_cpu.npz: what the reference's own CPU code
(oracle/_ref/libgbref.so, compiled from the reference sources by oracle/Makefile)
returns on the inputs that tests/test_oracle.py and tests/test_zz_ingest_gpu.py
compare against it.  Run where the reference sources are present; the file is
committed so that those comparisons run on every checkout.

Contents (keys):
  rmat<s>_*     R-MAT scale s in (8, 12) from the oracle generator: colind checksum,
                source (highest degree), BFS levels from the source and from 0,
                SSSP weights (seed 1, uniform_int[1,64], stored as uint8) and
                distances from the source, PageRank (alpha .85, eps 1e-8, 10
                iterations), triangle count of tril
  mtx_<name>_d<directed>_{rowptr,colind,val}
                readMtx + coo2csr of the bundled Matrix Market files
  rand_cases    (n, m, seed) of RANDOM_CASES undirected random graphs (edge cases
                first, then draws from a fixed seed); the graph is
                orc.build_csr(n, RandomState(seed).randint(0, n, m) x2)
  rand_nnz, rand_tc
                stored entries and triangle count of every graph
  rand_*        per graph, concatenated in case order: BFS levels from 0 and n-1
                and PageRank (n entries each), SSSP weights (seed % 1000; nnz
                entries) and distances from 0 (n entries, none when nnz is 0)
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
import oracle_binding as orc  # noqa: E402

RMAT_SCALES = (8, 12)
MTX_CASES = [("chesapeake.mtx", 0), ("chesapeake.mtx", 2), ("test_cc.mtx", 0),
             ("test_cc.mtx", 2), ("test_bc.mtx", 0), ("test_bc.mtx", 1),
             ("test_bc.mtx", 2)]
RANDOM_CASES = 100


def colind_checksum(ci):
    return int(np.sum(ci.astype(np.int64) * (np.arange(len(ci), dtype=np.int64) % 97 + 1)))


def weights_u8(w):
    u8 = w.astype(np.uint8)
    assert np.array_equal(u8.astype(np.float32), w)
    return u8


def random_graph(n, m, seed):
    rng = np.random.RandomState(seed)
    src = rng.randint(0, n, m).astype(np.int32)
    dst = rng.randint(0, n, m).astype(np.int32)
    return orc.build_csr(n, src, dst, True)


def random_cases():
    cases = [(2, 0, 0), (2, 400, 1), (60, 0, 2), (60, 400, 3), (3, 1, 4)]
    rng = np.random.RandomState(20240611)
    while len(cases) < RANDOM_CASES:
        cases.append((int(rng.randint(2, 61)), int(rng.randint(0, 401)),
                      int(rng.randint(0, 2**31 - 1))))
    return np.array(cases, dtype=np.int64)


def main():
    assert orc.ref() is not None, "oracle/_ref/libgbref.so missing: make -C oracle ref"
    out = {}
    for s in RMAT_SCALES:
        rp, ci = orc.rmat_csr(s)
        src = int(np.argmax(np.diff(rp)))
        w = orc.ref_uniform_weights(1, 1, 64, len(ci))
        lr, lc = orc.tril(rp, ci)
        k = "rmat%d_" % s
        out[k + "nnz"] = np.int64(len(ci))
        out[k + "colind_checksum"] = np.int64(colind_checksum(ci))
        out[k + "source"] = np.int64(src)
        out[k + "bfs_source"] = orc.ref_bfs(rp, ci, src)
        out[k + "bfs_0"] = orc.ref_bfs(rp, ci, 0)
        out[k + "weights"] = weights_u8(w)
        out[k + "sssp_source"] = orc.ref_sssp(rp, ci, w, src)
        out[k + "pr"] = orc.ref_pr(rp, ci)
        out[k + "tc"] = np.int64(orc.ref_tc(lr, lc))
    for name, directed in MTX_CASES:
        rp, ci, val = orc.ref_load_mtx(os.path.join(HERE, name), directed)
        k = "mtx_%s_d%d_" % (os.path.splitext(name)[0], directed)
        out[k + "rowptr"], out[k + "colind"], out[k + "val"] = rp, ci, val
    cases = random_cases()
    out["rand_cases"] = cases
    parts = {k: [] for k in ("bfs_0", "bfs_last", "weights", "sssp_0", "pr")}
    nnz, tcs = [], []
    for n, m, seed in cases.tolist():
        rp, ci = random_graph(n, m, seed)
        nnz.append(len(ci))
        parts["bfs_0"].append(orc.ref_bfs(rp, ci, 0))
        parts["bfs_last"].append(orc.ref_bfs(rp, ci, n - 1))
        if len(ci):
            w = orc.ref_uniform_weights(seed % 1000, 1, 64, len(ci))
            parts["weights"].append(weights_u8(w))
            parts["sssp_0"].append(orc.ref_sssp(rp, ci, w, 0))
        parts["pr"].append(orc.ref_pr(rp, ci))
        lr, lc = orc.tril(rp, ci)
        tcs.append(orc.ref_tc(lr, lc))
    for k, v in parts.items():
        out["rand_" + k] = np.concatenate(v)
    out["rand_nnz"] = np.array(nnz, dtype=np.int64)
    out["rand_tc"] = np.array(tcs, dtype=np.int64)
    path = os.path.join(HERE, "ref_cpu.npz")
    np.savez_compressed(path, **out)
    print("wrote %s (%d bytes)" % (path, os.path.getsize(path)))


if __name__ == "__main__":
    main()
