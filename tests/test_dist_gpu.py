"""GPU tests of the multi-GPU layer: the peer-memory exchange and the fused
traversal kernel (gb200_dist_bfs_fused) against the oracle.  World size 1 runs on
a single GPU (the owner stores into its own replica); the 2-rank test needs two
GPUs."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import oracle_binding as orc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _setup(scale, dev):
    import graphblast_b200 as gb
    from graphblast_b200 import dist as gdist
    rp, ci = orc.rmat_csr(scale)
    n = len(rp) - 1
    rowptr = torch.from_numpy(rp).to(dev)
    colind = torch.from_numpy(ci).to(dev)
    rp_l, ci_l, colptr, rowind = gdist.local_slice(rowptr, colind, 0, n, n)
    desc = gb.Descriptor(mxvmode=0, struconly=1, opreuse=0, earlyexit=1)
    ops = gdist.GpuLocalOps(gb, n, 0, n, rp_l, ci_l, colptr, rowind, desc)
    comm = gdist.Comm([0, n], dev)
    return gb, gdist, rp, ci, n, ops, comm


@pytest.mark.gpu
@pytest.mark.parametrize("scale", [10, 14, 17])
def test_native_level_loop_world1(scale):
    dev = torch.device("cuda", 0)
    gb, gdist, rp, ci, n, ops, comm = _setup(scale, dev)
    x = gdist.PeerExchange(gb, comm, dev)
    try:
        deg = np.diff(rp)
        for source in (int(np.argmax(deg)), int(np.nonzero(deg)[0][-1])):
            want = orc.bfs(rp, ci, source)
            for _ in range(2):                      # state is reset per traversal
                levels = x.bfs(ops, n, source)
                got = ops.levels().astype(np.int32)
                assert np.array_equal(got, want)
                assert levels == int(want.max())
    finally:
        x.close()


@pytest.mark.gpu
def test_python_and_native_loops_agree():
    dev = torch.device("cuda", 0)
    gb, gdist, rp, ci, n, ops, comm = _setup(13, dev)
    source = int(np.argmax(np.diff(rp)))
    gdist.run_bfs(ops, comm, source)
    a = ops.levels().copy()
    x = gdist.PeerExchange(gb, comm, dev)
    try:
        x.bfs(ops, n, source)
        b = ops.levels().copy()
    finally:
        x.close()
    assert np.array_equal(a, b)
    assert np.array_equal(a.astype(np.int32), orc.bfs(rp, ci, source))


@pytest.mark.gpu
def test_two_ranks_peer_exchange():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    env = dict(os.environ, GB200_BENCH_SCALE="18")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1",
           "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29533", os.path.join(ROOT, "bench.py"),
           "--gpus", "2", "--steps", "3", "--warmup", "1"]
    out = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, out.stdout
    res = json.loads(lines[0])
    assert res["n_gpus"] == 2
    assert res["parity_vs_cpu_reference"] is True
    assert "peer-memory" in res["config"]["exchange"]


@pytest.mark.gpu
@pytest.mark.parametrize("scale", [10, 15])
def test_native_pagerank_world1(scale):
    """gb200_dist_pr on one rank (the owner publishes into its own replica) against
    the oracle: 10 power iterations, 1e-5 relative."""
    import ctypes as C
    import graphblast_b200 as gb
    from graphblast_b200 import dist as gdist
    dev = torch.device("cuda", 0)
    rp, ci = orc.rmat_csr(scale)
    n = len(rp) - 1
    alpha = 0.85
    rowptr = torch.from_numpy(rp).to(dev)
    colind = torch.from_numpy(ci).to(dev)
    deg = (rowptr[1:] - rowptr[:-1]).to(torch.float32)
    val = (alpha / deg[colind.to(torch.int64)]).contiguous()
    lib = gb._lib.load()
    M = gb.Matrix(n, n)
    assert lib.gb200_matrix_adopt_csr(M._h, C.c_void_p(rowptr.data_ptr()),
                                      C.c_void_p(colind.data_ptr()),
                                      C.c_void_p(val.data_ptr()), int(len(ci))) == 0
    p = gb.Vector(n)
    desc = gb.Descriptor(mxvmode=0, max_niter=10)
    comm = gdist.Comm([0, n], dev)
    x = gdist.PeerExchange(gb, comm, dev, offsets=[0, n])
    try:
        for _ in range(2):
            iters = x.pr(p, M, n, alpha, 0.0, desc)
            assert iters == 10
            got = p.extractTuples()[:n]
            want = orc.pr(rp, ci, alpha, 0.0, 10)
            rel = np.abs(got - want) / np.maximum(np.abs(want), 1e-30)
            assert rel.max() <= 1e-5
    finally:
        x.close()


@pytest.mark.gpu
def test_two_ranks_pagerank():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    env = dict(os.environ, GB200_BENCH_SCALE="18")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1",
           "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29534", os.path.join(ROOT, "bench.py"),
           "--gpus", "2", "--algo", "pr", "--steps", "2", "--warmup", "1"]
    out = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, out.stdout
    res = json.loads(lines[0])
    assert res["n_gpus"] == 2
    assert res["parity_vs_cpu_reference"] is True, res["max_rel_err"]


@pytest.mark.gpu
@pytest.mark.parametrize("scale", [10, 15])
def test_native_sssp_world1(scale):
    """gb200_dist_sssp on one rank against the oracle: bit-exact distances."""
    import graphblast_b200 as gb
    from graphblast_b200 import dist as gdist, graphs
    dev = torch.device("cuda", 0)
    rp, ci = orc.rmat_csr(scale)
    n = len(rp) - 1
    nnz = len(ci)
    w = gb.api.host_uniform_weights(1, 1, 64, nnz)
    rowptr = torch.from_numpy(rp).to(dev)
    colind = torch.from_numpy(ci).to(dev)
    d_wt = graphs.transpose_values(n, rowptr, colind, torch.from_numpy(w).to(dev))
    M, keep = gdist.weighted_local_matrix(gb, n, rowptr, colind, d_wt, 0, n)
    v = gb.Vector(n)
    desc = gb.Descriptor(mxvmode=0, switchpoint=0.025)
    comm = gdist.Comm([0, n], dev)
    x = gdist.PeerExchange(gb, comm, dev, offsets=[0, n])
    try:
        deg = np.diff(rp)
        for source in (int(np.argmax(deg)), int(np.nonzero(deg)[0][-1])):
            want = orc.sssp(rp, ci, w, source)
            for _ in range(2):
                rounds = x.sssp(v, M, n, source, desc)
                assert 1 <= rounds < 200          # stops when the frontier is empty
                assert np.array_equal(v.extractTuples()[:n], want)
    finally:
        x.close()


@pytest.mark.gpu
def test_two_ranks_sssp():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    env = dict(os.environ, GB200_BENCH_SCALE="18")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1",
           "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29535", os.path.join(ROOT, "bench.py"),
           "--gpus", "2", "--algo", "sssp", "--steps", "2", "--warmup", "1"]
    out = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, out.stdout
    res = json.loads(lines[0])
    assert res["n_gpus"] == 2
    assert res["parity_vs_cpu_reference"] is True
