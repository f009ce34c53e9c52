#!/usr/bin/env python
"""bench.py — benchmark of the direction-optimised mxv/vxm path and its consumers.

Metric (BASELINE.json): MTEPS = stored entries of A / time of one full run of the
algorithm.  Workloads (`--algo`, defaults are the BASELINE.json configs):
  bfs   configs[2]  direction-optimised BFS (LogicalOrAnd vxm, push SpMSpV <-> pull
                    SpMV), R-MAT scale 24 ef 16, reference flags of run_bfs.sh:8-27
                    (--mxvmode 0 --struconly 1 --opreuse 1 --earlyexit 1)   [default]
  sssp  configs[1]  MinimumPlus SSSP, R-MAT scale 22, pull-only SpMV (--mxvmode 2)
  pr    configs[3]  PageRank (PlusMultiplies mxv), R-MAT-22 surrogate of
                    soc-LiveJournal1 (not on disk, no network), 10 iterations
  tc    configs[4]  triangle count (masked mxm on tril(A)), R-MAT scale 22
`--scale` / `--mxvmode` override the config.  A "step" is one full run from the same
source.  One JSON line on stdout:
  value         device-timed, graph resident in HBM, K steps between CUDA events
  e2e           the same run through the public API with host buffers: step input
                H2D from pinned memory + run + D2H of the n-float result, every step
  roofline      the dominant hot kernel: algorithmic bytes (SURVEY.md §8d) / CUDA-event
                time of its launches, against the measured HBM peak
  per_mxv       per hot kernel: launches, ms, edges touched per ms (§8d)
  cpu_baseline  the reference's own CPU code (oracle/_ref) on one host core
  parity_vs_cpu_reference   the GPU result against that CPU code (this file is the
                only place that touches oracle/; the package never does)

`--impl reference` times the reference's CPU implementation instead (rank 0 only).
`--dump-outputs DIR` also writes what the last timed step computed to DIR/*.npy
(levels / distances / ranks, or the triangle count; see dump_outputs).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

# one unit string for every line this file (and graphblast_b200.dist) prints
UNIT = "MTEPS (stored entries of A / traversal time x 1e-6)"

DEFAULT_SCALE = {"bfs": 24, "sssp": 22, "pr": 22, "tc": 22}
DEFAULT_MXVMODE = {"bfs": 0, "sssp": 2, "pr": 0, "tc": 0}
PR_ITERATIONS = 10
PR_ALPHA = 0.85
PR_TOLERANCE = 1e-5          # north_star: relative, PageRank / SSSP


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--algo", default="bfs", choices=["bfs", "sssp", "pr", "tc"])
    ap.add_argument("--scale", type=int, default=None,
                    help="R-MAT scale; default: GB200_BENCH_SCALE, else the scale "
                         "BASELINE.json names for the algorithm (bfs 24, others 22)")
    ap.add_argument("--mxvmode", type=int, default=None, choices=[0, 1, 2],
                    help="0 push-pull, 1 push only, 2 pull only (reference "
                         "--mxvmode); default per config: bfs 0, sssp 2")
    ap.add_argument("--edgefactor", type=int, default=16)
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step "
                         "computed to DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and (args.impl != "ours" or args.gpus != 1 or
                                          int(os.environ.get("WORLD_SIZE", "1")) != 1):
        ap.error("--dump-outputs writes the results of the single-GPU path: "
                 "use it with --impl ours --gpus 1 in a single process")
    if args.scale is None:
        env = os.environ.get("GB200_BENCH_SCALE")
        args.scale = int(env) if env else DEFAULT_SCALE[args.algo]
    if args.mxvmode is None:
        args.mxvmode = DEFAULT_MXVMODE[args.algo]
    return args


class ClockSampler(object):
    """SM clock and throttle reasons sampled DURING the timed region through NVML
    (a polling thread; nvidia-smi's own loop is too slow for millisecond regions).
    Falls back to one nvidia-smi query when pynvml is unavailable."""

    def __init__(self, index):
        self.index = index
        self.samples = []
        self.reasons = set()
        self.sm_max = None
        self.stop_flag = False
        self.thread = None
        self.nvml = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.sm_max = float(pynvml.nvmlDeviceGetMaxClockInfo(
                self.handle, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nvml = None
            return
        self.thread = threading.Thread(target=self._poll, daemon=True)
        self.thread.start()

    def _poll(self):
        nv = self.nvml
        names = [("hw_slowdown", "nvmlClocksThrottleReasonHwSlowdown"),
                 ("hw_thermal_slowdown", "nvmlClocksThrottleReasonHwThermalSlowdown"),
                 ("sw_thermal_slowdown", "nvmlClocksThrottleReasonSwThermalSlowdown"),
                 ("sw_power_cap", "nvmlClocksThrottleReasonSwPowerCap")]
        masks = [(n, getattr(nv, a, 0)) for n, a in names]
        while not self.stop_flag:
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(
                    self.handle, nv.NVML_CLOCK_SM)))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
                for n, m in masks:
                    if m and (r & m):
                        self.reasons.add(n)
            except Exception:
                pass
            time.sleep(0.0005)

    def stop(self):
        if self.nvml is None:
            try:
                q = subprocess.run(
                    ["nvidia-smi", "-i", str(self.index),
                     "--query-gpu=clocks.sm,clocks.max.sm",
                     "--format=csv,noheader,nounits"], stdout=subprocess.PIPE,
                    text=True, timeout=20).stdout.split(",")
                return {"sm_mhz": float(q[0]), "sm_max_mhz": float(q[1]),
                        "samples": 1, "reasons": ["sampled after the region"]}
            except Exception:
                return {"sm_mhz": None, "sm_max_mhz": None, "samples": 0,
                        "reasons": ["unavailable"]}
        self.stop_flag = True
        self.thread.join(timeout=2)
        return {"sm_mhz": statistics.median(self.samples) if self.samples else None,
                "sm_max_mhz": self.sm_max, "samples": len(self.samples),
                "reasons": sorted(self.reasons)}


def measured_peak_hbm():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def measured_traffic(args, kind):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant
    kernel, from the committed `ncu --set full` capture of this workload
    (profiles/traffic.json); None when no capture of this (algo, scale, kernel)
    has been taken."""
    path = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        table = json.load(open(path))
        return table.get("%s:%d:%d" % (args.algo, args.scale, kind))
    except Exception:
        return None


def build_graph(args, torch, graphs):
    """R-MAT on the device with the reference loader's semantics (undirected,
    no self-loops, no duplicates, sorted rows)."""
    n = 1 << args.scale
    src, dst = graphs.rmat_edges(args.scale, args.edgefactor, seed=args.seed)
    rowptr, colind = graphs.build_csr(n, src, dst, undirected=True)
    del src, dst
    torch.cuda.empty_cache()
    return n, rowptr, colind


# ---------------------------------------------------------------------------
# The checker: the reference's CPU code (oracle/_ref, else the oracle port) on the
# same graph.  Used by the single-GPU path below, by graphblast_b200.dist through
# args.verify, and timed by --impl reference.
# ---------------------------------------------------------------------------

def _orc():
    import oracle_binding as orc
    return orc, ("reference" if orc.ref() is not None else "port")


def pagerank_fp64(h_rp, h_ci, alpha, niter):
    """The iteration of reference test_pr.hpp:15-80 in float64 (the arithmetic
    truth both float32 results are measured against)."""
    import numpy as np
    import scipy.sparse as sp
    n = len(h_rp) - 1
    A = sp.csr_matrix((np.ones(len(h_ci), dtype=np.float64), h_ci, h_rp), shape=(n, n))
    outdeg = np.diff(h_rp).astype(np.float64)
    p = np.full(n, 1.0 / n)
    for _ in range(niter):
        contrib = np.divide(p, outdeg, out=np.zeros(n), where=outdeg > 0)
        p = (1.0 - alpha) / n + alpha * (A.T @ contrib)
    return p


def tc_golden(scale, nnz, h_ci):
    """Committed triangle count of this exact graph (tests/golden/tc_golden.json,
    counted once by the reference's SimpleReferenceTc), or None."""
    import numpy as np
    try:
        table = json.load(open(os.path.join(ROOT, "tests", "golden", "tc_golden.json")))
    except Exception:
        return None
    g = table.get("rmat%d" % scale)
    if g is None or g["nnz"] != nnz:
        return None
    check = int(np.sum(h_ci.astype(np.int64) *
                       (np.arange(len(h_ci), dtype=np.int64) % 97 + 1)))
    return g if check == g["colind_checksum"] else None


def tc_sample_rows(lr, budget_entries=3_000_000):
    """Leading principal submatrix L[0:r, 0:r] with about budget_entries stored
    entries: closed under the intersections of a triangle count on tril (every
    neighbour of a row is a lower row), so it is a well-defined bounded sample of
    the same workload for timing the sequential CPU code."""
    import numpy as np
    r = int(np.searchsorted(lr, budget_entries, side="left"))
    return max(min(r, len(lr) - 1), 1)


def verify(args, algo, h_rp, h_ci, got, ctx):
    """(parity, cpu_baseline, extra) — got: the GPU result (levels / distances /
    ranks as float32[n], or the triangle count)."""
    import numpy as np
    orc, kind = _orc()
    nnz = int(len(h_ci))
    extra = None
    base = {"unit": "MTEPS", "cores": 1, "kind": kind,
            "host_cores_total": os.cpu_count()}
    if algo == "bfs":
        fn = orc.ref_bfs if kind == "reference" else orc.bfs
        t0 = time.perf_counter()
        want = fn(h_rp, h_ci, ctx["source"])
        dt = time.perf_counter() - t0
        parity = bool(np.array_equal(np.asarray(got).astype(np.int32), want))
        base.update(value=nnz / (dt * 1e6), ms=dt * 1e3,
                    sample="one full BFS of the same graph from the same source")
    elif algo == "sssp":
        fn = orc.ref_sssp if kind == "reference" else orc.sssp
        t0 = time.perf_counter()
        want = fn(h_rp, h_ci, ctx["weights"], ctx["source"])
        dt = time.perf_counter() - t0
        parity = bool(np.array_equal(np.asarray(got), want))
        base.update(value=nnz / (dt * 1e6), ms=dt * 1e3,
                    sample="one full SSSP of the same graph from the same source")
    elif algo == "pr":
        fn = orc.ref_pr if kind == "reference" else orc.pr
        alpha, niter = ctx["alpha"], ctx["niter"]
        t0 = time.perf_counter()
        want = fn(h_rp, h_ci, alpha, 0.0, niter)   # exactly the iterations the GPU ran
        dt = time.perf_counter() - t0
        truth = pagerank_fp64(h_rp, h_ci, alpha, niter)
        got64 = np.asarray(got, dtype=np.float64)

        def rel(x, y):
            return float(np.max(np.abs(x - y) / np.maximum(np.abs(y), 1e-300)))
        gpu_vs_ref = rel(got64, want.astype(np.float64))
        gpu_vs_truth = rel(got64, truth)
        ref_vs_truth = rel(want.astype(np.float64), truth)
        # north_star: within 1e-5 relative of the reference.  Both sides compute the
        # same float32 iteration with different summation orders; where the
        # reference's own float32 error against the float64 iteration exceeds the
        # tolerance (hub rows: >1e5 sequential float32 adds), agreement with the
        # reference cannot be better than that error, so the test is: the GPU is
        # within tolerance of the float64 iteration AND no further from the
        # reference than the reference is from the float64 iteration (+ tolerance).
        parity = bool(gpu_vs_truth <= PR_TOLERANCE and
                      gpu_vs_ref <= ref_vs_truth + PR_TOLERANCE)
        extra = {"tolerance": PR_TOLERANCE,
                 "max_rel_err_vs_reference": gpu_vs_ref,
                 "max_rel_err_vs_fp64_iteration": gpu_vs_truth,
                 "reference_max_rel_err_vs_fp64_iteration": ref_vs_truth,
                 "within_tolerance_of_reference": bool(gpu_vs_ref <= PR_TOLERANCE)}
        base.update(value=nnz / (dt * 1e6), ms=dt * 1e3,
                    sample="one full PageRank (%d iterations) of the same graph" % niter)
    else:  # tc — ctx: lr, lc (host tril), scale
        lr, lc = ctx["lr"], ctx["lc"]
        fn = orc.ref_tc if kind == "reference" else orc.tc
        g = tc_golden(ctx["scale"], nnz, h_ci)
        if g is not None and ctx["scale"] > 18:
            want = int(g["triangles_tril"])
            r = tc_sample_rows(lr)
            t0 = time.perf_counter()
            fn(lr[:r + 1].copy(), lc[:lr[r]].copy())
            dt = time.perf_counter() - t0
            sample_nnz = 2 * int(lr[r])
            base.update(value=sample_nnz / (dt * 1e6), ms=dt * 1e3,
                        sample="triangle count of the leading %d rows of tril(A) "
                               "(%d stored entries, a neighbour-closed part of the "
                               "same graph); the full count (%d, %.0f s on one core) "
                               "is the committed golden tests/golden/tc_golden.json"
                               % (r, int(lr[r]), want, g["cpu_seconds"]))
            extra = {"expected": want, "source": "tests/golden/tc_golden.json"}
        else:
            t0 = time.perf_counter()
            want = int(fn(lr, lc))
            dt = time.perf_counter() - t0
            base.update(value=nnz / (dt * 1e6), ms=dt * 1e3,
                        sample="one full triangle count of the same graph")
            extra = {"expected": want, "source": "counted in this run"}
            if g is not None:
                extra["golden_agrees"] = bool(want == int(g["triangles_tril"]))
        parity = bool(int(got) == want)
    return parity, base, extra


def run_reference_arm(args):
    """The reference's CPU implementation (SimpleReferenceBfs / Sssp / Pr / Tc, built
    from the reference sources into oracle/_ref; oracle port when that is absent) on
    the same graph and source; one run per step, single host thread (the reference's
    CPU code is sequential).  Triangle counting above scale 18 times a bounded,
    neighbour-closed sample (tc_sample_rows) per step."""
    import numpy as np
    import torch
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import graphblast_b200 as gb
    from graphblast_b200 import graphs
    orc, kind = _orc()
    torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
    gb.init(int(os.environ.get("LOCAL_RANK", "0")))
    n, rowptr, colind = build_graph(args, torch, graphs)
    h_rp = rowptr.cpu().numpy()
    h_ci = colind.cpu().numpy()
    nnz = int(h_ci.shape[0])
    source = int(np.argmax(np.diff(h_rp)))
    del rowptr, colind
    work = nnz
    sample = ("one full run of the same algorithm on the same graph per step "
              "(sequential code: 1 host thread)")
    if args.algo == "sssp":
        w = gb.api.host_uniform_weights(args.seed, 1, 64, nnz)
        step = (lambda: orc.ref_sssp(h_rp, h_ci, w, source)) if kind == "reference" \
            else (lambda: orc.sssp(h_rp, h_ci, w, source))
    elif args.algo == "pr":
        step = (lambda: orc.ref_pr(h_rp, h_ci, PR_ALPHA, 0.0, PR_ITERATIONS)) \
            if kind == "reference" \
            else (lambda: orc.pr(h_rp, h_ci, PR_ALPHA, 0.0, PR_ITERATIONS))
    elif args.algo == "tc":
        lr, lc = orc.tril(h_rp, h_ci)        # the reference driver counts on tril(A)
        fn = orc.ref_tc if kind == "reference" else orc.tc
        if args.scale > 18:
            r = tc_sample_rows(lr)
            slr, slc = lr[:r + 1].copy(), lc[:lr[r]].copy()
            work = 2 * int(lr[r])
            sample = ("triangle count of the leading %d rows of tril(A), %d stored "
                      "entries (a neighbour-closed part of the same graph; the full "
                      "sequential count takes about an hour)" % (r, int(lr[r])))
            step = lambda: fn(slr, slc)      # noqa: E731
        else:
            step = lambda: fn(lr, lc)        # noqa: E731
    else:
        step = (lambda: orc.ref_bfs(h_rp, h_ci, source)) if kind == "reference" \
            else (lambda: orc.bfs(h_rp, h_ci, source))
    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = time.perf_counter() - t0
    ms = dt * 1e3 / args.steps
    mteps = work / (ms * 1e3)
    out = {
        "impl": "reference",
        "metric": "MTEPS", "value": mteps, "unit": UNIT,
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, n, nnz, source),
        "cpu_baseline": {"value": mteps, "unit": "MTEPS", "cores": 1,
                         "kind": kind, "sample": sample},
        "e2e": {"value": mteps, "unit": "MTEPS", "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
    }
    print(json.dumps(out), flush=True)


def workload_config(args, n, nnz, source):
    names = {"bfs": "direction-optimised BFS (LogicalOrAnd vxm, push<->pull)",
             "sssp": "SSSP (MinimumPlus vxm)",
             "pr": "PageRank (PlusMultiplies vxm, %d iterations)" % PR_ITERATIONS,
             "tc": "triangle count (masked mxm on tril)"}
    flags = "--mxvmode %d" % args.mxvmode
    if args.algo == "bfs":
        flags += " --struconly 1 --opreuse 1 --earlyexit 1"
    return {"workload": "%s on R-MAT scale-%d ef-%d (a,b,c,d)=(.57,.19,.19,.05) "
                        "seed %d, symmetrised, no self-loops/duplicates"
                        % (names[args.algo], args.scale, args.edgefactor,
                           args.seed),
            "n": n, "nnz": nnz, "source": source, "flags": flags,
            "l2_policy": "inputs larger than L2 (graph arrays >> 126 MB)",
            "partition": "1-D row slices" if args.gpus > 1 else "single GPU"}


# --dump-outputs: the result a caller of the timed path receives, one float32 or
# float64 .npy file per array.  A vector longer than DUMP_SAMPLE entries is written
# as a fixed sample (DUMP_SEED) of DUMP_SAMPLE entries in index order, with the
# sampled indices in <name>_index.npy, which keeps the files under DUMP_LIMIT bytes
# in all.  The inputs depend on the arguments only, so two builds of the library
# run with the same arguments can be compared entry for entry.
DUMP_NAMES = {"bfs": "levels", "sssp": "distances", "pr": "ranks"}
DUMP_SAMPLE = 1 << 22
DUMP_SEED = 1
DUMP_LIMIT = 64 * 10**6


def dump_outputs(out_dir, outputs):
    """outputs: name -> 1-D array; written as out_dir/<name>.npy."""
    import numpy as np
    files = {}
    for name, a in outputs.items():
        a = np.asarray(a)
        a = a.astype(np.float32 if a.dtype == np.float32 else np.float64)
        if a.size > DUMP_SAMPLE:
            idx = np.sort(np.random.default_rng(DUMP_SEED).choice(
                a.size, DUMP_SAMPLE, replace=False))
            files[name + "_index"] = idx.astype(np.float64)
            a = a[idx]
        files[name] = a
    total = sum(a.nbytes for a in files.values())
    if total > DUMP_LIMIT:
        raise RuntimeError("--dump-outputs: %d bytes exceed the %d-byte limit"
                           % (total, DUMP_LIMIT))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in files.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


KINDS = ["spmvMergeKernel / spmvHubKernel (generic pull SpMV)",
         "spmvMaskedOrPullKernel (fused Boolean pull)",
         "spmspvPushKernel (push SpMSpV expand)",
         "spgemmHashKernel x6 per call (masked SpGEMM, hash formulation)"]


def per_mxv_rates(args, prof, n, nnz, fused=None):
    """Edges touched per millisecond of every hot kernel (SURVEY.md §8d), from the
    algorithmic bytes the library accumulates per kind:
      generic pull  : every stored entry, per launch;
      Boolean pull  : (bytes - 12n - 4 per launch) / 4 = colind entries inspected;
      push          : (bytes - frontier/output terms) / bytes per expanded edge
                      (colind 4 + value 4 if key-value + mask lookup 4 if masked:
                      8 for the BFS and SSSP pushes)."""
    out = {}
    for k, (ms, ln, by) in enumerate(prof):
        if ln == 0:
            continue
        if k == 0:
            edges = float(ln) * nnz
        elif k == 1 and fused is not None:
            # one launch per traversal: inspected + pushed entries of the last
            # traversal (every traversal from the same source does the same work)
            edges = float(ln) * (fused[1] + fused[4])
        elif k == 1:
            edges = max(by - ln * (12.0 * n + 4.0), 0.0) / 4.0
        elif k == 2:
            edges = by / 8.0
        else:
            edges = float(ln) * nnz
        out[KINDS[k]] = {"launches": ln, "ms": ms, "alg_bytes": by,
                         "edges_touched": edges,
                         "edges_touched_per_ms": edges / ms if ms > 0 else None}
    return out


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference_arm(args)
        return

    import numpy as np
    import torch
    import graphblast_b200 as gb
    from graphblast_b200 import algorithm, graphs, _lib
    import ctypes as C

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    gb.init(local_rank)
    lib = _lib.load()

    if world > 1:
        from graphblast_b200 import dist as gdist
        assert gdist.UNIT == UNIT
        args.verify = lambda algo, rp, ci, got, ctx: verify(args, algo, rp, ci, got, ctx)
        result = gdist.bench_distributed(args, world, rank, local_rank)
        if rank == 0:
            print(json.dumps(result), flush=True)
        return

    n, rowptr, colind = build_graph(args, torch, graphs)
    nnz = int(colind.numel())
    deg = rowptr[1:] - rowptr[:-1]
    source = int(torch.argmax(deg).item())

    desc_flags = dict(mxvmode=args.mxvmode)
    if args.algo == "bfs":
        desc_flags.update(struconly=1, opreuse=1, earlyexit=1)
    if args.algo == "sssp":
        desc_flags.update(switchpoint=0.025)
    if args.algo == "pr":
        desc_flags.update(max_niter=PR_ITERATIONS)
    desc = gb.Descriptor(**desc_flags)

    keep = []
    w = None
    h_tril = None
    if args.algo == "bfs":
        A = graphs.matrix_from_csr(n, rowptr, colind)
    elif args.algo in ("sssp", "pr"):
        if args.algo == "sssp":
            w = gb.api.host_uniform_weights(args.seed, 1, 64, nnz)
            d_w = torch.from_numpy(w).cuda()
        else:
            d_w = torch.ones(nnz, dtype=torch.float32, device="cuda")
        d_wt = graphs.transpose_values(n, rowptr, colind, d_w)
        A = graphs.matrix_from_csr(n, rowptr, colind, d_w, cscval=d_wt)
        keep += [d_w, d_wt]
        if args.algo == "pr":
            A.pr_normalize(PR_ALPHA, desc)
    else:
        # L = tril(A) through the library's own tril (reference gtc.cu:76-80)
        A = graphs.matrix_from_csr(n, rowptr, colind, dtype=gb.api.INT32,
                                   symmetric=True)
        A.tril(desc)
        h_tril = A.extract_csr()[:2]
        B = gb.Matrix(n, n, dtype=gb.api.INT32)

    result_vec = gb.Vector(n)
    tc_count = [0]

    def step():
        if args.algo == "bfs":
            algorithm.bfs(result_vec, A, source, desc)
        elif args.algo == "sssp":
            algorithm.sssp(result_vec, A, source, desc)
        elif args.algo == "pr":
            algorithm.pr(result_vec, A, PR_ALPHA, 0.0, desc)
        else:
            tc_count[0] = algorithm.tc(A, B, desc)[0]

    # ---- warm-up ---------------------------------------------------------
    for _ in range(max(args.warmup, 1)):
        step()
    torch.cuda.synchronize()

    # ---- device-timed region -----------------------------------------------
    launches0 = C.c_ulonglong(0)
    lib.gb200_launch_count(C.byref(launches0))
    lib.gb200_profile_enable(1)
    lib.gb200_profile_reset()
    sampler = ClockSampler(local_rank)
    sampler.start()
    ev0 = torch.cuda.Event(enable_timing=True)
    ev1 = torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    ev0.record()
    for _ in range(args.steps):
        step()
    ev1.record()
    torch.cuda.synchronize()
    clocks = sampler.stop()
    total_ms = ev0.elapsed_time(ev1)
    launches1 = C.c_ulonglong(0)
    lib.gb200_launch_count(C.byref(launches1))
    ms_per_step = total_ms / args.steps
    mteps = nnz / (ms_per_step * 1e3)

    prof = []
    for k in range(4):
        ms, ln, by = C.c_double(0), C.c_longlong(0), C.c_double(0)
        lib.gb200_profile_read(k, C.byref(ms), C.byref(ln), C.byref(by))
        prof.append((ms.value, ln.value, by.value))
    lib.gb200_profile_enable(0)
    fused_stats = None
    if args.algo == "bfs":
        st = (C.c_ulonglong * 6)()
        lib.gb200_bfs_stats(desc._h, n, st)
        if st[0] > 0:
            fused_stats = [int(x) for x in st]
            KINDS[1] = "bfsFusedKernel (whole traversal: Boolean pull + push levels)"
    if args.dump_outputs is not None:
        # before the end-to-end runs below overwrite the result
        if args.algo == "tc":
            dump_outputs(args.dump_outputs, {"triangles": [tc_count[0]]})
        else:
            dump_outputs(args.dump_outputs,
                         {DUMP_NAMES[args.algo]: result_vec.extractTuples()})
    dom = max(range(4), key=lambda k: prof[k][0])
    peak, peak_src = measured_peak_hbm()
    dom_ms, dom_launches, dom_bytes = prof[dom]
    achieved = (dom_bytes / 1e9) / (dom_ms / 1e3) if dom_ms > 0 else 0.0
    roofline = {
        "kernel": KINDS[dom], "bound": "hbm",
        "achieved": achieved, "peak": peak, "unit": "GB/s",
        "frac": achieved / peak if peak else None,
        "peak_source": peak_src,
        "launches": dom_launches,
        "bytes_per_launch": dom_bytes / dom_launches if dom_launches else 0,
        "ms_per_launch": dom_ms / dom_launches if dom_launches else 0,
        "share_of_step": dom_ms / total_ms if total_ms else 0,
        "traffic": measured_traffic(args, dom),
    }
    if args.algo == "tc":
        roofline["note"] = ("achieved = index-list bytes streamed through the tables / "
                            "time of the six hash launches; about half of them are L2 "
                            "hits and the kernels are issue-bound (profiles/), so this "
                            "is not a DRAM fraction")
    if fused_stats is not None:
        roofline["fused_traversal"] = dict(zip(
            ["levels", "entries_inspected_pulling", "pull_levels", "vertices_pushed",
             "edges_pushed", "discovered_pushing"], fused_stats))

    # ---- end-to-end through the public API, host buffers -----------------------
    host_out = torch.empty(n, dtype=torch.float32).pin_memory()
    host_src = torch.tensor([source], dtype=torch.int32).pin_memory()
    dev_src = torch.empty(1, dtype=torch.int32, device="cuda")
    for _ in range(2):
        step()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        dev_src.copy_(host_src, non_blocking=True)           # H2D: step input
        s = int(dev_src.item()) if args.algo in ("bfs", "sssp") else source
        if args.algo == "bfs":
            algorithm.bfs(result_vec, A, s, desc)
        elif args.algo == "sssp":
            algorithm.sssp(result_vec, A, s, desc)
        else:
            step()
        if args.algo != "tc":
            result_vec.extract_into(host_out)                # D2H: step result
    torch.cuda.synchronize()
    e2e_ms = (time.perf_counter() - t0) * 1e3 / args.steps
    e2e = {"value": nnz / (e2e_ms * 1e3), "unit": "MTEPS",
           "ms_per_step": e2e_ms,
           "h2d_bytes_per_step": 4,
           "d2h_bytes_per_step": 4 * n if args.algo != "tc" else 8,
           "note": "graph resident (built once, like the reference's "
                   "Matrix::build before its timed loop); per step: source id "
                   "H2D, run, n-float result D2H into pinned memory"}

    # ---- CPU baseline + parity: the reference's own CPU code on one host core -----
    cpu_baseline = None
    parity = None
    extra = None
    if not args.no_cpu_baseline:
        h_rp = rowptr.cpu().numpy()
        h_ci = colind.cpu().numpy()
        if args.algo == "tc":
            got = tc_count[0]
            ctx = {"lr": h_tril[0], "lc": h_tril[1], "scale": args.scale}
        else:
            got = result_vec.extractTuples()
            ctx = {"source": source, "weights": w, "alpha": PR_ALPHA,
                   "niter": PR_ITERATIONS}
        parity, cpu_baseline, extra = verify(args, args.algo, h_rp, h_ci, got, ctx)

    out = {
        "metric": "MTEPS", "value": mteps, "unit": UNIT,
        "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_per_step, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": workload_config(args, n, nnz, source),
        "clocks": clocks,
        "e2e": e2e,
        "gpu_launches": int(launches1.value - launches0.value),
        "roofline": roofline,
        "per_mxv": per_mxv_rates(args, prof, n, nnz, fused_stats),
        "cpu_baseline": cpu_baseline,
        "parity_vs_cpu_reference": parity,
    }
    if args.algo == "tc":
        out["triangles"] = int(tc_count[0])
        out["triangle_check"] = extra
    if args.algo == "pr":
        out["pagerank_check"] = extra
    print(json.dumps(out), flush=True)


def _guard_stdout():
    """The contract is ONE JSON line on stdout.  Native code (NCCL's version
    banner, printf in libraries) writes to file descriptor 1 directly, so fd 1 is
    pointed at stderr and Python's sys.stdout keeps the real stdout."""
    real = os.dup(1)
    os.dup2(2, 1)
    sys.stdout = os.fdopen(real, "w", buffering=1)


if __name__ == "__main__":
    _guard_stdout()
    main()
