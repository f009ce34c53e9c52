"""1-D row-partitioned multi-GPU traversal (SURVEY.md §8e).

One process per GPU (torchrun), `torch.distributed` for rendezvous and the NCCL
collective.  Rank p owns the output vertices [bounds[p], bounds[p+1]) and stores
the rows of A^T for them as a rectangular local matrix M (n_local x n, CSR for the
pull direction, CSC for the push direction), so both directions produce only
owned outputs and no reduction across ranks is needed.  After each local mxv the
new frontier is exchanged with ONE collective: every rank contributes the bitmap
of its owned slice (n/8 bytes in total for n vertices, plus its count), and every
rank receives the whole bitmap = the replicated input vector of the next level.

The reference has no distributed path at all (SURVEY.md §2 "Parallelism
strategies": none); the per-level operation sequence is the reference's BFS loop
(graphblas/algorithm/bfs.hpp:46-79) applied to the owned slice:
    assign(v_own<f_own> = level); f2_own<!v_own> = M (||.&&) f_global; exchange.

The generic driver `run_bfs` only talks to a `LocalOps` object and a `Comm`
object, so its partition / exchange / termination logic is testable on CPU with
the gloo backend and a host-side stand-in for the local operations (tests/).
"""
import ctypes as C

import numpy as np
import torch


# ---------------------------------------------------------------------------
# Partition
# ---------------------------------------------------------------------------

# The one unit string of every bench line (both arms, every N): the driver divides
# lines only when their units agree.
UNIT = "MTEPS (stored entries of A / traversal time x 1e-6)"


class _DevView(object):
    """A raw device pointer as something torch.as_tensor understands."""

    def __init__(self, ptr, count):
        self.__cuda_array_interface__ = {
            "shape": (count,), "typestr": "<f4", "data": (int(ptr), False),
            "version": 2}


class ResultGather(object):
    """End-to-end result path of the partitioned runs: the owned float slice of
    every rank is gathered over NCCL into one n-float vector on rank 0's GPU and
    copied into rank 0's pinned host buffer — the same 4n bytes of device->host
    traffic per step as the single-GPU run."""

    def __init__(self, bounds, world, rank, device):
        self.bounds, self.world, self.rank, self.device = bounds, world, rank, device
        self.sizes = [bounds[p + 1] - bounds[p] for p in range(world)]
        self.pad = max(self.sizes)
        self.n = bounds[world]
        self.buf = torch.zeros(self.pad, dtype=torch.float32, device=device)
        self.allv = torch.zeros(self.pad * world, dtype=torch.float32, device=device)
        self.host = (torch.empty(self.n, dtype=torch.float32).pin_memory()
                     if rank == 0 else None)

    def run(self, vec):
        """vec: gb.Vector holding this rank's owned slice.  Returns the host buffer
        on rank 0 (valid after the call), None elsewhere."""
        import torch.distributed as dist
        nl = self.sizes[self.rank]
        if nl > 0:
            view = torch.as_tensor(_DevView(vec.device_ptr(), nl), device=self.device)
            self.buf[:nl].copy_(view)
        dist.all_gather_into_tensor(self.allv, self.buf)
        if self.rank == 0:
            for p in range(self.world):
                if self.sizes[p]:
                    self.host[self.bounds[p]:self.bounds[p + 1]].copy_(
                        self.allv[p * self.pad:p * self.pad + self.sizes[p]],
                        non_blocking=True)
            torch.cuda.synchronize()
            return self.host
        return None

    d2h_bytes = property(lambda self: 4 * self.n)


def timed_e2e(args, step, gather, vec, dev, h2d_bytes):
    """K steps through the public call path with host buffers: per step the step's
    input goes host->device from pinned memory, the traversal runs, and the full
    n-float result lands in rank 0's pinned host memory.  Wall clock, max over
    ranks.  Returns (ms per step, e2e dict without the value)."""
    import time
    import torch.distributed as dist
    host_in = torch.zeros(max(h2d_bytes // 4, 1), dtype=torch.int32).pin_memory()
    dev_in = torch.zeros_like(host_in, device=dev)
    for _ in range(2):
        step()
        gather.run(vec)
    torch.cuda.synchronize()
    dist.barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        dev_in.copy_(host_in, non_blocking=True)
        step()
        gather.run(vec)
    torch.cuda.synchronize()
    wall = torch.tensor([(time.perf_counter() - t0) * 1e3], device=dev)
    dist.all_reduce(wall, op=dist.ReduceOp.MAX)
    return float(wall.item()) / args.steps



def partition_bounds(rowptr, world, align=1024, row_weight=0.0):
    """Contiguous vertex ranges with (nearly) equal COST, cost of a vertex =
    its stored entries + row_weight; every boundary is a multiple of `align`
    (>= 32, so bitmap slices are whole words).  row_weight = 0 balances stored
    entries (what an SpMV iteration costs); the Boolean pull of a BFS mostly
    pays per ROW it has to look at (first-neighbour probe), so the BFS bench
    passes a row weight (GB200_DIST_ROW_WEIGHT; default 1e9 = equal vertex counts,
    measured best on R-MAT scale 24 at 2 GPUs: 0.464 ms entries-balanced, 0.428 at
    weight 32, 0.390 at 128, 0.385 with equal vertex counts).  rowptr: 1-D integer tensor/array of length n+1.  Returns a
    list of world+1 ints."""
    rp = rowptr if isinstance(rowptr, np.ndarray) else rowptr.cpu().numpy()
    n = len(rp) - 1
    assert align % 32 == 0
    cost = rp.astype(np.float64) + row_weight * np.arange(n + 1, dtype=np.float64)
    total = float(cost[-1])
    bounds = [0]
    for p in range(1, world):
        target = total * p / world
        v = int(np.searchsorted(cost, target, side="left"))
        v = min(n, max(bounds[-1], (v + align // 2) // align * align))
        bounds.append(v)
    bounds.append(n)
    for p in range(world):
        if bounds[p + 1] < bounds[p]:
            bounds[p + 1] = bounds[p]
    return bounds


def words_of(lo, hi):
    return (hi - lo + 31) // 32


def local_slice(rowptr, colind, lo, hi, n, return_order=False):
    """CSR and CSC (device tensors when the inputs are) of rows [lo, hi) of a
    structurally symmetric matrix, i.e. of A^T restricted to the owned outputs.
    Returns rp_local[n_local+1], ci_local[nnz_l], colptr[n+1], rowind[nnz_l]
    (+ the CSR->CSC permutation of the local entries when return_order)."""
    e0 = int(rowptr[lo])
    e1 = int(rowptr[hi])
    rp_local = (rowptr[lo:hi + 1] - rowptr[lo]).to(torch.int32).contiguous()
    ci_local = colind[e0:e1].contiguous()
    nl = hi - lo
    rows = torch.repeat_interleave(
        torch.arange(nl, device=colind.device, dtype=torch.int64),
        (rp_local[1:] - rp_local[:-1]).to(torch.int64))
    key = ci_local.to(torch.int64) * nl + rows
    order = torch.argsort(key)
    rowind = rows[order].to(torch.int32).contiguous()
    counts = torch.bincount(ci_local.to(torch.int64), minlength=n)
    colptr = torch.zeros(n + 1, dtype=torch.int64, device=colind.device)
    torch.cumsum(counts, 0, out=colptr[1:])
    if return_order:
        return (rp_local, ci_local, colptr.to(torch.int32).contiguous(), rowind,
                order)
    return rp_local, ci_local, colptr.to(torch.int32).contiguous(), rowind


# ---------------------------------------------------------------------------
# Frontier exchange
# ---------------------------------------------------------------------------

class Comm(object):
    """Bitmap all-gather with uneven owned slices.  Each rank sends a fixed-size
    record: max_words bitmap words followed by two words holding its 64-bit
    count; the records are unpacked into the global bitmap (slices are whole
    words because every boundary is a multiple of 32)."""

    def __init__(self, bounds, device, group=None):
        import torch.distributed as dist
        self.dist = dist
        self.group = group
        self.bounds = bounds
        self.world = len(bounds) - 1
        self.rank = dist.get_rank(group) if self.world > 1 else 0
        self.words = [words_of(bounds[p], bounds[p + 1]) for p in range(self.world)]
        self.max_words = max(self.words) if self.words else 0
        self.max_words += self.max_words & 1          # 8-byte aligned count cell
        self.rec = self.max_words + 2
        self.device = torch.device(device)
        self.sendbuf = torch.zeros(self.rec, dtype=torch.int32, device=device)
        self.recvbuf = torch.zeros(self.rec * self.world, dtype=torch.int32,
                                   device=device)
        self.total_words = sum(self.words)
        self.gbits = torch.zeros(self.total_words + 8, dtype=torch.int32,
                                 device=device)
        self.offsets = np.concatenate([[0], np.cumsum(self.words)]).tolist()

    def send_bits(self):
        """Device view the owner writes its bitmap words into."""
        return self.sendbuf

    def count_ptr(self):
        """Device address of the 64-bit count cell in the send record."""
        return self.sendbuf.data_ptr() + 4 * self.max_words

    def set_host_record(self, local_bits, local_count):
        """Fill the send record from host-known values (seed level, CPU tests)."""
        w = self.words[self.rank]
        self.sendbuf[:w] = local_bits[:w]
        tail = torch.tensor([int(local_count) & 0xffffffff,
                             int(local_count) >> 32], dtype=torch.int64)
        tail = torch.where(tail >= 2 ** 31, tail - 2 ** 32, tail).to(torch.int32)
        self.sendbuf[self.max_words:self.max_words + 2] = tail.to(self.device)

    def exchange(self):
        """All-gathers the send records; returns (global bitmap, global count)."""
        if self.world > 1:
            if self.device.type == "cpu":      # gloo (CPU tests)
                parts = [torch.zeros(self.rec, dtype=torch.int32)
                         for _ in range(self.world)]
                self.dist.all_gather(parts, self.sendbuf, group=self.group)
                self.recvbuf.copy_(torch.cat(parts))
            else:
                self.dist.all_gather_into_tensor(self.recvbuf, self.sendbuf,
                                                 group=self.group)
        else:
            self.recvbuf.copy_(self.sendbuf)
        rec = self.recvbuf.view(self.world, self.rec)
        torch.cat([rec[p, :self.words[p]] for p in range(self.world)],
                  out=self.gbits[:self.total_words])
        tails = rec[:, self.max_words:self.max_words + 2].to("cpu")   # one D2H
        lo = tails[:, 0].to(torch.int64) & 0xffffffff
        hi = tails[:, 1].to(torch.int64) & 0xffffffff
        total = int((lo + (hi << 32)).sum())
        return self.gbits, total


class PeerExchange(object):
    """The library's own exchange (include/graphblast_b200.h, gb200_xchg_*): every
    rank maps every other rank's exchange block through CUDA IPC; the owner's
    kernel stores its frontier slice, count and epoch flag into all peers over
    NVLink, and the whole traversal runs as one cooperative kernel per GPU
    (gb200_dist_bfs_fused).  torch.distributed is used once, to pass the 64-byte
    IPC handles around."""

    def __init__(self, gb, comm, device, offsets=None):
        """offsets: partition of the replicated array in 32-bit words; default =
        the bitmap partition (one bit per vertex), pass the vertex bounds for
        float payloads (one word per vertex)."""
        import torch.distributed as dist
        self.lib = gb._lib.load()
        self.world, self.rank = comm.world, comm.rank
        for p in range(self.world + 1):
            assert comm.bounds[p] % 32 == 0 or p == self.world
        if offsets is None:
            offsets = comm.offsets
        offs = (C.c_longlong * (self.world + 1))(*[int(o) for o in offsets])
        self._h = C.c_void_p()
        rc = self.lib.gb200_xchg_create(C.byref(self._h), self.world, self.rank,
                                        offs)
        if rc != 0:
            raise RuntimeError("gb200_xchg_create failed: %d" % rc)
        mine = (C.c_ubyte * 64)()
        rc = self.lib.gb200_xchg_handle(self._h, mine)
        if rc != 0:
            raise RuntimeError("gb200_xchg_handle failed: %d" % rc)
        t = torch.tensor(list(mine), dtype=torch.uint8, device=device)
        allh = torch.zeros(64 * self.world, dtype=torch.uint8, device=device)
        if self.world > 1:
            dist.all_gather_into_tensor(allh, t)
        else:
            allh.copy_(t)
        buf = allh.cpu().numpy().tobytes()
        rc = self.lib.gb200_xchg_connect(self._h, buf)
        if rc != 0:
            raise RuntimeError("gb200_xchg_connect failed: %d" % rc)

    def bfs(self, ops, n, source):
        levels = C.c_int(0)
        rc = self.lib.gb200_dist_bfs_fused(self._h, ops.v._h, ops.M._h, n, source,
                                           ops.desc._h, C.byref(levels))
        if rc != 0:
            raise RuntimeError("gb200_dist_bfs_fused failed: %d" % rc)
        return levels.value

    def pr(self, p_own, M, n, alpha, eps, desc):
        iters = C.c_int(0)
        rc = self.lib.gb200_dist_pr(self._h, p_own._h, M._h, n, alpha, eps,
                                    desc._h, C.byref(iters))
        if rc != 0:
            raise RuntimeError("gb200_dist_pr failed: %d" % rc)
        return iters.value

    def sssp(self, v_own, M, n, source, desc):
        rounds = C.c_int(0)
        rc = self.lib.gb200_dist_sssp(self._h, v_own._h, M._h, n, source,
                                      desc._h, C.byref(rounds))
        if rc != 0:
            raise RuntimeError("gb200_dist_sssp failed: %d" % rc)
        return rounds.value

    def close(self):
        if self._h:
            self.lib.gb200_xchg_free(self._h)
            self._h = C.c_void_p()


# ---------------------------------------------------------------------------
# Local operations through the C ABI (GPU)
# ---------------------------------------------------------------------------

class GpuLocalOps(object):
    """The owned slice's part of one BFS level, as GraphBLAS operations of this
    library: assign on the owned visited vector and a masked mxv with the
    rectangular local matrix."""

    def __init__(self, gb, n, lo, hi, rp_local, ci_local, colptr, rowind, desc):
        self.gb = gb
        self.n, self.lo, self.hi = n, lo, hi
        self.nl = hi - lo
        self.desc = desc
        dev = ci_local.device
        self._keep = [rp_local, ci_local, colptr, rowind]
        self.val = torch.ones(max(ci_local.numel(), 1), dtype=torch.float32,
                              device=dev)
        self.cscval = torch.ones(max(ci_local.numel(), 1), dtype=torch.float32,
                                 device=dev)
        self.M = gb.Matrix(max(self.nl, 1), n)
        if self.nl > 0 and ci_local.numel() > 0:
            self.M.build_device_csr(rp_local, ci_local, self.val,
                                    ci_local.numel(), colptr, rowind,
                                    self.cscval, symmetric=False)
            self.has_edges = True
        else:
            self.has_edges = False
        nl1 = max(self.nl, 1)
        self.v = gb.Vector(nl1)
        self.f_own = gb.Vector(nl1)
        self.f2 = gb.Vector(nl1)
        self.f_global = gb.Vector(n)
        self.lib = gb._lib.load()

    def reset(self):
        self.v.fill(0.0)

    def assign_level(self, gbits, word_lo, level):
        """v_own<f_own> = level, f_own = owned slice of the global frontier."""
        if self.nl == 0:
            return
        ptr = gbits.data_ptr() + 4 * word_lo
        rc = self.lib.gb200_vector_import_bits(self.f_own._h, C.c_void_p(ptr), -1)
        assert rc == 0, rc
        self.gb.assign(self.v, self.f_own, None, float(level), None, self.nl,
                       self.desc)

    def expand(self, gbits, gcount, comm):
        """f2_own<!v_own> = M (||.&&) f_global; the new owned frontier goes into
        comm's send record (bitmap words + device-side count, no host sync)."""
        if self.nl == 0 or not self.has_edges:
            comm.sendbuf.zero_()
            return
        rc = self.lib.gb200_vector_import_bits(self.f_global._h,
                                               C.c_void_p(gbits.data_ptr()),
                                               int(gcount))
        assert rc == 0, rc
        gb = self.gb
        self.desc.toggle(gb.Desc_field.GrB_MASK)
        try:
            gb.mxv(self.f2, self.v, None, gb.LogicalOrAndSemiring, self.M,
                   self.f_global, self.desc)
        finally:
            self.desc.toggle(gb.Desc_field.GrB_MASK)
        rc = self.lib.gb200_vector_export_bits_async(
            self.f2._h, C.c_void_p(comm.send_bits().data_ptr()),
            C.c_void_p(comm.count_ptr()))
        assert rc == 0, rc

    def levels(self):
        if self.nl == 0:
            return np.zeros(0, dtype=np.float32)
        return self.v.extractTuples()[:self.nl]


# ---------------------------------------------------------------------------
# Driver
# ---------------------------------------------------------------------------

def run_bfs(ops, comm, source, max_levels=10000):
    """Level-synchronous BFS over the 1-D partition.  Returns the number of
    levels executed."""
    bounds = comm.bounds
    rank = comm.rank
    lo = bounds[rank]
    word_lo = comm.offsets[rank]
    ops.reset()
    # level-1 frontier: the source, published by its owner through the exchange
    nw = comm.words[rank]
    seed = torch.zeros(max(nw, 1) + 8, dtype=torch.int32, device=comm.device)
    own = 1 if (bounds[rank] <= source < bounds[rank + 1]) else 0
    if own:
        rel = source - lo
        bit = rel & 31
        seed[rel >> 5] = (1 << bit) if bit < 31 else -(1 << 31)
    comm.set_host_record(seed, own)
    gbits, total = comm.exchange()
    level = 0
    while total > 0 and level < max_levels:
        level += 1
        ops.assign_level(gbits, word_lo, level)
        ops.expand(gbits, total, comm)
        gbits, total = comm.exchange()
    return level


def bench_distributed(args, world, rank, local_rank):
    """bench.py body for WORLD_SIZE > 1: strong scaling of the headline BFS
    (--algo pr: of PageRank, BASELINE.json configs[3])."""
    if args.algo == "pr":
        return bench_distributed_pr(args, world, rank, local_rank)
    if args.algo == "sssp":
        return bench_distributed_sssp(args, world, rank, local_rank)
    if args.algo != "bfs":
        raise SystemExit("--algo %s has no multi-GPU path (bfs, sssp, pr)" % args.algo)
    import os
    import sys
    import time
    import torch.distributed as dist
    import graphblast_b200 as gb
    from graphblast_b200 import graphs

    # keep stdout to the single JSON line: NCCL's banner goes to stderr
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)

    n = 1 << args.scale
    src, dst = graphs.rmat_edges(args.scale, args.edgefactor, seed=args.seed,
                                 device=dev)
    rowptr, colind = graphs.build_csr(n, src, dst, undirected=True)
    del src, dst
    nnz = int(colind.numel())
    deg = rowptr[1:] - rowptr[:-1]
    source = int(torch.argmax(deg).item())
    import os as _os
    bounds = partition_bounds(rowptr, world, row_weight=float(
        _os.environ.get("GB200_DIST_ROW_WEIGHT", "1e9")))
    lo, hi = bounds[rank], bounds[rank + 1]
    rp_l, ci_l, colptr, rowind = local_slice(rowptr, colind, lo, hi, n)
    h_rowptr = rowptr.cpu().numpy() if rank == 0 else None
    h_colind = colind.cpu().numpy() if rank == 0 else None
    nnz_local = int(ci_l.numel())
    del rowptr, colind, deg
    torch.cuda.empty_cache()

    desc = gb.Descriptor(mxvmode=0, struconly=1, opreuse=0, earlyexit=1)
    ops = GpuLocalOps(gb, n, lo, hi, rp_l, ci_l, colptr, rowind, desc)
    comm = Comm(bounds, dev)

    # Exchange: the library's peer-memory path unless it cannot be set up on some
    # rank (no IPC / peer access); then every rank takes the NCCL all-gather path.
    why = "failed on another rank"
    try:
        xchg = PeerExchange(gb, comm, dev)
    except Exception as e:               # noqa: BLE001
        why = str(e)
        xchg = None
    agree = torch.tensor([1 if xchg is not None else 0], device=dev)
    dist.all_reduce(agree, op=dist.ReduceOp.MIN)
    if int(agree.item()) == 0:
        if xchg is not None:
            xchg.close()
        xchg = None
        if rank == 0:
            print("peer exchange unavailable (%s): NCCL all-gather path" % why,
                  file=sys.stderr)

    def traverse():
        if xchg is not None:
            return xchg.bfs(ops, n, source)
        return run_bfs(ops, comm, source)

    torch.cuda.synchronize()
    dist.barrier()
    for _ in range(max(args.warmup, 1)):
        traverse()
    torch.cuda.synchronize()
    dist.barrier()

    lib = gb._lib.load()
    launches0 = C.c_ulonglong(0)
    lib.gb200_launch_count(C.byref(launches0))
    lib.gb200_profile_enable(1)
    lib.gb200_profile_reset()
    sampler = None
    try:
        from bench import ClockSampler, measured_peak_hbm
        sampler = ClockSampler(local_rank)
        sampler.start()
    except Exception:                        # noqa: BLE001
        measured_peak_hbm = lambda: (6650.0, "fallback (B200_PROFILING.md)")  # noqa: E731
    ev0 = torch.cuda.Event(enable_timing=True)
    ev1 = torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    dist.barrier()
    t0 = time.perf_counter()
    ev0.record()
    levels = 0
    for _ in range(args.steps):
        levels = traverse()
    ev1.record()
    torch.cuda.synchronize()
    wall_ms = (time.perf_counter() - t0) * 1e3
    clocks = sampler.stop() if sampler is not None else None
    dist.barrier()
    # fused Boolean pull on this rank: CUDA-event time and algorithmic bytes
    k_ms, k_n, k_b = C.c_double(0), C.c_longlong(0), C.c_double(0)
    lib.gb200_profile_read(1, C.byref(k_ms), C.byref(k_n), C.byref(k_b))
    lib.gb200_profile_enable(0)
    kern = torch.tensor([k_ms.value, float(k_n.value), k_b.value], device=dev,
                        dtype=torch.float64)
    kern_all = [torch.zeros_like(kern) for _ in range(world)]
    dist.all_gather(kern_all, kern)
    ms = torch.tensor([ev0.elapsed_time(ev1), wall_ms], device=dev)
    dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    launches1 = C.c_ulonglong(0)
    lib.gb200_launch_count(C.byref(launches1))
    ms_per_step = float(ms[0].item()) / args.steps

    # end to end: source id H2D, traversal, full level vector to rank 0's host memory
    gather = ResultGather(bounds, world, rank, dev)
    e2e_ms = timed_e2e(args, traverse, gather, ops.v, dev, 4)
    # parity: the gathered result against the CPU code (the checker lives in
    # bench.py: nothing in this package touches oracle/)
    host = gather.run(ops.v)
    parity = None
    cpu_baseline = None
    nnz_per_rank = torch.tensor([nnz_local], device=dev, dtype=torch.int64)
    gathered = [torch.zeros_like(nnz_per_rank) for _ in range(world)]
    dist.all_gather(gathered, nnz_per_rank)
    verify = getattr(args, "verify", None)
    if rank == 0 and verify is not None and not args.no_cpu_baseline:
        parity, cpu_baseline, _ = verify("bfs", h_rowptr, h_colind, host.numpy(),
                                         {"source": source})
    result = {
        "metric": "MTEPS", "value": nnz / (ms_per_step * 1e3),
        "unit": UNIT,
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_per_step, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {
            "workload": "direction-optimised BFS (LogicalOrAnd mxv, push<->pull) "
                        "on R-MAT scale-%d ef-%d seed %d, symmetrised"
                        % (args.scale, args.edgefactor, args.seed),
            "n": n, "nnz": nnz, "source": source, "levels": levels,
            "partition": "1-D row slices balanced on stored entries + %s per row, "
                         "bounds %s" % (_os.environ.get("GB200_DIST_ROW_WEIGHT", "1e9"), bounds),
            "nnz_per_rank": [int(g.item()) for g in gathered],
            "exchange": ("peer-memory stores of the owned frontier slice into "
                         "every rank's replica (CUDA IPC over NVLink), flag + "
                         "count per level, level loop in C++"
                         if xchg is not None else
                         "NCCL all-gather of the frontier bitmap (%d bytes per "
                         "level) + counts, level loop in Python"
                         % (4 * comm.rec * world)),
            "flags": "--struconly 1 --earlyexit 1; pull levels probe the "
                     "replicated cumulative visited bitmap (global operand reuse)"
                     if xchg is not None else
                     "--mxvmode 0 --struconly 1 --earlyexit 1 (opreuse off: the "
                     "visited mask is local)",
            "l2_policy": "inputs larger than L2"},
        "e2e": {"value": nnz / (e2e_ms * 1e3), "unit": "MTEPS",
                "ms_per_step": e2e_ms, "h2d_bytes_per_step": 4,
                "d2h_bytes_per_step": gather.d2h_bytes,
                "note": "per step: source id H2D, traversal, NCCL gather of the "
                        "owned level slices to rank 0 and the n-float result D2H "
                        "into rank 0's pinned memory; wall clock, max over ranks"},
        "gpu_launches": int(launches1.value - launches0.value),
        "cpu_baseline": cpu_baseline,
        "parity_vs_cpu_reference": parity,
    }
    # roofline of the dominant kernel on the slowest rank (same definition as N=1)
    slow = max(kern_all, key=lambda k: float(k[0].item()))
    s_ms, s_n, s_b = (float(slow[0].item()), float(slow[1].item()),
                      float(slow[2].item()))
    peak, peak_src = measured_peak_hbm()
    ach = (s_b / 1e9) / (s_ms / 1e3) if s_ms > 0 else 0.0
    result["roofline"] = {
        "kernel": "spmvMaskedOrPullKernel (fused Boolean pull), slowest rank",
        "bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s",
        "frac": ach / peak if peak else None, "peak_source": peak_src,
        "launches": int(s_n), "ms_per_launch": s_ms / s_n if s_n else 0.0,
        "bytes_per_launch": s_b / s_n if s_n else 0.0,
        "share_of_step": s_ms / (ms_per_step * args.steps) if ms_per_step else 0.0,
        "traffic": None}
    result["clocks"] = clocks
    if xchg is not None:
        xchg.close()
    dist.destroy_process_group()
    return result


def bench_distributed_pr(args, world, rank, local_rank):
    """PageRank (10 power iterations) over the 1-D row partition: local merge-path
    SpMV on the owned rows, p exchanged through peer memory after every mxv."""
    import os
    import sys
    import time
    import torch.distributed as dist
    import graphblast_b200 as gb
    from graphblast_b200 import graphs

    dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)
    alpha, niter = 0.85, 10
    n = 1 << args.scale
    src, dst = graphs.rmat_edges(args.scale, args.edgefactor, seed=args.seed,
                                 device=dev)
    rowptr, colind = graphs.build_csr(n, src, dst, undirected=True)
    del src, dst
    nnz = int(colind.numel())
    deg = (rowptr[1:] - rowptr[:-1]).to(torch.float32)
    bounds = partition_bounds(rowptr, world)
    lo, hi = bounds[rank], bounds[rank + 1]
    nl = hi - lo
    e0, e1 = int(rowptr[lo]), int(rowptr[hi])
    rp_l = (rowptr[lo:hi + 1] - rowptr[lo]).to(torch.int32).contiguous()
    ci_l = colind[e0:e1].contiguous()
    # (alpha * A ./ outdeg)^T restricted to the owned rows: entry (i, j) = alpha/deg(j)
    val_l = (alpha / deg[ci_l.to(torch.int64)]).contiguous()
    h_rowptr = rowptr.cpu().numpy() if rank == 0 else None
    h_colind = colind.cpu().numpy() if rank == 0 else None
    del rowptr, colind, deg
    torch.cuda.empty_cache()

    lib = gb._lib.load()
    M = gb.Matrix(max(nl, 1), n)
    M._keep = [rp_l, ci_l, val_l]
    rc = lib.gb200_matrix_adopt_csr(M._h, C.c_void_p(rp_l.data_ptr()),
                                    C.c_void_p(ci_l.data_ptr()),
                                    C.c_void_p(val_l.data_ptr()), int(ci_l.numel()))
    assert rc == 0, rc
    p_own = gb.Vector(max(nl, 1))
    desc = gb.Descriptor(mxvmode=0, max_niter=niter)
    comm = Comm(bounds, dev)
    xchg = PeerExchange(gb, comm, dev, offsets=bounds)

    torch.cuda.synchronize()
    dist.barrier()
    for _ in range(max(args.warmup, 1)):
        xchg.pr(p_own, M, n, alpha, 0.0, desc)
    torch.cuda.synchronize()
    dist.barrier()
    launches0 = C.c_ulonglong(0)
    lib.gb200_launch_count(C.byref(launches0))
    lib.gb200_profile_enable(1)
    lib.gb200_profile_reset()
    sampler = None
    try:
        from bench import ClockSampler
        sampler = ClockSampler(local_rank)
        sampler.start()
    except Exception:                        # noqa: BLE001
        sampler = None
    ev0 = torch.cuda.Event(enable_timing=True)
    ev1 = torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    ev0.record()
    iters = 0
    for _ in range(args.steps):
        iters = xchg.pr(p_own, M, n, alpha, 0.0, desc)
    ev1.record()
    torch.cuda.synchronize()
    wall_ms = (time.perf_counter() - t0) * 1e3
    clocks = sampler.stop() if sampler is not None else None
    dist.barrier()
    ms = torch.tensor([ev0.elapsed_time(ev1), wall_ms], device=dev)
    dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    launches1 = C.c_ulonglong(0)
    lib.gb200_launch_count(C.byref(launches1))
    ms_per_step = float(ms[0].item()) / args.steps
    # merge-kernel time on this rank (CUDA events inside the library)
    k_ms, k_n, k_b = C.c_double(0), C.c_longlong(0), C.c_double(0)
    lib.gb200_profile_read(0, C.byref(k_ms), C.byref(k_n), C.byref(k_b))
    kern = torch.tensor([k_ms.value / max(k_n.value, 1),
                         k_b.value / max(k_n.value, 1)], device=dev,
                        dtype=torch.float64)
    kern_all = [torch.zeros_like(kern) for _ in range(world)]
    dist.all_gather(kern_all, kern)

    gather = ResultGather(bounds, world, rank, dev)
    e2e_ms = timed_e2e(args, lambda: xchg.pr(p_own, M, n, alpha, 0.0, desc), gather,
                       p_own, dev, 4)
    host = gather.run(p_own)
    parity = None
    max_rel = None
    cpu_baseline = None
    pr_check = None
    verify = getattr(args, "verify", None)
    if rank == 0 and verify is not None and not args.no_cpu_baseline:
        parity, cpu_baseline, pr_check = verify("pr", h_rowptr, h_colind, host.numpy(),
                                                {"alpha": alpha, "niter": niter})
        max_rel = pr_check.get("max_rel_err_vs_reference") if pr_check else None
    from json import loads
    peak = None
    try:
        with open(os.path.join(os.path.dirname(os.path.dirname(
                os.path.abspath(__file__))), "MEASURED_PEAKS.json")) as f:
            peak = float(loads(f.read()).get("hbm_gbs"))
    except Exception:                        # noqa: BLE001
        peak = 7700.0
    slow = max(float(k[0].item()) for k in kern_all)
    ach = max(float(k[1].item()) for k in kern_all) / (slow * 1e-3) / 1e9 if slow > 0 else 0.0
    result = {
        "metric": "MTEPS", "value": nnz / (ms_per_step * 1e3),
        "unit": UNIT,
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_per_step, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {
            "workload": "PageRank (PlusMultiplies mxv, %d iterations) on R-MAT "
                        "scale-%d ef-%d seed %d, symmetrised"
                        % (niter, args.scale, args.edgefactor, args.seed),
            "n": n, "nnz": nnz, "iterations": iters,
            "partition": "1-D nnz-balanced row slices, bounds %s" % bounds,
            "exchange": "peer-memory stores of the owned float slice into every "
                        "rank's replica (CUDA IPC over NVLink) + residual partial "
                        "per iteration, loop in C++",
            "l2_policy": "inputs larger than L2"},
        "e2e": {"value": nnz / (e2e_ms * 1e3), "unit": "MTEPS",
                "ms_per_step": e2e_ms, "h2d_bytes_per_step": 4,
                "d2h_bytes_per_step": gather.d2h_bytes,
                "note": "per step: one PageRank run, NCCL gather of the owned rank "
                        "slices to rank 0 and the n-float result D2H into rank 0's "
                        "pinned memory; wall clock, max over ranks"},
        "gpu_launches": int(launches1.value - launches0.value),
        "roofline": {"kernel": "spmvMergeKernel (merge-path pull SpMV), slowest rank",
                     "bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s",
                     "frac": ach / peak if peak else None, "traffic": None,
                     "ms_per_launch": slow},
        "cpu_baseline": cpu_baseline,
        "parity_vs_cpu_reference": parity,
        "max_rel_err": max_rel, "pagerank_check": pr_check,
        "clocks": clocks,
    }
    xchg.close()
    dist.destroy_process_group()
    return result


def weighted_local_matrix(gb, n, rowptr, colind, cscval, lo, hi):
    """(owned x n) matrix of the owned rows of A^T with weights: CSR entries
    (j_owned, i) = A(i, j) = cscval of the symmetric structure's entry, CSC = the
    same entries by source column.  Returns (Matrix, tensors to keep alive)."""
    rp_l, ci_l, colptr, rowind, order = local_slice(rowptr, colind, lo, hi, n,
                                                    return_order=True)
    e0, e1 = int(rowptr[lo]), int(rowptr[hi])
    val_l = cscval[e0:e1].contiguous()
    cval_l = val_l[order].contiguous()
    nl = hi - lo
    M = gb.Matrix(max(nl, 1), n)
    if nl > 0 and ci_l.numel() > 0:
        M.build_device_csr(rp_l, ci_l, val_l, ci_l.numel(), colptr, rowind, cval_l,
                           symmetric=False)
    return M, [rp_l, ci_l, colptr, rowind, val_l, cval_l]


def bench_distributed_sssp(args, world, rank, local_rank):
    """SSSP over the 1-D row partition (gb200_dist_sssp): frontier values exchanged
    through peer memory after every mxv, direction chosen per round by mxv."""
    import os
    import sys
    import time
    import torch.distributed as dist
    import graphblast_b200 as gb
    from graphblast_b200 import graphs

    dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)
    n = 1 << args.scale
    src, dst = graphs.rmat_edges(args.scale, args.edgefactor, seed=args.seed,
                                 device=dev)
    rowptr, colind = graphs.build_csr(n, src, dst, undirected=True)
    del src, dst
    nnz = int(colind.numel())
    deg = rowptr[1:] - rowptr[:-1]
    source = int(torch.argmax(deg).item())
    w = gb.api.host_uniform_weights(args.seed, 1, 64, nnz)
    d_w = torch.from_numpy(w).to(dev)
    d_wt = graphs.transpose_values(n, rowptr, colind, d_w)
    bounds = partition_bounds(rowptr, world)
    lo, hi = bounds[rank], bounds[rank + 1]
    nl = hi - lo
    M, keep = weighted_local_matrix(gb, n, rowptr, colind, d_wt, lo, hi)
    h_rowptr = rowptr.cpu().numpy() if rank == 0 else None
    h_colind = colind.cpu().numpy() if rank == 0 else None
    del rowptr, colind, deg, d_w, d_wt
    torch.cuda.empty_cache()

    lib = gb._lib.load()
    v_own = gb.Vector(max(nl, 1))
    desc = gb.Descriptor(mxvmode=0, switchpoint=0.025)
    comm = Comm(bounds, dev)
    xchg = PeerExchange(gb, comm, dev, offsets=bounds)
    torch.cuda.synchronize()
    dist.barrier()
    for _ in range(max(args.warmup, 1)):
        xchg.sssp(v_own, M, n, source, desc)
    torch.cuda.synchronize()
    dist.barrier()
    launches0 = C.c_ulonglong(0)
    lib.gb200_launch_count(C.byref(launches0))
    lib.gb200_profile_enable(1)
    lib.gb200_profile_reset()
    sampler = None
    try:
        from bench import ClockSampler, measured_peak_hbm
        sampler = ClockSampler(local_rank)
        sampler.start()
    except Exception:                        # noqa: BLE001
        measured_peak_hbm = lambda: (6650.0, "fallback (B200_PROFILING.md)")  # noqa: E731
    ev0 = torch.cuda.Event(enable_timing=True)
    ev1 = torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    ev0.record()
    rounds = 0
    for _ in range(args.steps):
        rounds = xchg.sssp(v_own, M, n, source, desc)
    ev1.record()
    torch.cuda.synchronize()
    wall_ms = (time.perf_counter() - t0) * 1e3
    clocks = sampler.stop() if sampler is not None else None
    dist.barrier()
    ms = torch.tensor([ev0.elapsed_time(ev1), wall_ms], device=dev)
    dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    launches1 = C.c_ulonglong(0)
    lib.gb200_launch_count(C.byref(launches1))
    ms_per_step = float(ms[0].item()) / args.steps
    k_ms, k_n, k_b = C.c_double(0), C.c_longlong(0), C.c_double(0)
    lib.gb200_profile_read(0, C.byref(k_ms), C.byref(k_n), C.byref(k_b))
    lib.gb200_profile_enable(0)
    kern = torch.tensor([k_ms.value, float(k_n.value), k_b.value], device=dev,
                        dtype=torch.float64)
    kern_all = [torch.zeros_like(kern) for _ in range(world)]
    dist.all_gather(kern_all, kern)

    gather = ResultGather(bounds, world, rank, dev)
    e2e_ms = timed_e2e(args, lambda: xchg.sssp(v_own, M, n, source, desc), gather,
                       v_own, dev, 4)
    host = gather.run(v_own)
    parity = None
    cpu_baseline = None
    verify = getattr(args, "verify", None)
    if rank == 0 and verify is not None and not args.no_cpu_baseline:
        parity, cpu_baseline, _ = verify("sssp", h_rowptr, h_colind, host.numpy(),
                                         {"source": source, "weights": w})
    slow = max(kern_all, key=lambda k: float(k[0].item()))
    s_ms, s_n, s_b = (float(slow[0].item()), float(slow[1].item()),
                      float(slow[2].item()))
    peak, peak_src = measured_peak_hbm()
    ach = (s_b / 1e9) / (s_ms / 1e3) if s_ms > 0 else 0.0
    result = {
        "metric": "MTEPS", "value": nnz / (ms_per_step * 1e3),
        "unit": UNIT,
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_per_step, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {
            "workload": "SSSP (MinimumPlus mxv, push<->pull) on R-MAT scale-%d "
                        "ef-%d seed %d, symmetrised, uniform integer weights 1..64"
                        % (args.scale, args.edgefactor, args.seed),
            "n": n, "nnz": nnz, "source": source, "rounds": rounds,
            "partition": "1-D nnz-balanced row slices, bounds %s" % bounds,
            "exchange": "peer-memory stores of the owned frontier values into every "
                        "rank's replica (CUDA IPC over NVLink) + improved count per "
                        "round, loop in C++",
            "l2_policy": "inputs larger than L2"},
        "e2e": {"value": nnz / (e2e_ms * 1e3), "unit": "MTEPS",
                "ms_per_step": e2e_ms, "h2d_bytes_per_step": 4,
                "d2h_bytes_per_step": gather.d2h_bytes,
                "note": "per step: source id H2D, traversal, NCCL gather of the "
                        "owned distance slices to rank 0 and the n-float result D2H "
                        "into rank 0's pinned memory; wall clock, max over ranks"},
        "gpu_launches": int(launches1.value - launches0.value),
        "roofline": {"kernel": "spmvMergeKernel (merge-path pull SpMV), slowest rank",
                     "bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s",
                     "frac": ach / peak if peak else None, "peak_source": peak_src,
                     "launches": int(s_n),
                     "ms_per_launch": s_ms / s_n if s_n else 0.0, "traffic": None},
        "cpu_baseline": cpu_baseline,
        "parity_vs_cpu_reference": parity,
        "clocks": clocks,
    }
    xchg.close()
    dist.destroy_process_group()
    return result
