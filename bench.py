#!/usr/bin/env python
"""bench.py — Mnodes/s of the GPU-offloaded tree search on B200, BASELINE.json's metric.

HEADLINE (value / e2e / roofline, BASELINE configs[1]): the N-Queens N=17 search with the reference's defaults
g=1 m=25 --M 50000.  A *step* is one whole search; Mnodes/s = explored tree / time, the quantity the reference
prints (nqueens_gpu_chpl.chpl:39-46).  Every step the explored tree and the solution count are checked against
the reference's (8 017 021 931 / 95 815 104).
  value : step 2 (the offload loop, nqueens_gpu_chpl.chpl:197-215) with the warm-up pool already resident in HBM
          on pre-created handles — what the search driver does: the pool split (the reference's strided split) into
          four device pools, tsb_nq_pool_run_multi until all are dry (a dry pool takes half of the fullest), CUDA
          events around it; children produced / event time
  e2e   : the whole search through the reference-facing C-ABI call with host inputs and outputs
          (tsb_nq_search_on: step 1 on the CPU, the warm-up pool copied host->device, all rounds, the leftover
          nodes and the counters copied device->host, step 3 on the CPU), wall clock; explored tree / time
  roofline : nq_rounds_ll_kernel, the one kernel of that timed region: 21 B read per parent + 21 B written per child
          (= 42 B per explored node) / event time.  At --M 50000 a round moves ~2 MB and is bound by the L2 round
          trips that order it after the previous round, not by HBM; the bandwidth-bound kernels are listed
          under "kernels" with their own fractions
  N > 1 (torchrun) : the same search split over N GPUs (static split of the warm-up pool + stealing between the
          device pools over NVLink), driven by rank 0 in one process with one host thread per GPU, as the
          reference's multi-GPU driver is one process with one task per GPU; the other ranks hold their GPU and
          the NCCL barrier.  scaling = strong (the tree is fixed).
SECONDARY (same line):
  batch   : the batch evaluators of round 1 — device-resident value, host-buffer e2e (registered arrays, zero-copy
            over PCIe) and HBM roofline of tsb_nq_evaluate (N=17, --big-M and 50000 parents), tsb_pfsp_evaluate
            lb1 (ta014) and lb2 (ta020); with N > 1 ranks every rank evaluates its own batch (weak scaling)
  search  : other whole searches on pre-created handles: N=17 at --big-M (two bandwidth-bound kernels per round),
            PFSP ta014/lb1 and ta020/lb2 at --M 50000 (BASELINE configs 2-3), ta020/lb1_d with the Chapel min_heads
            (836 490 312 nodes); at N = 8: N=19 --D 8 (BASELINE configs[4])
  kernels : per kernel: us per launch, achieved GB/s, fraction of the measured HBM peak, DRAM traffic of the ncu
            capture under profiles/ (parsed at run time)
  cpu_baseline : the reference's own sequential search code (oracle/_ref: nqueens_c.c's pool / isSafe / decompose)
            on all host cores (subtrees handed out dynamically) and on one core

`--impl reference`: the reference's CPU search on all host threads as its own arm; each step is a bounded sample of
the workload (the whole N=16 / 15 / 14 search, by core count: the same code per node, 1/7 .. 1/300 of the tree).

`--dump-outputs DIR`: after the headline's timed steps, what its last step returned, so that two builds can be
compared output for output (the inputs are the same every run: the warm-up pool of step 1 is deterministic):
  step2_pools    float64 [pools, 5] of the resident-pool offload loop (1 GPU): per device pool the rounds, parents
                 popped, children pushed and solutions that tsb_nq_pool_run_multi returned over the step, and the
                 nodes left in the pool when all pools held fewer than m
  search_counts  float64 [explored tree, solutions] of the last whole search (the only file with N > 1)
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "gpu-accelerated-tree-search-chapel_b200")
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)

L2_BYTES = 126 * 2**20

# explored-tree nodes per depth of the N=17 search = depth histogram of the parents its offload loop evaluates
# (exact counts, tests/golden/nqueens_depth_hist.json; sum over depths 1..17 = 8 017 021 931 = exploredTree)
_HIST_PATH = os.path.join(ROOT, "tests", "golden", "nqueens_depth_hist.json")
# SURVEY.md Appendix C: depth histogram of offloaded parents, ta014 lb1 (depth: count)
PFSP_TA014_LB1_HIST = {1: 1, 2: 39, 3: 165, 4: 639, 5: 2252, 6: 7003, 7: 19626, 8: 50445, 9: 116575, 10: 231523,
                       11: 366493, 12: 464303, 13: 466099, 14: 366546, 15: 240078, 16: 144463, 17: 72917,
                       18: 21829, 19: 2648}


# SURVEY.md Appendix C: depth histogram of offloaded parents, ta020 lb2
PFSP_TA020_LB2_HIST = {1: 8, 2: 92, 3: 597, 4: 3538, 5: 17546, 6: 71163, 7: 224227, 8: 533085, 9: 947932, 10: 1193333,
                       11: 1044659, 12: 572606, 13: 205065, 14: 47233, 15: 7546, 16: 1526, 17: 208, 18: 13}


# ----------------------------------------------------------------------------------------- synthetic inputs
def nq_depth_hist(N):
    with open(_HIST_PATH) as f:
        h = json.load(f)[str(N)]
    return {int(k): int(v) for k, v in h.items()}


def synth_nq_parents(N, count, seed, dtype):
    """parents as the reference's pool holds them: board[0..depth) a conflict-free placement (random walk of
    the search tree), board[depth..N) the remaining values in random order; depth ~ explored-tree histogram"""
    rng = np.random.default_rng(seed)
    hist = nq_depth_hist(N)
    depths = np.array(sorted(hist), dtype=np.int64)
    prob = np.array([hist[int(d)] for d in depths], dtype=np.float64)
    base = min(count, 1 << 18)  # distinct random walks; replicated by random gather up to `count`
    target = rng.choice(depths, size=base, p=prob / prob.sum())
    board = np.zeros((base, 20), dtype=np.uint8)
    todo = np.arange(base)
    full = (1 << N) - 1
    while todo.size:
        n = todo.size
        cols = np.zeros(n, dtype=np.int64)
        ld = np.zeros(n, dtype=np.int64)
        rd = np.zeros(n, dtype=np.int64)
        ok = np.ones(n, dtype=bool)
        tgt = target[todo]
        rows = np.zeros((n, N), dtype=np.uint8)
        for r in range(int(tgt.max())):
            act = ok & (tgt > r)
            free = ~(cols | ld | rd) & full
            act &= free != 0
            ok &= (tgt <= r) | (free != 0)
            # choose a uniformly random set bit of `free`
            cnt = np.zeros(n, dtype=np.int64)
            for b in range(N):
                cnt += (free >> b) & 1
            pick = (rng.random(n) * np.maximum(cnt, 1)).astype(np.int64)
            chosen = np.zeros(n, dtype=np.int64)
            seen = np.zeros(n, dtype=np.int64)
            for b in range(N):
                bit = (free >> b) & 1
                hit = (bit == 1) & (seen == pick)
                chosen = np.where(hit, b, chosen)
                seen += bit
            bitv = np.where(act, 1 << chosen, 0)
            rows[:, r] = np.where(act, chosen, 0)
            cols |= bitv
            ld = ((ld | bitv) << 1) & full
            rd = (rd | bitv) >> 1
        done = ok
        idx = todo[done]
        # remaining values in random order after the placed prefix
        for i, src in zip(idx, np.nonzero(done)[0]):
            d = int(target[i])
            placed = rows[src, :d]
            rest = np.setdiff1d(np.arange(N, dtype=np.uint8), placed)
            board[i, :d] = placed
            board[i, d:N] = rng.permutation(rest)
        todo = todo[~done]
    sel = rng.integers(0, base, size=count) if count > base else np.arange(count)
    out = np.zeros(count, dtype=dtype)
    out["depth"] = target[sel]
    out["board"] = board[sel]
    return out


def synth_pfsp_parents(count, seed, dtype, hist=PFSP_TA014_LB1_HIST, jobs=20):
    rng = np.random.default_rng(seed)
    depths = np.array(sorted(hist), dtype=np.int64)
    prob = np.array([hist[int(d)] for d in depths], dtype=np.float64)
    d = rng.choice(depths, size=count, p=prob / prob.sum())
    out = np.zeros(count, dtype=dtype)
    out["depth"] = d
    out["limit1"] = d - 1
    out["prmu"][:, :jobs] = np.argsort(rng.random((count, jobs)), axis=1).astype(np.int32)
    return out


# ----------------------------------------------------------------------------------------- clocks
class ClockSampler:
    """samples SM clock and throttle reasons of one GPU while a timed region runs (NVML)"""

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _run(self):
        nv = self.nv
        names = {"hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40,
                 "sw_power_cap": 0x4, "hw_power_brake": 0x80}
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            self._stop.wait(0.02)

    def __enter__(self):
        if self.nv:
            self._thread = threading.Thread(target=self._run, daemon=True)
            self._thread.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self._thread:
            self._thread.join()

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["nvml_unavailable"]}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


# ----------------------------------------------------------------------------------------- distributed helpers
def dist_env():
    return int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))


def dist_init(backend):
    import torch.distributed as dist
    _, local_rank, world = dist_env()
    if world > 1 and not dist.is_initialized():
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29511")
        if backend == "nccl":
            import torch
            torch.cuda.set_device(local_rank)
            dist.init_process_group(backend=backend, device_id=torch.device(f"cuda:{local_rank}"))
        else:
            dist.init_process_group(backend=backend)
    return world


_CPU_GROUP = None


def dist_barrier(world, cpu=False):
    """cpu=True: wait on the host (a gloo group).  An NCCL barrier is a kernel that spins on every waiting rank's
    GPU — while rank 0 drives all GPUs through a multi-GPU search that would take SMs away from the search."""
    global _CPU_GROUP
    if world > 1:
        import torch.distributed as dist
        if cpu and dist.get_backend() != "gloo":
            if _CPU_GROUP is None:
                _CPU_GROUP = dist.new_group(backend="gloo")
            dist.barrier(group=_CPU_GROUP)
        else:
            dist.barrier()


def dist_max_sum(world, t_seconds, units, device):
    """(max over ranks of t_seconds, sum over ranks of units)"""
    if world <= 1:
        return t_seconds, units
    import torch
    import torch.distributed as dist
    t = torch.tensor([t_seconds], dtype=torch.float64, device=device)
    u = torch.tensor([float(units)], dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dist.all_reduce(u, op=dist.ReduceOp.SUM)
    return float(t.item()), float(u.item())



N_HEAD, M_HEAD, m_HEAD = 17, 50000, 25
GOLDEN_NQ = {12: (856188, 14200), 13: (4674889, 73712), 14: (27358552, 365596), 15: (171129071, 2279184),
             16: (1141190302, 14772512), 17: (8017021931, 95815104), 18: (59365844490, 666090624),
             19: (461939618823, 4968057848)}  # tests/golden/counts.json (reference binaries) + known solution counts
GOLDEN_PFSP = {(14, "lb1"): (2573652, 2648, 1377), (20, "lb2"): (4870386, 0, 1591),
               (20, "lb1_d"): (836490312, 3764, 1591)}  # (20, lb1_d): Chapel min_heads semantics (SURVEY A.1)
NODE_BYTES = 42  # 21 B read per parent + 21 B written per child: algorithmic HBM bytes per explored node


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def make_config(gpus, M=M_HEAD):
    return {"workload": f"N-Queens N={N_HEAD} g=1 m={m_HEAD} --M {M}: whole search, Mnodes/s = explored tree / time "
                        "(BASELINE configs[1]; the reference's default chunk size)",
            "N": N_HEAD, "g": 1, "m": m_HEAD, "M": M,
            "parallelism": f"{gpus} GPU(s): static split of the warm-up pool over the GPUs (one task per GPU, as the "
                           "reference's --D) and, on each GPU, once more into 4 device pools whose rounds (chunks of "
                           "<= M parents each, popBackBulk(m, M) per pool) share every launch of the persistent kernel; "
                           "stealing between device pools.  TSB200_POOLS=1: one pool per GPU (the reference's D = 1 "
                           "chunk sequence, 0.74 s per search instead of 0.41 s)",
            "pools_per_gpu": 4,
            "l2": "every step streams its whole pool through HBM (8.0 G nodes x 42 B >> the 126 MB L2); no buffer "
                  "is reused between steps"}


# ----------------------------------------------------------------------------------------- our arm
def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic(kernel_substr, files):
    """dram__bytes_read.sum + dram__bytes_write.sum of the first kernel whose name contains `kernel_substr` in the
    ncu summaries under profiles/ (newest round first); None if there is no capture"""
    import re
    unit = {"byte": 1, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    for f in files:
        path = os.path.join(ROOT, "profiles", f)
        if not os.path.exists(path):
            continue
        cur, got = None, {}
        for line in open(path):
            if line.startswith("kernel:"):
                if got:
                    break
                cur, got = (line if kernel_substr in line else None), {}
            elif cur:
                mm = re.match(r"\s+dram__bytes_(read|write)\.sum\s+([\d.]+)\s+(\w+)", line)
                if mm:
                    got[mm.group(1)] = float(mm.group(2)) * unit.get(mm.group(3), 1)
        if "read" in got:  # (the summaries leave out counters that are 0)
            return {"bytes": got["read"] + got.get("write", 0.0), "source": f"profiles/{f}"}
    return None


def run_headline_1gpu(steps, warmup, device_index, M=M_HEAD, N=N_HEAD):
    """value (step 2 on a resident pool, CUDA events) and e2e (whole search through the C ABI) on one GPU"""
    import torch

    import tsb200
    dev = torch.device(f"cuda:{device_index}")
    torch.cuda.set_device(dev)
    t_c0 = time.perf_counter()
    ev = tsb200.NQueensEvaluator(N, 1, M, device=device_index)
    t_create = time.perf_counter() - t_c0
    # pools per GPU: what the search driver uses (tsb_host.cpp nq_pools_of): the task's warm-up pool is split once more
    # (the reference's strided split) into P device pools whose rounds share every launch of the persistent kernel
    P = max(1, min(int(os.environ.get("TSB200_POOLS", "4")), ev.pools_per_launch(M)))
    evs = [ev] + [tsb200.NQueensEvaluator(N, 1, M, device=device_index) for _ in range(P - 1)]
    warm, wtree, wsol = tsb200.nqueens_warmup(N, P * m_HEAD)
    c = warm.shape[0] // P
    parts = [np.ascontiguousarray(warm[g:P * c:P]) for g in range(P)]
    parts[-1] = np.ascontiguousarray(np.concatenate([parts[-1], warm[P * c:]]))  # static_split's remainder rule
    floor = 2 * m_HEAD  # steal_floor of the persistent kernel's range

    def step2():
        """the driver's step 2 on resident pools (nq_devpool_multi_rounds): shared launches, dry pools take the oldest
        half of the fullest one; -> [rounds, parents, children, solutions] per pool"""
        per = [[0, 0, 0, 0] for _ in evs]
        while True:
            sizes = [e.pool_size for e in evs]
            for i, e in enumerate(evs):
                if sizes[i] < m_HEAD:
                    v = max(range(P), key=lambda j: sizes[j])
                    if v != i and sizes[v] >= floor:
                        e.pool_steal_from(evs[v], m_HEAD)
                        sizes = [x.pool_size for x in evs]
            if max(sizes) < m_HEAD:
                return per
            for i, r in enumerate(tsb200.nqueens_pool_run_multi(evs, m_HEAD, M, 2048)):
                per[i] = [a + b for a, b in zip(per[i], r)]

    stream = torch.cuda.ExternalStream(ev.stream, device=dev)
    want = GOLDEN_NQ[N]
    for _ in range(warmup):
        st = ev.search(m_HEAD, M)
        assert (st.explored_tree, st.explored_sol) == want, "search counts differ from the reference's"
    # ---- value: the offload loop on a pool that is already in HBM
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_dev, nodes, rounds = 0.0, 0, 0
    n_launches = lambda: sum(e.kernel_launches for e in evs)  # noqa: E731
    l0 = n_launches()
    torch.cuda.synchronize()
    with ClockSampler(device_index) as clk:
        for _ in range(steps):
            for e, part in zip(evs, parts):
                e.pool_push(part)
            torch.cuda.synchronize()
            launches_before = n_launches()
            # (every launch inside is followed by a stream synchronisation, so the two events bracket all of it
            # whichever pool's stream a launch went to)
            e0.record(stream)
            per = step2()
            e1.record(stream)
            torch.cuda.synchronize()
            t_dev += e0.elapsed_time(e1) / 1e3
            nr, _, nc, ns = (sum(p[k] for p in per) for k in range(4))
            nodes += nc
            rounds += nr
            launches_per_step = n_launches() - launches_before
            left = [e.pool_drain().shape[0] for e in evs]
            assert wtree + nc + sum(left) <= want[0] and ns + wsol <= want[1]
        launches = n_launches() - l0
        # ---- e2e: the whole search, host in / host out
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        tree = 0
        for _ in range(steps):
            st = ev.search(m_HEAD, M)
            tree += st.explored_tree
            assert (st.explored_tree, st.explored_sol) == want, "search counts differ from the reference's"
        torch.cuda.synchronize()
        t_e2e = time.perf_counter() - t0
    for e in evs:
        e.close()
    outputs = {"step2_pools": np.array([p + [n] for p, n in zip(per, left)], dtype=np.float64),
               "search_counts": np.array([st.explored_tree, st.explored_sol], dtype=np.float64)}
    return {"pools": P, "t_dev": t_dev, "nodes": nodes, "rounds": rounds, "t_e2e": t_e2e, "tree": tree, "launches": launches,
            "launches_per_step": launches_per_step, "clocks": clk.summary(), "create_ms": t_create * 1e3,
            "h2d": warm.nbytes, "d2h": 64 + P * m_HEAD * 21, "offloads": int(st.offloads), "steps": steps,
            "outputs": outputs}


def run_headline_multi(steps, warmup, world, rank, M=M_HEAD, N=N_HEAD):
    """N > 1: rank 0 drives all `world` GPUs in one process (one host thread, handle and device pool per GPU, the
    reference's multi-GPU structure); the other ranks keep their GPU busy with nothing and meet rank 0 at barriers"""
    import torch

    import tsb200
    dev = torch.device(f"cuda:{rank}")
    out = None
    dist_barrier(world)
    torch.cuda.synchronize(dev)
    dist_barrier(world, cpu=True)  # from here on the waiting ranks leave their GPUs alone
    if rank == 0:
        want = GOLDEN_NQ[N]
        for _ in range(warmup):
            st = tsb200.nqueens_search_device(N, 1, m_HEAD, M, world)
            assert (st.explored_tree, st.explored_sol) == want
        t2, tree, launches, steals = 0.0, 0, 0, 0
        shares = None
        with ClockSampler(0) as clk:
            t0 = time.perf_counter()
            for _ in range(steps):
                st = tsb200.nqueens_search_device(N, 1, m_HEAD, M, world)
                assert (st.explored_tree, st.explored_sol) == want, "search counts differ from the reference's"
                t2 += st.t_step2
                tree += st.explored_tree
                launches += st.kernel_launches
                steals += st.steals
                shares = [st.per_gpu_tree[i] / st.explored_tree for i in range(world)]
            t_e2e = time.perf_counter() - t0
        out = {"t_dev": t2, "nodes": tree, "t_e2e": t_e2e, "tree": tree, "launches": launches, "clocks": clk.summary(),
               "launches_per_step": launches // steps, "rounds": int(st.offloads) * steps, "offloads": int(st.offloads),
               "steps": steps, "h2d": 21 * m_HEAD * 4 * world, "d2h": (64 + 21 * m_HEAD * 4) * world, "steals": steals / steps,
               "pools": 4,
               "per_gpu_share": shares, "create_ms": None,
               "outputs": {"search_counts": np.array([st.explored_tree, st.explored_sol], dtype=np.float64)}}
    dist_barrier(world, cpu=True)
    return out


def run_workload(kind, M, steps, warmup, device_index, world, N=17):
    """one batch-evaluation workload at chunk size M: device-resident launches (CUDA events) and the host-buffer C-ABI call"""
    import torch

    import tsb200
    dev = torch.device(f"cuda:{device_index}")
    torch.cuda.set_device(dev)
    rank, _, _ = dist_env()
    if kind == "nq":
        in_rec, out_rec = 21, N
        make = lambda seed: synth_nq_parents(N, M, seed, tsb200.NQ_NODE_DTYPE)  # noqa: E731
        ev = tsb200.NQueensEvaluator(N, 1, M, device=device_index)
        call_dev = lambda i, o, s: ev.evaluate_device(i, M, o, s)  # noqa: E731
        out_dtype, out_elems = np.uint8, M * N
        call_host = lambda par, out: ev.evaluate_gpu(par, M * N, out)  # noqa: E731
    else:
        in_rec, out_rec = 88, 80
        inst, lb, best, hist = (14, "lb1", 1377, PFSP_TA014_LB1_HIST) if kind == "pfsp" else \
            (20, "lb2", 1591, PFSP_TA020_LB2_HIST)
        make = lambda seed: synth_pfsp_parents(M, seed, tsb200.PFSP_NODE_DTYPE, hist)  # noqa: E731
        ev = tsb200.PfspEvaluator(inst, M=M, device=device_index)
        call_dev = lambda i, o, s: ev.evaluate_device(lb, i, M, best, o, s)  # noqa: E731
        out_dtype, out_elems = np.int32, M * 20
        call_host = lambda par, out: ev.evaluate_gpu(par, M * 20, best, lb, out)  # noqa: E731
    bytes_per_set = M * (in_rec + out_rec)
    nsets = max(2, int(np.ceil(2.5 * L2_BYTES / bytes_per_set)))  # rotate over > 2.5x L2 of distinct buffers
    nsets = min(nsets, 64)
    base = make(1234 + rank)
    host_in = [base] + [np.roll(base, 7919 * (k + 1), axis=0) for k in range(min(nsets, 4) - 1)]
    d_in = [torch.from_numpy(host_in[k % len(host_in)].view(np.uint8).reshape(-1)).to(dev) for k in range(nsets)]
    d_out = [torch.empty(M * out_rec, dtype=torch.uint8, device=dev) for _ in range(nsets)]
    tstream = torch.cuda.Stream(device=dev)  # the kernels are launched on it and the CUDA events are recorded on it
    stream = tstream.cuda_stream
    assert stream != 0
    torch.cuda.synchronize()
    with torch.cuda.stream(tstream):
        for w in range(warmup):
            call_dev(d_in[w % nsets].data_ptr(), d_out[w % nsets].data_ptr(), stream)
    torch.cuda.synchronize()
    l0 = ev.kernel_launches
    dist_barrier(world)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(device_index) as clk, torch.cuda.stream(tstream):
        e0.record(tstream)
        for k in range(steps):
            call_dev(d_in[k % nsets].data_ptr(), d_out[k % nsets].data_ptr(), stream)
        e1.record(tstream)
        torch.cuda.synchronize()
    dist_barrier(world)
    t_dev = e0.elapsed_time(e1) / 1e3
    launches = ev.kernel_launches - l0
    t_dev_max, units = dist_max_sum(world, t_dev, M * steps, dev)
    # ---- the host-buffer C-ABI call.  The driver's chunk arrays live for the whole search and are page-locked once
    # (tsb_*_register_host, as the C++ drivers do and INTEGRATION.md tells the Chapel drivers to)
    host_out = [np.empty(out_elems, dtype=out_dtype) for _ in range(len(host_in))]
    for a in host_in + host_out:
        ev.register_host(a)
    for w in range(max(warmup, len(host_in))):
        call_host(host_in[w % len(host_in)], host_out[w % len(host_in)])
    dist_barrier(world)
    torch.cuda.synchronize()
    with ClockSampler(device_index) as clk2:
        t0 = time.perf_counter()
        for k in range(steps):
            call_host(host_in[k % len(host_in)], host_out[k % len(host_in)])
        torch.cuda.synchronize()
        t_e2e = time.perf_counter() - t0
    clk.samples += clk2.samples
    clk.reasons |= clk2.reasons
    dist_barrier(world)
    t_e2e_max, _ = dist_max_sum(world, t_e2e, M * steps, dev)
    ev.close()
    del d_in, d_out
    torch.cuda.empty_cache()
    return {"M": M, "steps": steps, "units": units, "t_dev": t_dev_max, "t_dev_local": t_dev, "t_e2e": t_e2e_max,
            "launches": launches, "in_rec": in_rec, "out_rec": out_rec, "nsets": nsets, "clocks": clk.summary(),
            "footprint_mb": nsets * bytes_per_set / 2**20}


def summarize(r, peak, peak_src, traffic=None):
    alg_bytes = r["M"] * (r["in_rec"] + r["out_rec"])
    t_kernel = r["t_dev_local"] / r["steps"]
    achieved = alg_bytes / t_kernel / 1e9
    return {"M": r["M"], "value": r["units"] / r["t_dev"] / 1e6, "unit": "Mnodes/s",
            "ms_per_step": r["t_dev"] / r["steps"] * 1e3,
            "e2e": {"value": r["units"] / r["t_e2e"] / 1e6, "unit": "Mnodes/s",
                    "h2d_bytes_per_step": r["M"] * r["in_rec"], "d2h_bytes_per_step": r["M"] * r["out_rec"],
                    "ms_per_step": r["t_e2e"] / r["steps"] * 1e3},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic["bytes"] if traffic else None,
                         "traffic_source": traffic["source"] if traffic else None, "peak_source": peak_src,
                         "bytes_per_launch": alg_bytes, "kernel_us": t_kernel * 1e6},
            "gpu_launches": r["launches"], "buffer_sets": r["nsets"], "footprint_mb": round(r["footprint_mb"], 1)}


# ----------------------------------------------------------------------------------------- other whole searches
def search_on_handle(kind, reps, device_index, **kw):
    """best-of-`reps` whole search on a pre-created handle (set-up reported separately)"""
    import tsb200
    t0 = time.perf_counter()
    if kind == "nq":
        ev = tsb200.NQueensEvaluator(kw["N"], 1, kw["M"], device=device_index)
        go = lambda: ev.search(m_HEAD, kw["M"])  # noqa: E731
        want = GOLDEN_NQ[kw["N"]]
    else:
        ev = tsb200.PfspEvaluator(kw["inst"], M=kw["M"], device=device_index)
        go = lambda: ev.search(kw["inst"], kw["lb"], 1, m_HEAD, kw["M"])  # noqa: E731
        want = GOLDEN_PFSP[(kw["inst"], kw["lb"])]
    setup = time.perf_counter() - t0
    go()  # first search: arena allocation, kernel attributes
    best_t, st = None, None
    for _ in range(reps):
        t0 = time.perf_counter()
        st = go()
        dt = time.perf_counter() - t0
        best_t = dt if best_t is None else min(best_t, dt)
    got = (st.explored_tree, st.explored_sol) + ((int(st.best),) if kind != "nq" else ())
    ev.close()
    return {"explored_tree": int(st.explored_tree), "explored_sol": int(st.explored_sol), "seconds": best_t,
            "value": st.explored_tree / best_t / 1e6, "unit": "Mnodes/s", "offloads": int(st.offloads),
            "gpu_launches": int(st.kernel_launches), "M": kw["M"], "reps": reps, "setup_ms": setup * 1e3,
            "counts_match_reference": got == want,
            "hbm_frac_42B_per_node": st.explored_tree * NODE_BYTES / best_t / 1e9 / peaks()[0] if kind == "nq" else None}


def search_multi(N, M, D):
    import tsb200
    t0 = time.perf_counter()
    st = tsb200.nqueens_search_device(N, 1, m_HEAD, M, D)
    dt = time.perf_counter() - t0
    return {"explored_tree": int(st.explored_tree), "explored_sol": int(st.explored_sol), "seconds": dt,
            "t_step2": st.t_step2, "value": st.explored_tree / dt / 1e6, "unit": "Mnodes/s", "M": M, "D": D,
            "offloads": int(st.offloads), "steals": int(st.steals),
            "per_gpu_share": [round(st.per_gpu_tree[i] / st.explored_tree, 4) for i in range(D)],
            "counts_match_reference": (st.explored_tree, st.explored_sol) == GOLDEN_NQ[N]}


# ----------------------------------------------------------------------------------------- CPU arms
def cpu_search_sample_N(cores):
    """the bounded sample of the workload a CPU step explores: a whole smaller search (same code per node), sized by
    a short probe (the N=14 search) so that a step takes a few seconds on THIS host (the threads a container may use and the cores it
    gets are two different things: 128 threads ran like 10 cores on the round-1 bench box, like 60 on another)"""
    from oracle import pyoracle as po
    tree, _, dt, _ = po.nq_cpu_search(14, cores, depth=4)
    rate = tree / max(dt, 1e-3)
    for N in (16, 15):
        if GOLDEN_NQ[N][0] / rate <= 4.0:
            return N
    return 14


def cpu_baseline_search(cores):
    from oracle import pyoracle as po
    Nref = cpu_search_sample_N(cores)
    tree, sol, dt, src = po.nq_cpu_search(Nref, cores, depth=4)
    assert (tree, sol) == GOLDEN_NQ[Nref]
    t1, s1, dt1, _ = po.nq_cpu_search(13, 1)
    return {"value": tree / dt / 1e6, "unit": "Mnodes/s", "cores": cores, "kind": src,
            "sample": f"whole N={Nref} search ({tree} nodes, {dt:.2f} s) with the reference's sequential search code on "
                      f"{cores} host threads (subtrees of the depth-4 frontier handed out dynamically)",
            "value_1core": t1 / dt1 / 1e6, "sample_1core": f"whole N=13 search, one thread ({dt1:.2f} s)"}


def write_outputs(path, arrays):
    """--dump-outputs: DIR/<name>.npy per array (float32 / float64; the headline's outputs are a few KB)"""
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        assert a.dtype in (np.float32, np.float64), name
        np.save(os.path.join(path, f"{name}.npy"), a)


def emit(line):
    """print THE one JSON line on the real stdout (fd 1 is pointed at stderr while the bench runs, so that
    libraries that write to stdout on their own — NCCL prints its version there — cannot pollute it)"""
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


_REAL_STDOUT = 1


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--big-M", type=int, default=1 << 22, help="parents per step of the bandwidth-bound batch legs")
    ap.add_argument("--pfsp-M", type=int, default=1 << 20)
    ap.add_argument("--no-batch", action="store_true", help="skip the batch-evaluator legs")
    ap.add_argument("--no-search", action="store_true", help="skip the secondary whole searches")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the headline's last step returned as DIR/<name>.npy")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3)
    rank, local_rank, world = dist_env()
    config = make_config(args.gpus)
    cores = host_cores()

    if args.impl == "reference":
        if rank != 0:
            return
        from oracle import pyoracle as po
        Nref = cpu_search_sample_N(cores)
        for _ in range(min(args.warmup, 3)):
            po.nq_cpu_search(Nref, cores, depth=4)
        t, tree, src = 0.0, 0, "port"
        for _ in range(args.steps):
            tr, so, dt, src = po.nq_cpu_search(Nref, cores, depth=4)
            assert (tr, so) == GOLDEN_NQ[Nref]
            t += dt
            tree += tr
        v = tree / t / 1e6
        t1, s1, dt1, _ = po.nq_cpu_search(13, 1)
        sample = (f"each step = the whole N={Nref} search ({GOLDEN_NQ[Nref][0]} nodes: a bounded sample of the N={N_HEAD} "
                  f"tree, same code per node) with the reference's own sequential search code "
                  f"(baselines/nqueens/nqueens_c.c pool / isSafe / decompose, compiled into oracle/_ref) on {cores} host "
                  "threads; the reference's CPU program itself is single-threaded (value_1core)")
        line = {"impl": "reference", "metric": "Mnodes/s", "value": v, "unit": "Mnodes/s", "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": t / args.steps * 1e3,
                "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
                "config": config,
                "cpu_baseline": {"value": v, "unit": "Mnodes/s", "cores": cores, "kind": src, "sample": sample,
                                 "value_1core": t1 / dt1 / 1e6},
                "e2e": {"value": v, "unit": "Mnodes/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        emit(line)
        return

    import torch
    assert torch.cuda.is_available(), "bench.py needs a CUDA device; there is no CPU fallback"
    world = dist_init("nccl")
    device_index = local_rank if world > 1 else 0
    peak, peak_src = peaks()
    numa_cores = None
    if world > 1:  # one process per GPU: run (and first-touch the host buffers) on the cores next to that GPU
        import tsb200
        rc = tsb200.lib().tsb_bind_thread_to_device(device_index)
        numa_cores = rc if rc > 0 else None

    # ------------------------------------------------------------------ headline: the N=17 --M 50000 search
    if world == 1:
        h = run_headline_1gpu(args.steps, args.warmup, 0)
    else:
        h = run_headline_multi(args.steps, args.warmup, world, rank)
    line = None
    if rank == 0 and args.dump_outputs:
        write_outputs(args.dump_outputs, h["outputs"])
    if rank == 0:
        value = h["nodes"] / h["t_dev"] / 1e6
        e2e = h["tree"] / h["t_e2e"] / 1e6
        kernel_s = h["t_dev"] / h["steps"]  # one launch (per GPU) runs all rounds of a step
        achieved = h["nodes"] / h["steps"] * NODE_BYTES / kernel_s / 1e9
        line = {"metric": "Mnodes/s", "value": value, "unit": "Mnodes/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": h["t_dev"] / h["steps"] * 1e3, "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": config,
                "clocks": h["clocks"],
                "e2e": {"value": e2e, "unit": "Mnodes/s", "h2d_bytes_per_step": h["h2d"], "d2h_bytes_per_step": h["d2h"],
                        "ms_per_step": h["t_e2e"] / h["steps"] * 1e3},
                "gpu_launches": h["launches"],
                "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak * world, "unit": "GB/s",
                             "frac": achieved / (peak * world), "peak_source": peak_src,
                             "traffic": None,
                             "traffic_note": "profiles/nq_rounds_pools_r2_ncu.txt (first launch of this search: 2 048 rounds of each "
                                             "of the four pools, ~0.4 G nodes = 17 GB algorithmic): 98 MB read + 313 MB written "
                                             "in DRAM — a 2 MB round lives in the 126 MB L2; profiles/nq_rounds_r2_ncu.txt (one "
                                             "pool, the whole N=15 search in one launch): 0.75 MB read + 4.8 MB written",
                             "kernel": "nq_rounds_ll_kernel<17> (persistent, cooperative; four independent pools per "
                                       "launch, 74 CTAs each, two CTAs per SM)",
                             "bytes_per_launch": h["nodes"] / h["steps"] * NODE_BYTES, "kernel_us": kernel_s * 1e6,
                             "rounds_per_launch": h["rounds"] / h["steps"],
                             "us_per_round": kernel_s * 1e6 / max(1.0, h["rounds"] / h["steps"]),
                             "note": "42 algorithmic bytes per explored node; a round of 50 000 parents moves ~2 MB and "
                                     "is a chain of L2 round trips (one count exchange among the pool's CTAs, one "
                                     "store -> poll hop for the nodes; tools/flag_exchange.py) with ~1 us of work in "
                                     "between, not HBM-bound; the rounds of the four pools of a GPU overlap (us_per_round "
                                     "= kernel time / rounds of all pools) — see kernels.* for the bandwidth-bound kernels"},
                "numa": {"rank0_bound_to_cores_of_its_gpu": numa_cores, "note": "tsb_bind_thread_to_device: every rank (and "
                         "every per-GPU host thread of the multi-GPU search) is pinned to the cores local to its GPU"},
                "headline": {"explored_tree": GOLDEN_NQ[N_HEAD][0], "explored_sol": GOLDEN_NQ[N_HEAD][1],
                             "counts_match_reference": True, "offloads_per_search": h["offloads"],
                             "pools_per_gpu": h.get("pools"),
                             "launches_per_search": h["launches_per_step"], "handle_create_ms": h["create_ms"],
                             "steals_per_search": h.get("steals"), "per_gpu_share": h.get("per_gpu_share")}}

    # ------------------------------------------------------------------ secondary: batch evaluators (weak scaling)
    kernels = {}
    if not args.no_batch:
        bsteps = max(args.steps, 20)
        big = summarize(run_workload("nq", args.big_M, bsteps, args.warmup, device_index, world),
                        peak, peak_src, ncu_traffic("nq_evaluate_kernel", ["nq_eval_r2_ncu.txt", "nq_eval_r1_ncu.txt"]))
        small = summarize(run_workload("nq", 50000, bsteps * 10, args.warmup, device_index, world), peak, peak_src)
        pf = summarize(run_workload("pfsp", args.pfsp_M, bsteps, args.warmup, device_index, world),
                       peak, peak_src, ncu_traffic("pfsp_lb1_kernel", ["pfsp_lb1_r2_ncu.txt", "pfsp_lb1_r1_ncu.txt"]))
        pf_small = summarize(run_workload("pfsp", 50000, bsteps * 5, args.warmup, device_index, world), peak, peak_src)
        l2 = summarize(run_workload("lb2", 1 << 18, max(3, bsteps // 4), args.warmup, device_index, world),
                       peak, peak_src, ncu_traffic("pfsp_lb2_kernel", ["pfsp_lb2_r2_ncu.txt", "pfsp_lb2_r1_ncu.txt"]))
        if rank == 0:
            line["batch"] = {
                "note": "batch node evaluation (round 1's headline): parents per second; value = device-resident, one "
                        "launch per step, CUDA events; e2e = tsb_*_evaluate on registered host arrays; scaling weak "
                        "(every rank its own batch)",
                "nqueens_N17": dict(big, workload="N-Queens N=17, synthetic parents, depth ~ explored-tree histogram"),
                "nqueens_N17_M50000": dict(small, note="one offload of the unmodified driver: 1.9 MB per launch"),
                "pfsp_ta014_lb1": dict(pf, workload="PFSP ta014 lb1 ub=1, ta014/lb1 offload depth histogram", dtype="int32"),
                "pfsp_ta014_lb1_M50000": pf_small,
                "pfsp_ta020_lb2": dict(l2, workload="PFSP ta020 lb2 ub=1 (best=1591), ta020/lb2 offload depth "
                                                     "histogram; int-ALU bound (O(pairs*jobs) per child)", dtype="int32")}
            for name, r in (("nq_evaluate_kernel<17>", big), ("pfsp_lb1_kernel<ta014>", pf), ("pfsp_lb2_kernel<ta020>", l2)):
                kernels[name] = {k: r["roofline"][k] for k in ("kernel_us", "achieved", "frac", "traffic", "bytes_per_launch")}
    # ------------------------------------------------------------------ secondary: other whole searches
    torch.cuda.synchronize()
    dist_barrier(world, cpu=True)
    if not args.no_search and rank == 0:
        srch = {"note": "explored tree / wall time of whole searches on pre-created handles (tsb_*_search_on: step 1 and "
                        "3 on the CPU, pool of step 2 resident in HBM); set-up (handle, tables, first arena) in setup_ms"}
        if world == 1:
            srch["nqueens_N17_bigM"] = search_on_handle("nq", 3, 0, N=17, M=args.big_M)
            srch["pfsp_ta014_lb1_M50000"] = search_on_handle("pfsp", 7, 0, inst=14, lb="lb1", M=50000)
            srch["pfsp_ta020_lb2_M50000"] = search_on_handle("pfsp", 7, 0, inst=20, lb="lb2", M=50000)
            srch["pfsp_ta020_lb1d_chapel_minheads"] = search_on_handle("pfsp", 2, 0, inst=20, lb="lb1_d", M=1 << 20)
            r = srch["nqueens_N17_bigM"]
            kernels["nq_expand_count+build<17> (search at --big-M)"] = {
                "kernel_us": r["seconds"] * 1e6 / max(1, r["offloads"]), "frac": r["hbm_frac_42B_per_node"],
                "achieved": r["hbm_frac_42B_per_node"] * peak, "traffic": None,
                "bytes_per_launch": r["explored_tree"] * NODE_BYTES / max(1, r["offloads"])}
        else:
            srch["nqueens_N17_bigM"] = search_multi(17, args.big_M, world)
            srch["nqueens_N18_M50000"] = search_multi(18, 50000, world)
            if world == 8:  # BASELINE configs[4]
                srch["nqueens_N19_D8_M50000"] = search_multi(19, 50000, 8)
                srch["nqueens_N19_D8_bigM"] = search_multi(19, 1 << 24, 8)
        line["search"] = srch
    dist_barrier(world, cpu=True)
    if rank == 0:
        line["kernels"] = kernels
        if world == 1 and not args.no_cpu:
            line["cpu_baseline"] = cpu_baseline_search(cores)
        emit(line)
    if world > 1:
        import torch.distributed as dist
        dist_barrier(world, cpu=True)
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
