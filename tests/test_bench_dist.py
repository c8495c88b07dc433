"""CPU checks of bench.py: the multi-rank reduction used for N > 1 (world_size-2 gloo run: max over ranks
of the time, sum over ranks of the units — no collective in the data path) and the synthetic workloads; on a GPU,
the outputs --dump-outputs writes."""
import json
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

import bench
import tsb200
from oracle import pyoracle as po

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

WORKER = r"""
import os, sys, json
sys.path.insert(0, %r)
import torch, bench
world = bench.dist_init("gloo")
rank, local_rank, w = bench.dist_env()
assert world == w == 2
bench.dist_barrier(world)
# rank r "measured" (r+1) seconds and processed 1000*(r+1) units
t, u = bench.dist_max_sum(world, float(rank + 1), 1000 * (rank + 1), torch.device("cpu"))
print(json.dumps({"rank": rank, "t": t, "u": u}))
import torch.distributed as dist
dist.destroy_process_group()
""" % ROOT


def test_world_size_2_gloo_reduction(tmp_path):
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    procs = []
    for rank in range(2):
        env = dict(os.environ, RANK=str(rank), LOCAL_RANK=str(rank), WORLD_SIZE="2", MASTER_ADDR="127.0.0.1",
                   MASTER_PORT=str(port))
        procs.append(subprocess.Popen([sys.executable, "-c", WORKER], env=env, stdout=subprocess.PIPE, text=True))
    outs = [json.loads(p.communicate(timeout=300)[0].strip().splitlines()[-1]) for p in procs]
    assert all(p.returncode == 0 for p in procs)
    for o in outs:
        assert o["t"] == 2.0 and o["u"] == 3000.0  # max over ranks / whole-job units


def test_reference_arm_other_ranks_do_no_work():
    env = dict(os.environ, RANK="1", LOCAL_RANK="1", WORLD_SIZE="2")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"], env=env,
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_synthetic_nq_parents_are_valid_tree_nodes():
    N = 17
    p = bench.synth_nq_parents(N, 4096, 7, tsb200.NQ_NODE_DTYPE)
    hist = bench.nq_depth_hist(N)
    assert sum(hist.values()) == 8017021931  # the reference's explored-tree size for N = 17
    b = p["board"].astype(int)
    for i in range(0, 4096, 16):
        d = int(p["depth"][i])
        assert 1 <= d <= N and sorted(b[i, :N]) == list(range(N))
        for r in range(d):
            for r2 in range(r):
                assert abs(b[i, r] - b[i, r2]) != r - r2
    # the oracle agrees that every placed prefix is conflict-free: the parent of each node labels it safe
    par = p.copy()
    keep = par["depth"] > 0
    par["depth"][keep] -= 1
    lab = po.nq_evaluate(np.ascontiguousarray(par).view(po.NQ_NODE_DTYPE), N).reshape(-1, N)
    idx = np.nonzero(keep)[0]
    assert (lab[idx, par["depth"][idx].astype(int)] == 1).all()


def test_synthetic_pfsp_parents():
    p = bench.synth_pfsp_parents(2048, 3, tsb200.PFSP_NODE_DTYPE)
    assert (p["limit1"] == p["depth"] - 1).all() and p["depth"].min() >= 1 and p["depth"].max() <= 19
    assert (np.sort(p["prmu"], axis=1) == np.arange(20)).all()


@pytest.mark.gpu
def test_dump_outputs_of_the_headline_step(tmp_path):
    """--dump-outputs writes float32 / float64 arrays of the last timed step, and they are what that step computed:
    every node pushed (warm-up pool + children) was popped or left over, and with nothing left over, warm-up + step-2
    children and solutions = the reference's N=17 counts"""
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "0", "--no-batch",
                        "--no-search", "--no-cpu", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    assert json.loads(r.stdout)["steps"] == 1
    files = sorted(tmp_path.glob("*.npy"))
    assert sum(f.stat().st_size for f in files) <= 64 << 20
    out = {f.stem: np.load(f) for f in files}
    assert set(out) == {"step2_pools", "search_counts"}
    assert all(a.dtype in (np.float32, np.float64) and a.size for a in out.values())
    want = bench.GOLDEN_NQ[17]
    assert tuple(out["search_counts"]) == want
    pools = out["step2_pools"].astype(np.int64)
    assert pools.ndim == 2 and pools.shape[1] == 5 and (pools[:, 0] > 0).all()
    _, parents, children, solutions, left = pools.sum(axis=0)
    assert (pools[:, 4] < bench.m_HEAD).all()
    warm, wtree, wsol = tsb200.nqueens_warmup(17, pools.shape[0] * bench.m_HEAD)
    assert warm.shape[0] + children == parents + left  # steals move nodes between pools, none is lost
    if left == 0:  # every pool ran dry: the search has nothing left for step 3
        assert (wtree + children, wsol + solutions) == want
    else:
        assert wtree + children < want[0] and wsol + solutions <= want[1]
