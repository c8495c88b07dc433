"""GPU tests of the MAX_JOBS = 50 build (208-byte nodes, ta031..ta060) beyond evaluate: the fused evaluate +
generate_children (tsb_pfsp_expand / _expand_device), the device-resident pool and its stealing, and whole 3-step
searches (tsb_pfsp_search_wide / _search_device_wide), against the oracle built with OR_MAX_JOBS = 50 and the counts
of the reference's C program built with MAX_JOBS 50 (tests/golden/pfsp_jobs50_counts.json)."""
import ctypes as C
import json
import os

import numpy as np
import pytest

import tsb200
from oracle import pyoracle50 as po50
from tsb200 import _lib

pytestmark = pytest.mark.gpu
LBS = ("lb1", "lb1_d", "lb2")
OPT = {31: 2724, 32: 2834, 37: 2725, 38: 2683, 41: 2991, 51: 3846}


class SearchResult50(C.Structure):
    """or_search_result with OR_MAX_JOBS = 50"""
    _fields_ = [("tree", C.c_uint64), ("sol", C.c_uint64), ("best", C.c_int64), ("offloads", C.c_uint64),
                ("offloaded_parents", C.c_uint64), ("live_slots", C.c_uint64), ("depth_hist", C.c_uint64 * 52),
                ("seconds", C.c_double)]


def _o50():
    L = po50.lib()
    L.or_pfsp_expand_chunk.argtypes = [C.POINTER(po50.Tables), C.c_int, C.c_void_p, C.c_int, C.POINTER(C.c_int64),
                                       C.c_void_p, C.c_int64, C.POINTER(C.c_uint64)]
    L.or_pfsp_expand_chunk.restype = C.c_int64
    L.or_pfsp_search_offload.argtypes = [C.c_int] * 7 + [C.POINTER(SearchResult50)]
    return L


def oracle_expand(t, lb, parents, best):
    """(children, n_solutions, best_after) of one chunk: the oracle's evaluate + sequential generate_children"""
    parents = np.ascontiguousarray(parents).view(po50.PFSP_NODE_DTYPE)
    cap = parents.shape[0] * 50 + 1
    out = np.zeros(cap, dtype=po50.PFSP_NODE_DTYPE)
    sol, b = C.c_uint64(0), C.c_int64(int(best))
    n = _o50().or_pfsp_expand_chunk(C.byref(t), tsb200.LB_NAMES[lb], parents.ctypes.data, parents.shape[0], C.byref(b),
                                    out.ctypes.data, cap, C.byref(sol))
    return out[:n].view(tsb200.PFSP_NODE50_DTYPE).copy(), int(sol.value), int(b.value)


def oracle_search(inst, lb, ub, m, M, D):
    r = SearchResult50()
    _o50().or_pfsp_search_offload(inst, tsb200.LB_NAMES[lb], ub, m, M, D, 0, C.byref(r))
    return r


def rand_nodes(rng, count, depth_lo=1, depth_hi=50):
    nodes = np.zeros(count, dtype=tsb200.PFSP_NODE50_DTYPE)
    depth = rng.integers(depth_lo, depth_hi, size=count)
    nodes["depth"], nodes["limit1"] = depth, depth - 1
    nodes["prmu"] = np.argsort(rng.random((count, 50)), axis=1).astype(np.int32)
    return nodes


def check_expand(ev, t, parents, lb, best):
    got, gsol, gbest = ev.expand(parents, lb, best)
    want, wsol, wbest = oracle_expand(t, lb, parents, best)
    assert (gsol, gbest, got.shape[0]) == (wsol, wbest, want.shape[0])
    assert got.tobytes() == want.tobytes()
    return got.shape[0], gbest


@pytest.mark.parametrize("inst", [31, 41, 51])
@pytest.mark.parametrize("lb", LBS)
def test_expand_matches_oracle_children(inst, lb):
    """chunks around the 64-parent tile; best = optimum, optimum + 60; the root (limit1 = -1) for lb1_d"""
    rng = np.random.default_rng(500 + inst)
    t = po50.tables(inst)
    M = 3000
    with tsb200.PfspEvaluator(inst, M=M) as ev:
        assert ev.wide
        for count in (1, 63, 64, 65, 127, 3000, M):
            parents = rand_nodes(rng, count, depth_lo=0 if lb == "lb1_d" else 1)
            for best in (OPT[inst], OPT[inst] + 60):
                check_expand(ev, t, parents, lb, best)
        root = np.zeros(64, dtype=tsb200.PFSP_NODE50_DTYPE)
        root["limit1"] = -1
        root["prmu"] = np.argsort(rng.random((64, 50)), axis=1).astype(np.int32)
        if lb == "lb1_d":
            n, _ = check_expand(ev, t, root, lb, 2**31 - 1)
            assert n == 64 * 50


@pytest.mark.parametrize("lb", LBS)
def test_expand_when_a_leaf_improves_best(lb):
    """depth 47..49 parents: leaf children lower best in the middle of the chunk and the rest of the chunk is pruned
    against the lowered value (the reference's sequential rule, redone on the host)"""
    inst = 41
    rng = np.random.default_rng(78)
    t = po50.tables(inst)
    parents = rand_nodes(rng, 2000, depth_lo=47)
    _, _, low = oracle_expand(t, lb, parents, 2**31 - 1)
    with tsb200.PfspEvaluator(inst, M=2000) as ev:
        for best in (2**63 - 1, 2**31 - 1, low + 150):
            _, b = check_expand(ev, t, parents, lb, best)
            assert b < best
        assert ev.slow_rounds >= 3


def test_expand_device_matches_expand_and_checks_alignment():
    import torch
    inst, lb, best = 51, "lb1", OPT[51] + 60
    rng = np.random.default_rng(3)
    parents = rand_nodes(rng, 700)
    with tsb200.PfspEvaluator(inst, M=700) as ev:
        want, wsol, wbest = ev.expand(parents, lb, best)
        d_par = torch.from_numpy(parents.view(np.uint8).copy()).cuda()
        d_kids = torch.zeros(700 * 50 * 208 + 64, dtype=torch.uint8, device="cuda")
        nc, ns, b = C.c_uint64(0), C.c_uint64(0), C.c_int64(best)
        L = tsb200.lib()
        torch.cuda.synchronize()
        rc = L.tsb_pfsp_expand_device(ev._h, tsb200.LB_NAMES[lb], d_par.data_ptr(), 700, C.byref(b), d_kids.data_ptr(),
                                      C.byref(nc), C.byref(ns), None)
        assert rc == _lib.OK
        torch.cuda.synchronize()
        got = d_kids[: nc.value * 208].cpu().numpy().view(tsb200.PFSP_NODE50_DTYPE)
        assert (nc.value, ns.value, b.value) == (want.shape[0], wsol, wbest)
        assert got.tobytes() == want.tobytes()
        for p_off, c_off in ((4, 0), (0, 8)):  # 208-byte children are stored by 16-byte TMA copies
            b = C.c_int64(best)
            rc = L.tsb_pfsp_expand_device(ev._h, tsb200.LB_NAMES[lb], d_par.data_ptr() + p_off, 10, C.byref(b),
                                          d_kids.data_ptr() + c_off, C.byref(nc), C.byref(ns), None)
            assert rc == _lib.EALIGN


def _pool_vs_mirror(ev, t, host_pool, lb, m, M, best, rounds):
    for _ in range(rounds):
        n_par, n_child, n_sol, best2 = ev.pool_step(lb, m, M, best)
        if host_pool.shape[0] < m:
            assert n_par == 0
            break
        n = min(host_pool.shape[0], M)
        kids, sol, wbest = oracle_expand(t, lb, host_pool[host_pool.shape[0] - n:], best)
        host_pool = np.concatenate([host_pool[: host_pool.shape[0] - n], kids])
        assert (n_par, n_child, n_sol, best2) == (n, kids.shape[0], sol, wbest)
        best = best2
        assert ev.pool_size == host_pool.shape[0]
    return host_pool, best


@pytest.mark.parametrize("lb", LBS)
def test_device_pool_is_byte_identical_to_the_reference_pool(lb):
    inst, m, M = 41, 25, 300
    t = po50.tables(inst)
    rng = np.random.default_rng(12)
    start = rand_nodes(rng, 40, depth_lo=2, depth_hi=7)
    with tsb200.PfspEvaluator(inst, M=M) as ev:
        ev.pool_push(start)
        host_pool, _ = _pool_vs_mirror(ev, t, start.copy(), lb, m, M, OPT[inst], 60)
        rest = ev.pool_drain()
        assert rest.tobytes() == np.ascontiguousarray(host_pool).tobytes() and ev.pool_size == 0


@pytest.mark.parametrize("cap", [None, "4000"])
def test_device_pool_on_the_ta031_tree(monkeypatch, cap):
    """the real ta031 tree from the root (lb1, --ub 1, m = 1): 40 rounds of 300 parents, then 5 of 50 000 (several
    tiles per CTA); with a small initial arena the pool is also compacted and grown on the way"""
    if cap:
        monkeypatch.setenv("TSB200_POOL_CAP", cap)
    inst, lb = 31, "lb1"
    t = po50.tables(inst)
    root = np.zeros(1, dtype=tsb200.PFSP_NODE50_DTYPE)
    root["limit1"] = -1
    root["prmu"][0] = np.arange(50)
    with tsb200.PfspEvaluator(inst, M=50000) as ev:
        ev.pool_push(root)
        host_pool, best = _pool_vs_mirror(ev, t, root.copy(), lb, 1, 300, OPT[inst], 40)
        host_pool, best = _pool_vs_mirror(ev, t, host_pool, lb, 1, 50000, best, 5)
        assert host_pool.shape[0] > 0 and best == OPT[inst]
        rest = ev.pool_drain()
        assert rest.tobytes() == np.ascontiguousarray(host_pool).tobytes()


def test_steal_between_wide_handles_moves_the_oldest_half():
    rng = np.random.default_rng(9)
    nodes = rand_nodes(rng, 1001)
    with tsb200.PfspEvaluator(41, M=1000) as victim, tsb200.PfspEvaluator(41, M=1000) as thief, \
            tsb200.PfspEvaluator(14, M=1000) as narrow:
        victim.pool_push(nodes)
        got = thief.pool_steal_from(victim, 25)
        assert got == 500 and victim.pool_size == 501 and thief.pool_size == 500
        assert thief.pool_drain().tobytes() == nodes[:500].tobytes()
        assert victim.pool_drain().tobytes() == nodes[500:].tobytes()
        victim.pool_push(nodes)
        with pytest.raises(tsb200.TsbError) as e:
            narrow.pool_steal_from(victim, 25)
        assert e.value.code == _lib.EINVAL
        with pytest.raises(tsb200.TsbError) as e:
            victim.pool_steal_from(narrow, 25)
        assert e.value.code == _lib.EINVAL
        with pytest.raises(tsb200.TsbError) as e:  # an 88-byte node array on a 208-byte handle
            victim.pool_push(np.zeros(1, dtype=tsb200.PFSP_NODE_DTYPE))
        assert e.value.code == _lib.EINVAL


SEARCHES = [(32, "lb1"), (37, "lb1"), (38, "lb1"), (32, "lb2"), (37, "lb2"), (38, "lb2"),
            (31, "lb1_d"), (41, "lb1_d"), (51, "lb1_d")]


@pytest.mark.parametrize("inst,lb", SEARCHES)
@pytest.mark.parametrize("device_pool", [False, True])
@pytest.mark.parametrize("D", [1, 2])
@pytest.mark.parametrize("m", [1, 25])
def test_whole_searches(golden_dir, monkeypatch, inst, lb, device_pool, D, m):
    """tree / solutions / optimum and the chunk sequence of the reference driver (static split; with m = 1 the root
    goes through the device rounds), and the counts of the reference's C program built with MAX_JOBS 50 (lb1, lb2)"""
    monkeypatch.setenv("TSB200_NO_STEAL", "1")
    L, st = tsb200.lib(), _lib.SearchStats()
    fn = L.tsb_pfsp_search_device_wide if device_pool else L.tsb_pfsp_search_wide
    _lib.check(fn(50, inst, tsb200.LB_NAMES[lb], 1, m, 50000, D, C.byref(st)), "search_wide")
    ref = oracle_search(inst, lb, 1, m, 50000, D)
    assert (st.explored_tree, st.explored_sol, st.best) == (ref.tree, ref.sol, ref.best)
    assert (st.offloads, st.offloaded_parents) == (ref.offloads, ref.offloaded_parents)
    gold = json.load(open(os.path.join(golden_dir, "pfsp_jobs50_counts.json")))["pfsp"]
    g = gold.get(f"ta{inst:03d}_lb{tsb200.LB_NAMES[lb]}_ub1")
    if g:  # (lb1_d has no C-program count: it reads the min_heads where C and Chapel differ)
        assert (st.explored_tree, st.explored_sol, st.best) == (g["tree"], g["sol"], g["best"])
    else:
        assert lb == "lb1_d" and st.explored_tree == 0 and st.best == OPT[inst]


@pytest.mark.parametrize("inst,lb", [(32, "lb1"), (37, "lb2")])
def test_python_routes_50_job_instances_and_steals(golden_dir, inst, lb):
    """pfsp_search / pfsp_search_device take ta031..ta060 through the wide entry points; D = 2 device pools that
    steal from each other keep the counts (--ub 1)"""
    gold = json.load(open(os.path.join(golden_dir, "pfsp_jobs50_counts.json")))["pfsp"][f"ta{inst:03d}_lb{tsb200.LB_NAMES[lb]}_ub1"]
    for st in (tsb200.pfsp_search(inst, lb, 1, 1, 50000, 1), tsb200.pfsp_search_device(inst, lb, 1, 1, 64, 2)):
        assert (st.explored_tree, st.explored_sol, st.best) == (gold["tree"], gold["sol"], gold["best"])
    with tsb200.PfspEvaluator(inst, M=50000) as ev:
        st = ev.search(inst, lb, 1, 1, 50000)
        assert (st.explored_tree, st.explored_sol, st.best) == (gold["tree"], gold["sol"], gold["best"])


def test_max_jobs_20_forwards(golden_dir):
    counts = json.load(open(os.path.join(golden_dir, "counts.json")))["pfsp"]["ta014_lb1_ub1"]
    L = tsb200.lib()
    for fn in (L.tsb_pfsp_search_wide, L.tsb_pfsp_search_device_wide):
        st = _lib.SearchStats()
        _lib.check(fn(20, 14, tsb200.LB_NAMES["lb1"], 1, 25, 50000, 1, C.byref(st)), "search_wide(20)")
        assert (st.explored_tree, st.explored_sol, st.best) == (counts["tree"], counts["sol"], counts["best"])
