"""PFSP side of the offload interface (pfsp_gpu_chpl.chpl / pfsp_multigpu_chpl.chpl)."""
from __future__ import annotations

import ctypes as C

import numpy as np

from ._lib import EINVAL, LB1, LB1_D, LB2, PfspTables, PfspTables50, SearchStats, TsbError, check, lib

# lib/pfsp/PFSP_node.chpl:9-12
PFSP_NODE_DTYPE = np.dtype([("depth", np.int32), ("limit1", np.int32), ("prmu", np.int32, (20,))])
assert PFSP_NODE_DTYPE.itemsize == 88
# a build of the reference with MAX_JOBS = 50 (ta031..ta060)
PFSP_NODE50_DTYPE = np.dtype([("depth", np.int32), ("limit1", np.int32), ("prmu", np.int32, (50,))])
assert PFSP_NODE50_DTYPE.itemsize == 208
# the Chapel CLI spells the bounds as strings (pfsp_gpu_chpl.chpl:15), the C ABI as the C baseline's ints
LB_NAMES = {"lb1_d": LB1_D, "lb1": LB1, "lb2": LB2}


LB2_VARIANTS = {"full": 0, "nabeshima": 1, "lageweg": 2, "learn": 3}  # lib/pfsp/Bound_johnson.chpl:6


def taillard_tables(inst: int, variant="full") -> PfspTables:
    """lbound1 / lbound2 as built at pfsp_gpu_chpl.chpl:325-332 (Chapel semantics, incl. its min_heads); `variant`
    selects the machine pairs of lb2 (the reference compiles "full")"""
    t = PfspTables()
    v = LB2_VARIANTS[variant] if isinstance(variant, str) else int(variant)
    check(lib().tsb_pfsp_tables_build_variant(C.byref(t), inst, v), "tsb_pfsp_tables_build_variant")
    return t


def taillard_tables50(inst: int, variant="full") -> PfspTables50:
    t = PfspTables50()
    v = LB2_VARIANTS[variant] if isinstance(variant, str) else int(variant)
    check(lib().tsb_pfsp_tables50_build(C.byref(t), inst, v), "tsb_pfsp_tables50_build")
    return t


def _max_jobs(inst: int) -> int:
    """MAX_JOBS of the reference build that runs `inst`: 20 for ta001..ta030, 50 for ta031..ta060"""
    return 50 if lib().tsb_taillard_nb_jobs(inst) == 50 else 20


class PfspEvaluator:
    """Owns parents_d / bounds_d / lbound1_d / lbound2_d of pfsp_gpu_chpl.chpl:359-371.  Instances with more than
    20 jobs (ta031..ta060) create a MAX_JOBS = 50 handle: nodes are PFSP_NODE50_DTYPE, for every entry point."""

    def __init__(self, inst: int | None = None, tables=None, M: int = 50000, device: int = 0):
        if tables is None:
            tables = taillard_tables50(inst) if lib().tsb_taillard_nb_jobs(inst) > 20 else taillard_tables(inst)
        self.tables = tables
        self.jobs, self.machines, self.M = self.tables.jobs, self.tables.machines, M
        self.wide = isinstance(tables, PfspTables50)
        self.node_dtype = PFSP_NODE50_DTYPE if self.wide else PFSP_NODE_DTYPE
        self._h = C.c_void_p()
        if self.wide:
            check(lib().tsb_pfsp_create50_from_tables(C.byref(self._h), device, M, C.byref(self.tables)), "tsb_pfsp_create_wide")
        else:
            check(lib().tsb_pfsp_create_from_tables(C.byref(self._h), device, M, C.byref(self.tables)), "tsb_pfsp_create")

    def close(self):
        if self._h:
            lib().tsb_pfsp_destroy(self._h)
            self._h = C.c_void_p()

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def set_xfer(self, mode: int):
        check(lib().tsb_pfsp_set_xfer(self._h, mode), "tsb_pfsp_set_xfer")

    def register_host(self, arr: np.ndarray) -> None:
        """page-lock + map a long-lived host array (the driver's `parents` / `bounds`); see NQueensEvaluator"""
        check(lib().tsb_pfsp_register_host(self._h, arr.ctypes.data, arr.nbytes), "tsb_pfsp_register_host")

    def unregister_host(self, arr: np.ndarray) -> None:
        check(lib().tsb_pfsp_unregister_host(self._h, arr.ctypes.data), "tsb_pfsp_unregister_host")

    def _nodes(self, nodes: np.ndarray, where: str) -> None:
        """a node array of this handle's build (88-byte records, or 208-byte ones on a MAX_JOBS = 50 handle)"""
        if nodes.dtype != self.node_dtype or not nodes.flags.c_contiguous:
            raise TsbError(EINVAL, f"{where}: nodes must be a C-contiguous {self.node_dtype.itemsize}-byte node array")

    @property
    def kernel_launches(self) -> int:
        return int(lib().tsb_pfsp_kernel_launches(self._h))

    def evaluate_gpu(self, parents: np.ndarray, size: int, best: int, lb, bounds: np.ndarray) -> None:
        """evaluate_gpu(parents_d, size, best, lbound1_d, lbound2_d, bounds_d) of pfsp_gpu_chpl.chpl:257-270 with
        the copies of :384/:386; `size` = jobs * poolSize; lb is "lb1" | "lb1_d" | "lb2" or the int code"""
        assert parents.dtype == self.node_dtype and parents.flags.c_contiguous
        assert bounds.dtype == np.int32 and bounds.flags.c_contiguous
        kind = LB_NAMES[lb] if isinstance(lb, str) else int(lb)
        if size % self.jobs:
            raise ValueError("size must be jobs * poolSize")
        count = size // self.jobs
        assert parents.shape[0] >= count and bounds.size >= size
        check(lib().tsb_pfsp_evaluate(self._h, kind, parents.ctypes.data, count, int(best), bounds.ctypes.data),
              "tsb_pfsp_evaluate")

    def evaluate(self, parents: np.ndarray, lb, best: int) -> np.ndarray:
        bounds = np.empty(parents.shape[0] * self.jobs, dtype=np.int32)
        self.evaluate_gpu(parents, parents.shape[0] * self.jobs, best, lb, bounds)
        return bounds

    def evaluate_device(self, lb, parents_ptr: int, count: int, best: int, bounds_ptr: int, stream: int = 0) -> None:
        kind = LB_NAMES[lb] if isinstance(lb, str) else int(lb)
        check(lib().tsb_pfsp_evaluate_device(self._h, kind, parents_ptr, count, int(best), bounds_ptr, stream),
              "tsb_pfsp_evaluate_device")


    # ---- beyond the drop-in: fused evaluate_gpu + generate_children, device-resident pool
    def expand(self, parents: np.ndarray, lb, best: int):
        """(children, n_solutions, best_after): evaluate_gpu (pfsp_gpu_chpl.chpl:192-270) + generate_children
        (:273-303) of one chunk in one device pass"""
        self._nodes(parents, "tsb_pfsp_expand")
        kind = LB_NAMES[lb] if isinstance(lb, str) else int(lb)
        cap = parents.shape[0] * self.jobs
        out = np.empty(max(cap, 1), dtype=self.node_dtype)
        nc, ns, b = C.c_uint64(0), C.c_uint64(0), C.c_int64(int(best))
        check(lib().tsb_pfsp_expand(self._h, kind, parents.ctypes.data, parents.shape[0], C.byref(b), out.ctypes.data,
                                    cap, C.byref(nc), C.byref(ns)), "tsb_pfsp_expand")
        return out[: nc.value].copy(), int(ns.value), int(b.value)

    def pool_push(self, nodes: np.ndarray) -> None:
        self._nodes(nodes, "tsb_pfsp_pool_push")
        check(lib().tsb_pfsp_pool_push(self._h, nodes.ctypes.data, nodes.shape[0]), "tsb_pfsp_pool_push")

    @property
    def pool_size(self) -> int:
        return int(lib().tsb_pfsp_pool_size(self._h))

    @property
    def slow_rounds(self) -> int:
        return int(lib().tsb_pfsp_slow_rounds(self._h))

    def pool_step(self, lb, m: int, M: int, best: int):
        """(parents popped, children appended, solutions, best_after) of one device-side offload round"""
        kind = LB_NAMES[lb] if isinstance(lb, str) else int(lb)
        np_, nc, ns, b = C.c_int64(0), C.c_uint64(0), C.c_uint64(0), C.c_int64(int(best))
        check(lib().tsb_pfsp_pool_step(self._h, kind, m, M, C.byref(b), C.byref(np_), C.byref(nc), C.byref(ns)),
              "tsb_pfsp_pool_step")
        return int(np_.value), int(nc.value), int(ns.value), int(b.value)

    def search(self, inst: int, lb, ub: int = 1, m: int = 25, M: int | None = None) -> SearchStats:
        """the whole 3-step search (pfsp_gpu_chpl.chpl:306-431) with the pool of step 2 on this handle's device"""
        kind = LB_NAMES[lb] if isinstance(lb, str) else int(lb)
        st = SearchStats()
        check(lib().tsb_pfsp_search_on(self._h, inst, kind, ub, m, self.M if M is None else M, C.byref(st)),
              "tsb_pfsp_search_on")
        return st

    def pool_steal_from(self, victim: "PfspEvaluator", m: int) -> int:
        got = C.c_int64(0)
        check(lib().tsb_pfsp_pool_steal(victim._h, self._h, m, C.byref(got)), "tsb_pfsp_pool_steal")
        return int(got.value)

    def pool_drain(self) -> np.ndarray:
        n = self.pool_size
        out = np.empty(max(n, 1), dtype=self.node_dtype)
        got = C.c_int64(0)
        check(lib().tsb_pfsp_pool_drain(self._h, out.ctypes.data, n, C.byref(got)), "tsb_pfsp_pool_drain")
        return out[: got.value].copy()


def pfsp_search_device(inst: int = 14, lb="lb1", ub: int = 1, m: int = 25, M: int = 50000, D: int = 1) -> SearchStats:
    """same search, the pool(s) of step 2 resident on the device(s) (tsb_pfsp_pool_*); ta031..ta060 run as the
    MAX_JOBS = 50 build does"""
    kind = LB_NAMES[lb] if isinstance(lb, str) else int(lb)
    st = SearchStats()
    if _max_jobs(inst) == 50:
        check(lib().tsb_pfsp_search_device_wide(50, inst, kind, ub, m, M, D, C.byref(st)), "tsb_pfsp_search_device_wide")
    else:
        check(lib().tsb_pfsp_search_device(inst, kind, ub, m, M, D, C.byref(st)), "tsb_pfsp_search_device")
    return st


def pfsp_search(inst: int = 14, lb="lb1", ub: int = 1, m: int = 25, M: int = 50000, D: int = 1) -> SearchStats:
    """pfsp_gpu_chpl.chpl:306-431 (D = 1) / pfsp_multigpu_chpl.chpl (static split), C++ emulation driver; ta031..ta060
    run as the MAX_JOBS = 50 build does"""
    kind = LB_NAMES[lb] if isinstance(lb, str) else int(lb)
    st = SearchStats()
    if _max_jobs(inst) == 50:
        check(lib().tsb_pfsp_search_wide(50, inst, kind, ub, m, M, D, C.byref(st)), "tsb_pfsp_search_wide")
    else:
        check(lib().tsb_pfsp_search(inst, kind, ub, m, M, D, C.byref(st)), "tsb_pfsp_search")
    return st


def pfsp_search_device_part(inst: int, lb, ub: int, m: int, M: int, D: int, part: int, device: int = 0) -> SearchStats:
    kind = LB_NAMES[lb] if isinstance(lb, str) else int(lb)
    st = SearchStats()
    check(lib().tsb_pfsp_search_device_part(inst, kind, ub, m, M, D, part, device, C.byref(st)),
          "tsb_pfsp_search_device_part")
    return st
