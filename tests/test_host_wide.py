"""CPU-only checks of the MAX_JOBS = 50 search entry points (tsb_pfsp_search_wide / _search_device_wide): arguments
are validated before any device is touched, so these run without a GPU.  No search is started."""
import ctypes as C
import os
import subprocess

import pytest

import tsb200
from tsb200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FNS = ("tsb_pfsp_search_wide", "tsb_pfsp_search_device_wide")


@pytest.mark.parametrize("fn", FNS)
def test_wide_search_argument_checks(fn):
    f = getattr(tsb200.lib(), fn)
    st = _lib.SearchStats()
    lb1 = tsb200.LB_NAMES["lb1"]
    for max_jobs in (0, 19, 21, 30, 49, 51, 100):
        assert f(max_jobs, 31, lb1, 1, 25, 50000, 1, C.byref(st)) == _lib.EUNSUPPORTED
    for inst in (14, 30, 61, 120):  # the MAX_JOBS = 50 build takes the 50-job instances only
        assert f(50, inst, lb1, 1, 25, 50000, 1, C.byref(st)) == _lib.EUNSUPPORTED
    assert f(20, 31, lb1, 1, 25, 50000, 1, C.byref(st)) == _lib.EUNSUPPORTED  # 50 jobs > MAX_JOBS = 20
    for inst in (0, 121):
        assert f(50, inst, lb1, 1, 25, 50000, 1, C.byref(st)) == _lib.EINVAL
    for max_jobs, inst in ((50, 31), (20, 14)):
        assert f(max_jobs, inst, 3, 1, 25, 50000, 1, C.byref(st)) == _lib.EINVAL  # lb_kind
        assert f(max_jobs, inst, -1, 1, 25, 50000, 1, C.byref(st)) == _lib.EINVAL
        assert f(max_jobs, inst, lb1, 2, 25, 50000, 1, C.byref(st)) == _lib.EINVAL  # ub
        assert f(max_jobs, inst, lb1, 1, 0, 50000, 1, C.byref(st)) == _lib.EINVAL  # m
        assert f(max_jobs, inst, lb1, 1, 25, 0, 1, C.byref(st)) == _lib.EINVAL  # M
        assert f(max_jobs, inst, lb1, 1, 25, 50000, 9, C.byref(st)) == _lib.EINVAL  # D
        assert f(max_jobs, inst, lb1, 1, 25, 50000, 1, None) == _lib.EINVAL


def test_python_search_routes_by_instance():
    """pfsp_search / pfsp_search_device pick the wide entry points for ta031..ta060: a bad argument comes back from
    those (the 20-job entry points answer EUNSUPPORTED for ta031)"""
    for fn in (tsb200.pfsp_search, tsb200.pfsp_search_device):
        with pytest.raises(tsb200.TsbError) as e:
            fn(31, 3)
        assert e.value.code == _lib.EINVAL and "_wide" in str(e.value)
        with pytest.raises(tsb200.TsbError) as e:
            fn(14, 3)
        assert e.value.code == _lib.EINVAL and "_wide" not in str(e.value)
        with pytest.raises(tsb200.TsbError) as e:
            fn(61)
        assert e.value.code == _lib.EUNSUPPORTED


def test_driver_rejects_instances_beyond_50_jobs():
    exe = os.path.join(ROOT, "gpu-accelerated-tree-search-chapel_b200", "drivers", "pfsp_b200.out")
    if not os.path.exists(exe):
        pytest.skip("drivers not built")
    r = subprocess.run([exe, "--inst", "61"], capture_output=True, text=True, timeout=60)
    assert r.returncode == 2 and "ta061" in r.stderr
