"""Times the offload rounds of 50-job searches (a MAX_JOBS = 50 build, 208-byte nodes) two ways on the same chunk
sequence and checks that they count the same:
  device  tsb_pfsp_pool_step: the pool in HBM, fused evaluate + generate_children (count + build kernels);
  drop-in tsb_pfsp_evaluate of the chunk + generate_children on the host (the pool on the host), i.e. what a
          patched Chapel driver built with -sMAX_JOBS=50 does per round.
Per instance (ta031, ta041, ta051) and bound (lb1, lb2), --ub 1, M = 50 000: a host warm-up (drop-in rounds from the
root until the pool holds M nodes), then K rounds (default 50) of each path from that pool.  Reports us per round,
parents/s and children/s end to end; count- and build-kernel time from a separate profiled pass (torch.profiler,
CUDA activities); bytes moved (parents x 208 x 2 + children x 208) over kernel time as a share of 7.7 TB/s; the
card's name and power limit, read in the same run.  One JSON line per case; also written to OUT_DIR if given.

    python tools/pfsp_wide_rounds.py [--rounds K] [--max-pool NODES] [OUT_DIR]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                                "gpu-accelerated-tree-search-chapel_b200"))
import tsb200  # noqa: E402

HBM_BYTES_S = 7.7e12  # HGX B200 data sheet, one GPU


def generate_children(parents, bounds, best, jobs=50):
    """generate_children (pfsp_gpu_chpl.chpl:273-303) for a constant best (--ub 1): children in the reference's order"""
    b = bounds.reshape(-1, jobs)
    live = np.arange(jobs)[None, :] > parents["limit1"][:, None]
    leaf = (parents["depth"] + 1 == jobs)[:, None]
    sol = int((live & leaf).sum())
    keep = live & ~leaf & (b < best)
    i, j = np.nonzero(keep)  # row-major = parents in order, slots ascending
    kids = parents[i].copy()
    d = kids["depth"].astype(np.int64)
    r = np.arange(kids.shape[0])
    a, c = kids["prmu"][r, d].copy(), kids["prmu"][r, j].copy()
    kids["prmu"][r, d], kids["prmu"][r, j] = c, a
    kids["depth"] += 1
    kids["limit1"] += 1
    return kids, sol


def dropin_round(ev, pool, lb, M, best):
    n = min(pool.shape[0], M)
    chunk = np.ascontiguousarray(pool[pool.shape[0] - n:])
    bounds = ev.evaluate(chunk, lb, best)
    kids, sol = generate_children(chunk, bounds, best)
    return np.concatenate([pool[: pool.shape[0] - n], kids]), (n, kids.shape[0], sol)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = [x.strip() for x in q.split(",")[:2]]
        return {"gpu": name, "power_limit": power}
    except Exception as e:  # (the name still comes from the runtime)
        import torch
        return {"gpu": torch.cuda.get_device_name(0), "power_limit": f"unknown ({e})"}


def run_case(inst, lb, K, M, max_pool):
    import torch
    best = int(tsb200.lib().tsb_taillard_best_ub(inst))
    root = np.zeros(1, dtype=tsb200.PFSP_NODE50_DTYPE)
    root["limit1"] = -1
    root["prmu"][0] = np.arange(50)
    with tsb200.PfspEvaluator(inst, M=M) as ev:
        pool = root
        while 0 < pool.shape[0] < M:  # host warm-up
            pool, _ = dropin_round(ev, pool, lb, M, best)
        start = pool.copy()
        # drop-in path, on the host pool
        counts_d, t0 = [], time.perf_counter()
        for _ in range(K):  # (a case stops early when the host pool outgrows max_pool)
            if pool.shape[0] == 0 or pool.shape[0] > max_pool:
                break
            pool, c = dropin_round(ev, pool, lb, M, best)
            counts_d.append(c)
        t_dropin = time.perf_counter() - t0
        # device path, same start pool: warm once (modules, arena), then the timed rounds
        stream = torch.cuda.ExternalStream(tsb200.lib().tsb_pfsp_stream(ev._h))
        ev.pool_push(start)
        ev.pool_step(lb, 1, M, best)
        ev.pool_drain()

        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

        def device_rounds():  # (the events bracket the rounds only, not the push of the start pool or the drain)
            ev.pool_push(start)
            out = []
            e0.record(stream)
            for _ in range(len(counts_d)):
                n, c, s, _ = ev.pool_step(lb, 1, M, best)
                out.append((n, c, s))
            e1.record(stream)
            e1.synchronize()
            ev.pool_drain()
            return out

        counts_g = device_rounds()
        t_device = e0.elapsed_time(e1) / 1e3
        assert counts_g == counts_d, "device rounds and drop-in rounds differ"
        # kernel times: a separate pass under the profiler
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            assert device_rounds() == counts_d
            torch.cuda.synchronize()
        k = {"count": 0.0, "build": 0.0}
        for evt in prof.events():
            if evt.device_type.name == "CUDA":
                if "pfsp_wide_expand_count" in evt.name:
                    k["count"] += evt.device_time_total / 1e6
                elif "pfsp_wide_expand_build" in evt.name:
                    k["build"] += evt.device_time_total / 1e6
    rounds = len(counts_d)
    P = sum(c[0] for c in counts_d)
    Ch = sum(c[1] for c in counts_d)
    kt = k["count"] + k["build"]
    moved = P * 208 * 2 + Ch * 208
    return {"inst": inst, "lb": lb, "M": M, "rounds": rounds, "start_pool": int(start.shape[0]), "parents": P,
            "children": Ch, "solutions": sum(c[2] for c in counts_d),
            "device_us_per_round": t_device / max(rounds, 1) * 1e6, "dropin_us_per_round": t_dropin / max(rounds, 1) * 1e6,
            "device_parents_s": P / t_device, "device_children_s": Ch / t_device,
            "dropin_parents_s": P / t_dropin, "dropin_children_s": Ch / t_dropin,
            "count_kernel_s": k["count"], "build_kernel_s": k["build"],
            "bytes_over_kernel_time_share_of_hbm": moved / kt / HBM_BYTES_S if kt > 0 else None}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=50)
    ap.add_argument("--M", type=int, default=50000)
    ap.add_argument("--max-pool", type=int, default=12_000_000, help="stop a case when the host pool exceeds this")
    ap.add_argument("--inst", type=int, nargs="*", default=[31, 41, 51])
    ap.add_argument("--lb", nargs="*", default=["lb1", "lb2"])
    ap.add_argument("out_dir", nargs="?")
    a = ap.parse_args()
    info = card()
    lines = []
    for inst in a.inst:
        for lb in a.lb:
            r = dict(run_case(inst, lb, a.rounds, a.M, a.max_pool), **info)
            print(json.dumps(r), flush=True)
            lines.append(r)
    if a.out_dir:
        os.makedirs(a.out_dir, exist_ok=True)
        with open(os.path.join(a.out_dir, "pfsp_wide_rounds.json"), "w") as f:
            json.dump(lines, f, indent=1)


if __name__ == "__main__":
    main()
