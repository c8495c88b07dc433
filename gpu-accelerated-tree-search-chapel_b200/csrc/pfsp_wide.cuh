// pfsp_wide.cuh — PFSP bounds for the reference built with MAX_JOBS = 50 (SURVEY §8(f4), first slice).
//
// `config param MAX_JOBS = 20` (lib/pfsp/PFSP_node.chpl:7; C twin baselines/pfsp/lib/PFSP_node.h:10) is the
// compile-time width of a node's prmu; built with 50 the programs take ta031..ta060 (50 jobs x 5 / 10 / 20 machines)
// and every node is 8 + 4*50 = 208 bytes.  The tuned kernels of pfsp_kernels.cuh are specialised for 20 jobs
// (registers hold the whole permutation, 88-byte TMA tiles, 20-bit job masks, 5 groups of 4 slots).  This file is the
// general route: the same three evaluators (evaluate_gpu_lb1 / _lb1_d / _lb2, pfsp_gpu_chpl.chpl:192-254, and the
// device math of lib/pfsp/Bound_simple.chpl:29-222, Bound_johnson.chpl:179-289) for any jobs <= 50, machines <= 20,
// pairs <= 190, written for correctness and decent — not tuned — speed:
//   * persistent CTAs of 64 threads, one thread per parent, tiles of 64 nodes staged through shared memory with
//     coalesced 16-byte loads, bounds staged back the same way (only the defined slots k > limit1 are stored);
//   * all instance tables in shared memory (p_times job-major with an odd row stride; for lb2 one packed word per
//     (pair, position): job | p_a | p_b | lag, 38 KB for 190 pairs x 50 jobs);
//   * the parent's front / remain computed once per parent (as in pfsp_kernels.cuh), one child at a time;
//     lb1 on the child in the reference's own formulation (machine_bound_from_parts, :108-121), lb1_d as
//     add_front_and_bound (:197-222), lb2 with the scheduled set as a 64-bit mask and the reference's early exit.
#pragma once
#include <cstddef>

#include "tsb_ptx.cuh"

namespace tsb {

constexpr int PW_MAXJ = 50;
constexpr int PW_MAXM = 20;
constexpr int PW_MAXP = 190;
constexpr int PW_REC = 8 + 4 * PW_MAXJ;  // 208
constexpr int PW_THREADS = 64;
constexpr int PW_TILE = 64;
constexpr int PW_PSTRIDE = PW_MAXM + 1;  // odd row stride of the job-major processing times

struct PfspWideTables {
  int32_t jobs, machines, pairs, pad;
  int32_t total[PW_MAXM];
  int32_t min_heads[PW_MAXM];
  int32_t min_tails[PW_MAXM];
  int32_t pj[PW_MAXJ * PW_PSTRIDE];  // pj[job * PW_PSTRIDE + k]
  uint32_t pair[PW_MAXP + 4];        // in machine_pair_order: a | b << 5 | tail_a << 10 | tail_b << 21
  uint32_t jp[PW_MAXP * PW_MAXJ];    // jp[l * jobs + pos] = job | p_a << 6 | p_b << 13 | lag << 20
};
static_assert(sizeof(PfspWideTables) % 16 == 0 && offsetof(PfspWideTables, jp) % 16 == 0, "staged with 16-byte loads");

struct PfspWideSmem {
  alignas(16) PfspWideTables tab;
  alignas(16) int32_t in[PW_TILE * (PW_REC / 4)];
  alignas(16) int32_t out[PW_TILE * PW_MAXJ];
  int32_t fc[PW_MAXM * PW_THREADS];  // lb2: the child's front, [machine][thread] (dynamically indexed by pair)
};

// Bounds of the children of one parent — the per-parent part of evaluate_gpu_lb1 / _lb1_d / _lb2: the parent's
// front / remain (and, for lb2, its scheduled set) once, then emit(k, lb) for every slot k = limit1+1 .. jobs-1 in
// order, lb = the bound of the child that schedules prmu[k] next.  Shared by the evaluate kernel below and the count
// kernel of the fused expand (pfsp_wide_expand.cuh).  fc = this thread's column of PfspWideSmem::fc (stride
// PW_THREADS).  Returns the parent's limit1, clamped to [-1, jobs-1].
template <int KIND, int M, class Emit>
__device__ __forceinline__ int pw_parent_bounds(const PfspWideTables& tab, const int32_t* node, int32_t* fc, int best,
                                                Emit&& emit) {
  const int jobs = tab.jobs;
  const int limit1 = min(max(node[1], -1), jobs - 1);
  const int32_t* prmu = node + 2;
  int F[M], R[M];
#pragma unroll
  for (int j = 0; j < M; j++) {
    F[j] = 0;
    R[j] = tab.total[j];
  }
  if (KIND == 0 && limit1 < 0) {  // lb1_d on the root: front = min_heads (schedule_front, Bound_simple.chpl:53-57)
#pragma unroll
    for (int j = 0; j < M; j++) F[j] = tab.min_heads[j];
  }
  unsigned long long sched = 0;  // set_flags (Bound_johnson.chpl:179-186) as a bit mask
  for (int i = 0; i <= limit1; i++) {  // schedule_front / add_forward (:29-62); remain = total - scheduled
    const int job = prmu[i];
    const int32_t* row = &tab.pj[job * PW_PSTRIDE];
    sched |= 1ull << job;
    F[0] += row[0];
    R[0] -= row[0];
#pragma unroll
    for (int j = 1; j < M; j++) {
      F[j] = max(F[j - 1], F[j]) + row[j];
      R[j] -= row[j];
    }
  }
  for (int k = limit1 + 1; k < jobs; k++) {
    const int job = prmu[k];  // the child schedules prmu[k] next (prmu[depth] <=> prmu[k])
    const int32_t* row = &tab.pj[job * PW_PSTRIDE];
    int lb;
    if constexpr (KIND == 0) {  // add_front_and_bound (:197-222)
      lb = F[0] + R[0] + tab.min_tails[0];
      int tmp0 = F[0] + row[0];
#pragma unroll
      for (int i = 1; i < M; i++) {
        const int tmp1 = max(tmp0, F[i]);
        lb = max(lb, tmp1 + R[i] + tab.min_tails[i]);
        tmp0 = tmp1 + row[i];
      }
    } else if constexpr (KIND == 1) {  // lb1_bound on the child (:123-136): front_c, remain_c, running max
      int fcj = F[0] + row[0];
      int tmp0 = fcj + (R[0] - row[0]);
      lb = tmp0 + tab.min_tails[0];
#pragma unroll
      for (int i = 1; i < M; i++) {
        fcj = max(fcj, F[i]) + row[i];
        const int tmp1 = max(tmp0, fcj + (R[i] - row[i]));
        lb = max(lb, tmp1 + tab.min_tails[i]);
        tmp0 = tmp1;
      }
    } else {  // lb2_bound (Bound_johnson.chpl:274-289): child front, flags, lb_makespan with early exit
      int fcj = F[0] + row[0];
      fc[0 * PW_THREADS] = fcj;
#pragma unroll
      for (int i = 1; i < M; i++) {
        fcj = max(fcj, F[i]) + row[i];
        fc[i * PW_THREADS] = fcj;
      }
      const unsigned long long flags = sched | (1ull << job);
      lb = 0;
      for (int l = 0; l < tab.pairs; l++) {
        const uint32_t pw = tab.pair[l];
        const int a = pw & 31u, b = (pw >> 5) & 31u;
        int t0 = fc[a * PW_THREADS], t1 = fc[b * PW_THREADS];
        const uint32_t* jp = &tab.jp[l * jobs];
        for (int pos = 0; pos < jobs; pos++) {  // compute_cmax_johnson (:188-212)
          const uint32_t e = jp[pos];
          if (!((flags >> (e & 63u)) & 1ull)) {
            t0 += (e >> 6) & 127u;
            t1 = max(t1, t0 + static_cast<int>(e >> 20)) + static_cast<int>((e >> 13) & 127u);
          }
        }
        const int c = max(t1 + static_cast<int>(pw >> 21), t0 + static_cast<int>((pw >> 10) & 2047u));
        lb = max(lb, c);
        if (lb > best) break;  // :232-236
      }
    }
    emit(k, lb);
  }
  return limit1;
}

// the whole instance table into shared memory (lb1 / lb1_d never read the Johnson words); callers synchronise
template <int KIND>
__device__ __forceinline__ void pw_stage_tables(PfspWideTables* dst_tab, const PfspWideTables* __restrict__ tables) {
  const uint4* src = reinterpret_cast<const uint4*>(tables);
  uint4* dst = reinterpret_cast<uint4*>(dst_tab);
  const int n16 = static_cast<int>((KIND == 2 ? sizeof(PfspWideTables) : offsetof(PfspWideTables, jp)) / 16);
  for (int i = threadIdx.x; i < n16; i += blockDim.x) dst[i] = src[i];
}

template <int KIND, int M>
__global__ void __launch_bounds__(PW_THREADS) pfsp_wide_kernel(const uint8_t* __restrict__ parents,
                                                              int32_t* __restrict__ bounds, long long count,
                                                              const PfspWideTables* __restrict__ tables, int best) {
  extern __shared__ __align__(128) uint8_t smem_raw[];
  PfspWideSmem& sm = *reinterpret_cast<PfspWideSmem*>(smem_raw);
  const int t = threadIdx.x;
  pw_stage_tables<KIND>(&sm.tab, tables);
  __syncthreads();
  const PfspWideTables& tab = sm.tab;
  const int jobs = tab.jobs;
  const long long tiles = (count + PW_TILE - 1) / PW_TILE;
  for (long long tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
    const long long p0 = tile * PW_TILE;
    const int np = static_cast<int>(count - p0 < PW_TILE ? count - p0 : PW_TILE);
    {  // nodes of the tile: np * 208 bytes, 16-byte aligned (208 = 13 * 16)
      const uint4* src = reinterpret_cast<const uint4*>(parents + p0 * PW_REC);
      uint4* dst = reinterpret_cast<uint4*>(sm.in);
      for (int i = t; i < np * (PW_REC / 16); i += PW_THREADS) dst[i] = src[i];
    }
    __syncthreads();
    if (t < np) {
      int32_t* out = sm.out + t * jobs;
      pw_parent_bounds<KIND, M>(tab, sm.in + t * (PW_REC / 4), sm.fc + t, best, [&](int k, int lb) { out[k] = lb; });
    }
    __syncthreads();
    // bounds of the tile: only the defined slots (k > limit1) are stored
    for (int i = t; i < np * jobs; i += PW_THREADS) {
      const int p = i / jobs, k = i - p * jobs;
      if (k > sm.in[p * (PW_REC / 4) + 1]) bounds[(p0 + p) * jobs + k] = sm.out[i];
    }
    __syncthreads();
  }
}

}  // namespace tsb
