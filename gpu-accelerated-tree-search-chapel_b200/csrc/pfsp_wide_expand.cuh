// pfsp_wide_expand.cuh — fused evaluate + generate_children of one round for 208-byte nodes (a MAX_JOBS = 50
// build: ta031..ta060).  The same contract as pfsp_expand.cuh — children PACKED and IN THE REFERENCE'S ORDER,
// `best` the value at launch for the whole chunk, the minimum leaf bound reported through ExpandState so that the
// host redoes a round in which a leaf lowers `best` — and the same two-kernel shape:
//   pfsp_wide_expand_count : tiles of 64 parents read in place (TMA bulk copy + mbarrier, run_piece_tiles); the
//                            bounds of pw_parent_bounds (the code of the evaluate kernel, pfsp_wide.cuh); one 64-bit
//                            child mask per parent, one child count per tile, leaf statistics
//   pfsp_wide_expand_build : offsets of the CTA's own tiles (prologue), then per tile: one thread per child copies
//                            the parent (13 x 16 B) into a shared-memory image and patches depth, limit1 and the
//                            swap; one TMA bulk store writes the image.  208 = 13 * 16, so every child of a
//                            16-byte aligned destination is itself 16-byte aligned.
#pragma once
#include "expand_common.cuh"
#include "pfsp_expand.cuh"  // run_piece_tiles
#include "pfsp_wide.cuh"

namespace tsb {

constexpr int PW_EXP_CAP = 256;  // children per pass of the staging image (a tile of 64 parents has up to 64 * 49)

// ------------------------------------------------------------------------------------------- count
struct PwCountSmem {
  alignas(16) PfspWideTables tab;
  alignas(128) uint8_t in[2][PW_TILE * PW_REC];
  int32_t fc[PW_MAXM * PW_THREADS];
  alignas(8) uint64_t full[2];
  int red[PW_THREADS / 32];
};

template <int KIND, int M>
__global__ void __launch_bounds__(PW_THREADS) pfsp_wide_expand_count_kernel(const uint8_t* __restrict__ arena,
                                                                           const __grid_constant__ ExpandParams prm,
                                                                           const PfspWideTables* __restrict__ tables,
                                                                           unsigned long long* __restrict__ cmask,
                                                                           int* __restrict__ tile_sums,
                                                                           ExpandState* __restrict__ st) {
  extern __shared__ __align__(128) uint8_t smem_raw[];
  PwCountSmem& sm = *reinterpret_cast<PwCountSmem*>(smem_raw);
  pw_stage_tables<KIND>(&sm.tab, tables);  // (run_piece_tiles synchronises before the first tile)
  const int t = threadIdx.x, best = prm.best;
  unsigned my_solutions = 0;
  run_piece_tiles<2, PW_TILE, PW_REC>(
      sm.in[0], sm.full, arena, prm, [&](const uint8_t* in_tile, int lin, long long at, long long lo, long long hi) {
        const int rec_lo = static_cast<int>(lo - at * PW_TILE), rec_hi = static_cast<int>(hi - at * PW_TILE);
        unsigned long long m = 0;
        int leaves = 0;
        if (t >= rec_lo && t < rec_hi) {
          const int32_t* node = reinterpret_cast<const int32_t*>(in_tile) + t * (PW_REC / 4);
          unsigned long long live = 0;
          int leaf_lb = 0x7FFFFFFF;
          pw_parent_bounds<KIND, M>(sm.tab, node, sm.fc + t, best, [&](int k, int lb) {
            live |= 1ull << k;
            if (lb < best) m |= 1ull << k;
            leaf_lb = min(leaf_lb, lb);
          });
          if (live && node[0] + 1 == sm.tab.jobs) {  // every child is a leaf (pfsp_gpu_chpl.chpl:283-288)
            leaves = __popcll(live);
            m = 0;
            if (leaf_lb < best) atomicMin(&st->best, leaf_lb);
          }
        }
        // children of a tile <= 64 * 50 < 2^16, leaves likewise: one packed sum
        int packed = __popcll(m) | (leaves << 16);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) packed += __shfl_xor_sync(0xFFFFFFFFu, packed, o);
        if ((t & 31) == 0) sm.red[t >> 5] = packed;
        cmask[static_cast<long long>(lin) * PW_TILE + t] = m;
        __syncthreads();
        if (t == 0) {
          const int tot = sm.red[0] + sm.red[1];
          tile_sums[lin] = tot & 0xFFFF;
          my_solutions += static_cast<unsigned>(tot >> 16);
        }
      });
  if (t == 0 && my_solutions) atomicAdd(&st->solutions, static_cast<unsigned long long>(my_solutions));
}

// ------------------------------------------------------------------------------------------- build
struct PwBuildSmem {
  alignas(128) uint8_t in[2][PW_TILE * PW_REC];
  alignas(128) unsigned long long mask[2][PW_TILE];
  alignas(128) uint8_t stage[PW_EXP_CAP * PW_REC];
  alignas(8) uint64_t full[2];
  uint16_t item[PW_EXP_CAP];  // (record << 6) | slot, in child order
  int warp_tot[PW_THREADS / 32];
  ScanSmem scan;
};
static_assert(PW_THREADS == 64, "the scans below combine two warps");

// (min blocks 1: shared memory holds two CTAs per SM anyway; without it ptxas aims at 48 registers and spills)
__global__ void __launch_bounds__(PW_THREADS, 1) pfsp_wide_expand_build_kernel(const uint8_t* __restrict__ arena,
                                                                           const __grid_constant__ ExpandParams prm,
                                                                           const unsigned long long* __restrict__ cmask,
                                                                           const int* __restrict__ tile_sums,
                                                                           uint8_t* __restrict__ children,
                                                                           ExpandState* __restrict__ st,
                                                                           ExpandResult* __restrict__ res) {
  extern __shared__ __align__(128) uint8_t smem_raw[];
  PwBuildSmem& sm = *reinterpret_cast<PwBuildSmem*>(smem_raw);
  const int t = threadIdx.x, lane = t & 31, wid = t >> 5;
  constexpr uint32_t IN_BYTES = PW_TILE * PW_REC;
  const int first = blockIdx.x, stride = gridDim.x;
  if (t == 0) {
    mbar_init(&sm.full[0], 1);
    mbar_init(&sm.full[1], 1);
    mbar_fence_init();
  }
  __syncthreads();
  uint64_t pol = 0;
  if (t == 0) pol = policy_evict_first();
  auto issue = [&](int lin, int s) {  // thread 0: parents + masks of one tile
    long long at, lo, hi;
    piece_of(prm, lin, PW_TILE, at, lo, hi);
    const uint32_t nb = tile_load_bytes(at, hi, PW_TILE, PW_REC);
    mbar_arrive_expect_tx(&sm.full[s], nb + PW_TILE * 8);
    if (nb) bulk_g2s_stream(sm.in[s], arena + at * IN_BYTES, nb, &sm.full[s], pol);
    bulk_g2s_stream(sm.mask[s], cmask + static_cast<long long>(lin) * PW_TILE, PW_TILE * 8, &sm.full[s], pol);
  };
  if (t == 0) {
    if (first < prm.n_tiles) issue(first, 0);
    if (first + stride < prm.n_tiles) issue(first + stride, 1);
  }
  expand_own_offsets<PW_THREADS>(sm.scan, tile_sums, prm.n_tiles, first, stride);
  expand_publish(sm.scan, st, res, prm.epoch, 1);  // st->best restarts at INT_MAX every round
  unsigned it = 0;
  for (int lin = first; lin < prm.n_tiles; lin += stride, it++) {
    const int s = it & 1;
    mbar_wait(&sm.full[s], (it >> 1) & 1u);
    const unsigned long long cm = sm.mask[s][t];
    const int mine = __popcll(cm);
    int incl = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int y = __shfl_up_sync(0xFFFFFFFFu, incl, o);
      if (lane >= o) incl += y;
    }
    if (lane == 31) sm.warp_tot[wid] = incl;
    if (t == 0) bulk_wait_read<0>();  // the previous tile's bulk store has drained the staging image
    __syncthreads();  // (A)
    const int total = sm.warp_tot[0] + sm.warp_tot[1];
    const int pos0 = (wid ? sm.warp_tot[0] : 0) + incl - mine;  // index (within the tile) of this parent's first child
    uint8_t* const gtile = children + static_cast<long long>(sm.scan.own[it]) * PW_REC;
    for (int c0 = 0; c0 < total; c0 += PW_EXP_CAP) {  // windows of PW_EXP_CAP children
      const int cnt = min(PW_EXP_CAP, total - c0);
      if (c0 > 0 && t == 0) bulk_wait_read<0>();
      if (pos0 < c0 + PW_EXP_CAP && pos0 + mine > c0) {
        int pos = pos0 - c0;
        unsigned long long m = cm;
        while (m) {
          const int k = __ffsll(static_cast<long long>(m)) - 1;
          m &= m - 1;
          if (pos >= 0 && pos < PW_EXP_CAP) sm.item[pos] = static_cast<uint16_t>((t << 6) | k);
          pos++;
        }
      }
      __syncthreads();  // (B) items
      for (int c = t; c < cnt; c += PW_THREADS) {
        const int item = sm.item[c];
        const int r = item >> 6, k = item & 63;
        const uint4* src = reinterpret_cast<const uint4*>(sm.in[s] + r * PW_REC);
        uint4* d = reinterpret_cast<uint4*>(sm.stage + c * PW_REC);
        uint4 head = src[0];
#pragma unroll
        for (int i = 1; i < PW_REC / 16; i++) d[i] = src[i];
        const int depth = static_cast<int>(head.x);
        head.x = static_cast<uint32_t>(depth + 1);  // depth + 1
        head.y = head.y + 1u;                       // limit1 + 1
        d[0] = head;
        const int32_t* sp = reinterpret_cast<const int32_t*>(src) + 2;
        int32_t* dp = reinterpret_cast<int32_t*>(d) + 2;
        const int a = sp[depth], b = sp[k];  // child.prmu[depth] <=> child.prmu[k]
        dp[depth] = b;
        dp[k] = a;
      }
      fence_async_smem();
      __syncthreads();  // (C) image complete
      if (t == 0) {
        bulk_s2g(gtile + static_cast<long long>(c0) * PW_REC, sm.stage, static_cast<uint32_t>(cnt * PW_REC));
        bulk_commit();
      }
    }
    // a tile without children has no barrier after (A): without this one a fast warp could overwrite warp_tot
    // for tile it+1 while the other warp still reads the totals of tile it
    if (total == 0) __syncthreads();
    if (t == 0 && lin + 2 * stride < prm.n_tiles) issue(lin + 2 * stride, s);
  }
  if (t == 0) bulk_wait_all();
}

}  // namespace tsb
