// tsb200_api.cu — C ABI of libtsb200.so (include/tsb200.h): handles, transfers, kernel launches.
#include <cuda_runtime.h>

#include <sched.h>

#include <algorithm>
#include <cctype>
#include <atomic>
#include <chrono>
#include <climits>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <new>
#include <string>
#include <vector>

#include "nq_expand.cuh"
#include "nq_expand2.cuh"
#include "nq_rounds.cuh"
#include "nq_rounds_ll.cuh"
#include "pfsp_expand.cuh"
#include "nq_kernel.cuh"
#include "pfsp_kernels.cuh"
#include "pfsp_wide.cuh"
#include "pfsp_wide_expand.cuh"
#include "tsb200.h"

namespace {

thread_local std::string g_last_cuda_error;

#define TSB_CUDA(call)                                                                         \
  do {                                                                                         \
    cudaError_t e__ = (call);                                                                  \
    if (e__ != cudaSuccess) {                                                                  \
      g_last_cuda_error = std::string(#call) + ": " + cudaGetErrorString(e__);                 \
      (void)cudaGetLastError();                                                                \
      return e__ == cudaErrorMemoryAllocation ? TSB_ENOMEM : TSB_ECUDA;                        \
    }                                                                                          \
  } while (0)

// (env TSB200_POOL_CAP overrides the initial arena capacity, so that tests can force compaction and growth)
long long env_pool_cap() {
  const char* v = std::getenv("TSB200_POOL_CAP");
  return v ? std::atoll(v) : 0;
}
int env_xfer() {
  const char* s = std::getenv("TSB200_XFER");
  if (!s) return TSB_XFER_AUTO;
  if (!std::strcmp(s, "memcpy")) return TSB_XFER_MEMCPY;
  if (!std::strcmp(s, "zerocopy")) return TSB_XFER_ZEROCOPY;
  return TSB_XFER_AUTO;
}
bool env_no_register() {
  const char* s = std::getenv("TSB200_NO_REGISTER");
  return s && *s && *s != '0';
}

// Host ranges the CALLER asked to page-lock + map (tsb_*_register_host): cudaMemcpyAsync is truly asynchronous
// on them and the zero-copy kernels can address them.  Registration is explicit and the caller owns the
// lifetime: a range must stay allocated until it is unregistered or the handle is destroyed (a registration
// keyed on an address alone goes stale when the array is freed and another one lands on the same addresses).
// Arrays that were never registered go through the handle's own pinned staging buffers.
struct HostRange {
  uintptr_t base;
  size_t len;
};
struct HostRegistry {
  std::vector<HostRange> ranges;
  bool disabled = env_no_register();
  bool contains(const void* p, size_t bytes) const {
    if (!p || !bytes) return false;
    const uintptr_t a = reinterpret_cast<uintptr_t>(p), b = a + bytes;
    for (const auto& r : ranges)
      if (a >= r.base && b <= r.base + r.len) return true;
    return false;
  }
  // TSB_OK, or TSB_EINVAL for a range that partly overlaps a registered one, or TSB_ECUDA
  int add(void* p, size_t bytes) {
    if (!p || !bytes) return TSB_EINVAL;
    if (disabled || contains(p, bytes)) return TSB_OK;
    const uintptr_t a = reinterpret_cast<uintptr_t>(p), b = a + bytes;
    for (const auto& r : ranges)
      if (r.base < b && a < r.base + r.len) return TSB_EINVAL;
    TSB_CUDA(cudaHostRegister(p, bytes, cudaHostRegisterPortable | cudaHostRegisterMapped));
    ranges.push_back({a, bytes});
    return TSB_OK;
  }
  int remove(void* p) {
    const uintptr_t a = reinterpret_cast<uintptr_t>(p);
    for (size_t i = 0; i < ranges.size(); i++)
      if (ranges[i].base == a) {
        cudaHostUnregister(p);
        ranges.erase(ranges.begin() + i);
        return TSB_OK;
      }
    return disabled ? TSB_OK : TSB_EINVAL;
  }
  void release() {
    for (auto& r : ranges) cudaHostUnregister(reinterpret_cast<void*>(r.base));
    ranges.clear();
  }
};

struct DeviceInfo {
  int sms = 0;
  bool can_use_host_ptr = false;
  bool coop = false;  // cooperative launches (the persistent multi-round kernel)
};
int query_device(int device, DeviceInfo& di) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    (void)cudaGetLastError();
    return TSB_ENODEV;
  }
  if (device < 0 || device >= n) return TSB_ENODEV;
  TSB_CUDA(cudaSetDevice(device));
  TSB_CUDA(cudaDeviceGetAttribute(&di.sms, cudaDevAttrMultiProcessorCount, device));
  int v = 0;
  TSB_CUDA(cudaDeviceGetAttribute(&v, cudaDevAttrCanUseHostPointerForRegisteredMem, device));
  di.can_use_host_ptr = v != 0;
  TSB_CUDA(cudaDeviceGetAttribute(&v, cudaDevAttrCooperativeLaunch, device));
  di.coop = v != 0;
  return TSB_OK;
}

// common part of both handle types
struct Base {
  int device = 0, M_max = 0, xfer = TSB_XFER_AUTO;
  DeviceInfo di;
  cudaStream_t stream = nullptr, stream2 = nullptr;
  int pipe_min = 131072;  // records from which the memcpy path is split over two streams (env TSB200_PIPE_MIN)
  int pipe_chunk = 262144;
  uint8_t *d_in = nullptr, *d_out = nullptr;  // device chunk buffers (M_max records)
  uint8_t *h_in = nullptr, *h_out = nullptr;  // pinned+mapped staging, used when the caller's arrays cannot be locked
  size_t in_rec = 0, out_rec = 0;
  HostRegistry reg;
  uint64_t launches = 0;

  int init(int dev, int M, size_t irec, size_t orec) {
    device = dev;
    M_max = M;
    in_rec = irec;
    out_rec = orec;
    xfer = env_xfer();
    int rc = query_device(dev, di);
    if (rc != TSB_OK) return rc;
    TSB_CUDA(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
    TSB_CUDA(cudaStreamCreateWithFlags(&stream2, cudaStreamNonBlocking));
    if (const char* v = std::getenv("TSB200_PIPE_MIN")) pipe_min = std::max(1, std::atoi(v));
    if (const char* v = std::getenv("TSB200_PIPE_CHUNK")) pipe_chunk = std::max(1024, std::atoi(v)) & ~1023;
    TSB_CUDA(cudaMalloc(&d_in, in_rec * M + 256));
    TSB_CUDA(cudaMalloc(&d_out, out_rec * M + 256));
    return TSB_OK;
  }
  int ensure_staging() {
    if (!h_in) TSB_CUDA(cudaHostAlloc(&h_in, in_rec * M_max + 256, cudaHostAllocPortable | cudaHostAllocMapped));
    if (!h_out) TSB_CUDA(cudaHostAlloc(&h_out, out_rec * M_max + 256, cudaHostAllocPortable | cudaHostAllocMapped));
    return TSB_OK;
  }
  void fini() {
    cudaSetDevice(device);
    if (stream) cudaStreamSynchronize(stream);
    reg.release();
    if (d_in) cudaFree(d_in);
    if (d_out) cudaFree(d_out);
    if (h_in) cudaFreeHost(h_in);
    if (h_out) cudaFreeHost(h_out);
    if (bounce) cudaFreeHost(bounce);
    if (bounce_ev[0]) cudaEventDestroy(bounce_ev[0]);
    if (bounce_ev[1]) cudaEventDestroy(bounce_ev[1]);
    if (stream) cudaStreamDestroy(stream);
    if (stream2) cudaStreamDestroy(stream2);
  }

  // Copies between a caller-owned host range and the device, ordered on stream `s` (the stream the kernels
  // that produce / consume the data run on), synchronous.  Registered ranges are copied directly; anything else
  // bounces through two pinned buffers so that the host memcpy of one piece overlaps the DMA of the previous one.
  uint8_t* bounce = nullptr;
  cudaEvent_t bounce_ev[2] = {nullptr, nullptr};
  static constexpr size_t kBounce = 1 << 20;
  int ensure_bounce() {
    if (!bounce) {
      TSB_CUDA(cudaHostAlloc(&bounce, 2 * kBounce, cudaHostAllocPortable));
      TSB_CUDA(cudaEventCreateWithFlags(&bounce_ev[0], cudaEventDisableTiming));
      TSB_CUDA(cudaEventCreateWithFlags(&bounce_ev[1], cudaEventDisableTiming));
    }
    return TSB_OK;
  }
  int copy_h2d(void* dst_d, const void* src_h, size_t bytes, cudaStream_t s) {
    if (!bytes) return TSB_OK;
    if (reg.contains(src_h, bytes)) {
      TSB_CUDA(cudaMemcpyAsync(dst_d, src_h, bytes, cudaMemcpyHostToDevice, s));
      TSB_CUDA(cudaStreamSynchronize(s));
      return TSB_OK;
    }
    if (int rc = ensure_bounce(); rc != TSB_OK) return rc;
    int i = 0;
    for (size_t off = 0; off < bytes; off += kBounce, i++) {
      const size_t n = std::min(kBounce, bytes - off);
      uint8_t* b = bounce + (i & 1) * kBounce;
      if (i >= 2) TSB_CUDA(cudaEventSynchronize(bounce_ev[i & 1]));  // the DMA that last read this buffer is done
      std::memcpy(b, static_cast<const uint8_t*>(src_h) + off, n);
      TSB_CUDA(cudaMemcpyAsync(static_cast<uint8_t*>(dst_d) + off, b, n, cudaMemcpyHostToDevice, s));
      TSB_CUDA(cudaEventRecord(bounce_ev[i & 1], s));
    }
    TSB_CUDA(cudaStreamSynchronize(s));
    return TSB_OK;
  }
  int copy_d2h(void* dst_h, const void* src_d, size_t bytes, cudaStream_t s) {
    if (!bytes) return TSB_OK;
    if (reg.contains(dst_h, bytes)) {
      TSB_CUDA(cudaMemcpyAsync(dst_h, src_d, bytes, cudaMemcpyDeviceToHost, s));
      TSB_CUDA(cudaStreamSynchronize(s));
      return TSB_OK;
    }
    if (int rc = ensure_bounce(); rc != TSB_OK) return rc;
    const size_t pieces = (bytes + kBounce - 1) / kBounce;
    for (size_t i = 0; i <= pieces; i++) {  // DMA of piece i overlaps the host memcpy of piece i-1
      if (i < pieces) {
        const size_t off = i * kBounce, n = std::min(kBounce, bytes - off);
        TSB_CUDA(cudaMemcpyAsync(bounce + (i & 1) * kBounce, static_cast<const uint8_t*>(src_d) + off, n,
                                 cudaMemcpyDeviceToHost, s));
        TSB_CUDA(cudaEventRecord(bounce_ev[i & 1], s));
      }
      if (i >= 1) {
        const size_t off = (i - 1) * kBounce, n = std::min(kBounce, bytes - off);
        TSB_CUDA(cudaEventSynchronize(bounce_ev[(i - 1) & 1]));
        std::memcpy(static_cast<uint8_t*>(dst_h) + off, bounce + ((i - 1) & 1) * kBounce, n);
      }
    }
    return TSB_OK;
  }

  // Host-buffer evaluation shared by N-Queens and PFSP.  `launch(in_dev, out_dev, count, stream)`
  // enqueues the evaluator kernel.
  template <class Launch>
  int evaluate_host(const void* in, int count, void* out, Launch&& launch) {
    const size_t in_b = in_rec * count, out_b = out_rec * count;
    const bool in_locked = reg.contains(in, in_b), out_locked = reg.contains(out, out_b);
    // AUTO: zero-copy whenever the caller registered its arrays (tsb_*_register_host) and they are 16-byte
    // aligned (measured fastest at every chunk size, profiles/xfer_sweep_r1.txt); otherwise copies, pipelined
    // when large, through the handle's pinned staging buffers for arrays that are not registered
    const bool aligned = ((reinterpret_cast<uintptr_t>(in) | reinterpret_cast<uintptr_t>(out)) & 15) == 0;
    const bool zc_ok = in_locked && out_locked && aligned && di.can_use_host_ptr;
    int mode = xfer == TSB_XFER_AUTO ? (zc_ok ? TSB_XFER_ZEROCOPY : TSB_XFER_MEMCPY) : xfer;
    if (mode == TSB_XFER_ZEROCOPY && !zc_ok) mode = TSB_XFER_MEMCPY;

    if (mode == TSB_XFER_ZEROCOPY) {
      // the kernel's TMA engine pulls the chunk over PCIe and pushes the results back: one launch,
      // reads and writes overlap on the full-duplex link
      int rc = launch(static_cast<const uint8_t*>(in), static_cast<uint8_t*>(out), count, stream);
      if (rc != TSB_OK) return rc;
      TSB_CUDA(cudaStreamSynchronize(stream));
      return TSB_OK;
    }
    const uint8_t* src = static_cast<const uint8_t*>(in);
    uint8_t* dst = static_cast<uint8_t*>(out);
    if (!in_locked || !out_locked) {
      int rc = ensure_staging();
      if (rc != TSB_OK) return rc;
    }
    if (!in_locked) src = h_in;
    if (!out_locked) dst = h_out;
    if (count >= pipe_min && count > pipe_chunk) {
      // large chunk: sub-chunks alternate between two streams so that the upload of one overlaps the
      // download of the previous one (PCIe is full duplex) and the kernel of the one in between; the host
      // memcpy into the staging buffer of sub-chunk i+1 overlaps the device work of sub-chunk i
      const cudaStream_t st[2] = {stream, stream2};
      int i = 0;
      for (int off = 0; off < count; off += pipe_chunk, ++i) {
        const int n = std::min(pipe_chunk, count - off);
        cudaStream_t s = st[i & 1];
        if (!in_locked) std::memcpy(h_in + in_rec * off, static_cast<const uint8_t*>(in) + in_rec * off, in_rec * n);
        TSB_CUDA(cudaMemcpyAsync(d_in + in_rec * off, src + in_rec * off, in_rec * n, cudaMemcpyHostToDevice, s));
        int rc = launch(d_in + in_rec * off, d_out + out_rec * off, n, s);
        if (rc != TSB_OK) return rc;
        TSB_CUDA(cudaMemcpyAsync(dst + out_rec * off, d_out + out_rec * off, out_rec * n, cudaMemcpyDeviceToHost, s));
      }
      TSB_CUDA(cudaStreamSynchronize(stream));
      TSB_CUDA(cudaStreamSynchronize(stream2));
    } else {
      if (!in_locked) std::memcpy(h_in, in, in_b);
      TSB_CUDA(cudaMemcpyAsync(d_in, src, in_b, cudaMemcpyHostToDevice, stream));
      int rc = launch(d_in, d_out, count, stream);
      if (rc != TSB_OK) return rc;
      TSB_CUDA(cudaMemcpyAsync(dst, d_out, out_b, cudaMemcpyDeviceToHost, stream));
      TSB_CUDA(cudaStreamSynchronize(stream));
    }
    if (!out_locked) std::memcpy(out, h_out, out_b);
    return TSB_OK;
  }
};

// persistent grid: enough CTAs to fill the GPU, never more than there are full tiles
template <class K>
int grid_for(K kernel, int threads, size_t smem, long long count, int tile, int sms, int* grid, int* cache) {
  int per_sm = *cache;
  if (per_sm <= 0) {
    TSB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, smem));
    if (per_sm < 1) per_sm = 1;
    *cache = per_sm;
  }
  const long long tiles = std::max<long long>(1, count / tile);
  *grid = static_cast<int>(std::min<long long>(tiles, static_cast<long long>(per_sm) * sms));
  return TSB_OK;
}

}  // namespace

// ============================================================================ N-Queens
struct PoolExtent {
  long long b, e;  // arena positions [b, e)
};

// state of the fused expand kernels of one handle (expand_common.cuh)
struct ExpandCtx {
  uint32_t* d_cmask = nullptr;  // side array of the round, `side_bytes` per tile: PFSP: one child mask per parent;
                                // N-Queens: the tile's items (one uint16 per child)
  int* d_tile = nullptr;        // per-tile child counts
  long long tile_cap = 0;       // tiles the two arrays above hold
  long long side_bytes = 0;
  tsb::ExpandState* d_st = nullptr;
  tsb::ExpandResult* h_res = nullptr;  // pinned + mapped: written by the scan kernel of a round
  tsb::ExpandResult* d_res = nullptr;  // device alias of h_res
  unsigned epoch = 0;
  int occ_count = 0, occ_build = 0, occ_count2 = 0, occ_build2 = 0;
  bool attr_set = false, attr_set2 = false;
  // (clears are ordered on the stream the kernels run on: the handle's streams do not synchronise with the
  // legacy default stream)
  int reserve(long long tiles, long long side_bytes_per_tile, cudaStream_t s, int best_init = 0x7FFFFFFF) {
    if (!d_st) {
      TSB_CUDA(cudaMalloc(&d_st, sizeof(tsb::ExpandState)));
      const tsb::ExpandState init{0ull, best_init, 0};
      TSB_CUDA(cudaMemcpyAsync(d_st, &init, sizeof(init), cudaMemcpyHostToDevice, s));
      TSB_CUDA(cudaStreamSynchronize(s));  // `init` lives on this stack frame
    }
    if (!h_res) {
      TSB_CUDA(cudaHostAlloc(&h_res, sizeof(tsb::ExpandResult), cudaHostAllocPortable | cudaHostAllocMapped));
      // (epochs start at 1: recycled pinned memory may hold another handle's old record, epoch included — the early
      // wait below would take it for this handle's first round)
      std::memset(h_res, 0, sizeof(tsb::ExpandResult));
      TSB_CUDA(cudaHostGetDevicePointer(reinterpret_cast<void**>(&d_res), h_res, 0));
    }
    if (tiles > tile_cap || side_bytes_per_tile > side_bytes) {
      side_bytes_per_tile = std::max(side_bytes_per_tile, side_bytes);
      if (d_cmask) cudaFree(d_cmask);
      if (d_tile) cudaFree(d_tile);
      d_cmask = nullptr;
      d_tile = nullptr;
      tile_cap = 0;
      const long long cap = std::max<long long>(tiles + tiles / 4 + 16, 1024);
      TSB_CUDA(cudaMalloc(&d_cmask, static_cast<size_t>(cap) * side_bytes_per_tile + 64));
      TSB_CUDA(cudaMalloc(&d_tile, static_cast<size_t>(cap) * sizeof(int)));
      tile_cap = cap;
      side_bytes = side_bytes_per_tile;
    }
    return TSB_OK;
  }
  // Wait for the round's result record.  `early`: return as soon as the build kernel's first CTA has published
  // the counts (it does so in its prologue) — the children are still being written, which is fine for a caller
  // whose next use of them is ordered on the same stream (the pool); the host then prepares and launches the next
  // round while this one finishes, which hides the launch + synchronisation latency of small rounds.
  int wait_result(unsigned want_epoch, cudaStream_t s, bool early) {
    if (early) {
      const volatile unsigned long long* ep = &h_res->epoch;
      for (unsigned spin = 0;; spin++) {
        if (*ep == want_epoch) return TSB_OK;
        if ((spin & 1023u) == 1023u) {  // a faulted kernel never publishes: ask the stream now and then
          const cudaError_t q = cudaStreamQuery(s);
          if (q == cudaSuccess) return *ep == want_epoch ? TSB_OK : TSB_ECUDA;
          if (q != cudaErrorNotReady) {
            g_last_cuda_error = std::string("expand kernels: ") + cudaGetErrorString(q);
            (void)cudaGetLastError();
            return TSB_ECUDA;
          }
        }
      }
    }
    TSB_CUDA(cudaStreamSynchronize(s));
    return h_res->epoch == want_epoch ? TSB_OK : TSB_ECUDA;
  }
  void release() {
    if (d_cmask) cudaFree(d_cmask);
    if (d_tile) cudaFree(d_tile);
    if (d_st) cudaFree(d_st);
    if (h_res) cudaFreeHost(h_res);
    d_cmask = nullptr;
    d_tile = nullptr;
    d_st = nullptr;
    h_res = d_res = nullptr;
  }
};

// Device-resident pool: a stack of extents inside one arena of `rec`-byte nodes.  A round reads the newest
// nodes in place (possibly spanning several extents) and appends the children above the top, so nothing is
// copied; the holes left behind are reclaimed by compacting into the second arena when the top reaches the end.
struct DevicePool {
  uint8_t* arena[2] = {nullptr, nullptr};
  // optional side array: `side_rec` bytes per arena position, moved with the nodes (N-Queens: nq_expand2.cuh)
  uint8_t* side[2] = {nullptr, nullptr};
  size_t side_rec = 0, side_slack = 0;
  long long cap = 0;  // nodes per arena
  int cur = 0;
  size_t rec = 0, slack = 0;
  std::vector<PoolExtent> ext;
  long long size = 0;
  uint64_t compactions = 0;
  long long top() const { return ext.empty() ? 0 : ext.back().e; }
  size_t bytes(long long nodes) const { return static_cast<size_t>(nodes) * rec + slack + 64; }
  size_t side_bytes(long long nodes) const { return static_cast<size_t>(nodes) * side_rec + side_slack + 64; }
  int ensure_arena(int which, long long nodes) {
    (void)nodes;
    if (!arena[which]) TSB_CUDA(cudaMalloc(&arena[which], bytes(cap)));
    if (side_rec && !side[which]) TSB_CUDA(cudaMalloc(&side[which], side_bytes(cap)));
    return TSB_OK;
  }
  // all extents -> [0, size) of the other arena (or of fresh, larger arenas when `new_cap` > cap)
  int compact(cudaStream_t s, long long new_cap) {
    uint8_t *dst = nullptr, *sdst = nullptr;
    const bool grow = new_cap > cap;
    if (grow) {
      TSB_CUDA(cudaMalloc(&dst, static_cast<size_t>(new_cap) * rec + slack + 64));
      if (side_rec) TSB_CUDA(cudaMalloc(&sdst, side_bytes(new_cap)));
    } else {
      int rc = ensure_arena(cur ^ 1, cap);
      if (rc != TSB_OK) return rc;
      dst = arena[cur ^ 1];
      sdst = side[cur ^ 1];
    }
    long long at = 0;
    for (const PoolExtent& x : ext) {
      TSB_CUDA(cudaMemcpyAsync(dst + at * rec, arena[cur] + x.b * rec, static_cast<size_t>(x.e - x.b) * rec,
                               cudaMemcpyDeviceToDevice, s));
      if (side_rec && side[cur])
        TSB_CUDA(cudaMemcpyAsync(sdst + at * side_rec, side[cur] + x.b * side_rec,
                                 static_cast<size_t>(x.e - x.b) * side_rec, cudaMemcpyDeviceToDevice, s));
      at += x.e - x.b;
    }
    TSB_CUDA(cudaStreamSynchronize(s));
    if (grow) {
      for (int i = 0; i < 2; i++) {
        if (arena[i]) cudaFree(arena[i]);
        if (side[i]) cudaFree(side[i]);
        arena[i] = side[i] = nullptr;
      }
      arena[0] = dst;
      side[0] = sdst;
      cur = 0;
      cap = new_cap;
    } else {
      cur ^= 1;
    }
    ext.clear();
    if (at) ext.push_back({0, at});
    ++compactions;
    return TSB_OK;
  }
  // room for `extra` nodes above the top
  int reserve(cudaStream_t s, long long extra, long long min_cap) {
    if (cap == 0) {
      cap = std::max<long long>(min_cap, extra + 1024);
      int rc = ensure_arena(cur, cap);
      if (rc != TSB_OK) return rc;
    }
    if (top() + extra <= cap) return TSB_OK;
    const long long need = size + extra;
    return compact(s, need > cap ? std::max<long long>(2 * cap, need + need / 2) : cap);
  }
  void release() {
    for (int i = 0; i < 2; i++) {
      if (arena[i]) cudaFree(arena[i]);
      if (side[i]) cudaFree(side[i]);
      arena[i] = side[i] = nullptr;
    }
    ext.clear();
    size = 0;
    cap = 0;
  }
};

// state of the persistent multi-round kernel of one handle (nq_rounds.cuh)
struct RoundsCtx {
  tsb::RoundsSync* d_sync = nullptr;
  tsb::RoundsState* h_state = nullptr;  // pinned + mapped: written by the kernel when it leaves
  tsb::RoundsState* d_state = nullptr;  // device alias of h_state
  unsigned epoch = 0;
  bool attr_set = false;
  int threads = 256;  // CTA size (env TSB200_ROUNDS_THREADS = 256 | 512)
  int ctas = 0;       // CTAs per pool (env TSB200_ROUNDS_CTAS; 0 = nq_ll_grid's measured defaults: an all-to-all flag
                      // exchange among 148 CTAs costs 2-3x one among 74 (tools/flag_exchange.py), the per-CTA work
                      // grows the other way)
  int occ = 2;        // env TSB200_ROUNDS_OCC=3: three CTAs per SM (several pools per launch)
  int ppt = 0;        // env TSB200_ROUNDS_PPT=3: the 768-parent slices also where 512 would do (experiments)
  int version = 3;    // 3 = the fence-free kernel on the fat arena (nq_rounds_ll.cuh); 2 = nq_rounds.cuh (env TSB200_ROUNDS_V)
  tsb::FatNode* d_fat = nullptr;  // the pool in the self-validating 64-byte format, while the LL kernel owns it
  long long fat_cap = 0;
  bool in_fat = false;            // the pool currently lives in d_fat (the plain arena is stale)
  bool attr_llv[4] = {false, false, false, false};
  tsb::LlSync* d_ll = nullptr;
  int ensure_fat(long long cap, cudaStream_t s) {
    if (!d_ll) {
      TSB_CUDA(cudaMalloc(&d_ll, sizeof(tsb::LlSync)));
      TSB_CUDA(cudaMemsetAsync(d_ll, 0, sizeof(tsb::LlSync), s));
    }
    if (cap <= fat_cap) return TSB_OK;
    if (d_fat) cudaFree(d_fat);
    d_fat = nullptr;
    fat_cap = 0;
    TSB_CUDA(cudaMalloc(&d_fat, static_cast<size_t>(cap) * sizeof(tsb::FatNode)));
    fat_cap = cap;
    return TSB_OK;
  }
  unsigned long long* d_aux = nullptr;  // side word per arena position (nq_rounds.cuh)
  long long aux_cap = 0, aux_valid = 0;
  int ensure_aux(long long cap) {
    if (cap <= aux_cap) return TSB_OK;
    if (d_aux) cudaFree(d_aux);
    d_aux = nullptr;
    aux_cap = aux_valid = 0;
    TSB_CUDA(cudaMalloc(&d_aux, static_cast<size_t>(cap) * sizeof(unsigned long long) + 256));
    aux_cap = cap;
    return TSB_OK;
  }
  RoundsCtx() {
    if (const char* v = std::getenv("TSB200_ROUNDS_THREADS")) {
      const int x = std::atoi(v);
      if (x == 256 || x == 512) threads = x;
    }
    if (const char* v = std::getenv("TSB200_ROUNDS_CTAS")) ctas = std::max(1, std::atoi(v));
    if (const char* v = std::getenv("TSB200_ROUNDS_PPT")) ppt = std::atoi(v) == 3 ? 3 : 0;
    if (const char* v = std::getenv("TSB200_ROUNDS_OCC")) occ = std::atoi(v) == 3 ? 3 : 2;
    if (const char* v = std::getenv("TSB200_ROUNDS_V")) version = std::atoi(v) == 2 ? 2 : 3;
  }
  int ensure(cudaStream_t s) {
    if (!d_sync) {
      TSB_CUDA(cudaMalloc(&d_sync, sizeof(tsb::RoundsSync)));
      TSB_CUDA(cudaMemsetAsync(d_sync, 0, sizeof(tsb::RoundsSync), s));
    }
    if (!h_state) {
      TSB_CUDA(cudaHostAlloc(&h_state, sizeof(tsb::RoundsState), cudaHostAllocPortable | cudaHostAllocMapped));
      std::memset(h_state, 0, sizeof(tsb::RoundsState));
      TSB_CUDA(cudaHostGetDevicePointer(reinterpret_cast<void**>(&d_state), h_state, 0));
    }
    return TSB_OK;
  }
  void release() {
    if (d_sync) cudaFree(d_sync);
    if (h_state) cudaFreeHost(h_state);
    if (d_aux) cudaFree(d_aux);
    if (d_fat) cudaFree(d_fat);
    if (d_ll) cudaFree(d_ll);
    d_sync = nullptr;
    h_state = d_state = nullptr;
    d_aux = nullptr;
    d_fat = nullptr;
    d_ll = nullptr;
    aux_cap = aux_valid = fat_cap = 0;
    in_fat = false;
  }
};

struct tsb_nq : Base {
  tsb_nq* sibling[3] = {nullptr, nullptr, nullptr};  // further pools on the same device, owned by this handle (tsb_nq_sibling)
  bool aux_ok = false;  // every node of the pool has its side word (nq_expand2.cuh)
  int N = 0, g = 1;
  RoundsCtx rounds;
  int variant = 0;  // env TSB200_NQ_VARIANT (kernel A/B experiments)
  int tile_threads = 0;  // env TSB200_NQ_TILE_THREADS = 128: always the TMA-pipelined kernel (A/B experiments)
  int occ[3] = {0, 0, 0};  // cached CTAs per SM, per tile size (128 / 64 / 32 threads)
  bool attr_set[3] = {false, false, false};
  // fused expand (evaluate + generate_children on the device) and the device-resident pool
  ExpandCtx ex;
  uint8_t* d_children = nullptr;  // host-buffer expand: device image of the children
  size_t d_children_bytes = 0;
  DevicePool pool;
};

namespace {

int nq_materialize(tsb_nq* h);  // (defined with the LL kernel's launch helpers below)

template <int N, int VAR, int T>
int launch_nq_nt(tsb_nq* h, int slot, const uint8_t* in, uint8_t* out, long long count, cudaStream_t s) {
  auto kernel = tsb::nq_evaluate_kernel<N, VAR, T>;
  const size_t smem = sizeof(tsb::NqSmem<N, T>) + 128;
  if (!h->attr_set[slot]) {
    TSB_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    h->attr_set[slot] = true;
  }
  int grid = 1;
  int rc = grid_for(kernel, T, smem, count, T * tsb::NQ_QUAD, h->di.sms, &grid, &h->occ[slot]);
  if (rc != TSB_OK) return rc;
  kernel<<<grid, T, smem, s>>>(in, out, count);
  TSB_CUDA(cudaGetLastError());
  h->launches++;
  return TSB_OK;
}
// small chunks (fewer than two 512-parent tiles per SM — the reference's default --M 50000 is 97 tiles) take the
// one-parent-per-thread kernel, everything else the TMA-pipelined one
template <int N, int VAR>
int launch_nq_n(tsb_nq* h, const uint8_t* in, uint8_t* out, long long count, cudaStream_t s) {
  if constexpr (VAR == 0) {
    if (count < 2LL * h->di.sms * tsb::NQ_TILE && h->tile_threads != 128) {
      const int grid = static_cast<int>((count + tsb::NQ_SMALL - 1) / tsb::NQ_SMALL);
      tsb::nq_evaluate_small_kernel<N><<<grid, tsb::NQ_SMALL, 0, s>>>(in, out, static_cast<int>(count));
      TSB_CUDA(cudaGetLastError());
      h->launches++;
      return TSB_OK;
    }
  }
  return launch_nq_nt<N, VAR, 128>(h, 0, in, out, count, s);
}

int launch_nq(tsb_nq* h, const uint8_t* in, uint8_t* out, long long count, cudaStream_t s) {
  if (h->N == 17 && h->variant == 1) return launch_nq_n<17, 1>(h, in, out, count, s);  // A/B experiment: byte alignment as IMAD.HI
  if (h->N == 17 && h->variant == 2) return launch_nq_n<17, 2>(h, in, out, count, s);  // A/B experiment: bytes by LDS.U8
  switch (h->N) {
#define TSB_NQ_CASE(n) \
  case n:              \
    return launch_nq_n<n, 0>(h, in, out, count, s);
    TSB_NQ_CASE(1) TSB_NQ_CASE(2) TSB_NQ_CASE(3) TSB_NQ_CASE(4) TSB_NQ_CASE(5) TSB_NQ_CASE(6) TSB_NQ_CASE(7)
    TSB_NQ_CASE(8) TSB_NQ_CASE(9) TSB_NQ_CASE(10) TSB_NQ_CASE(11) TSB_NQ_CASE(12) TSB_NQ_CASE(13)
    TSB_NQ_CASE(14) TSB_NQ_CASE(15) TSB_NQ_CASE(16) TSB_NQ_CASE(17) TSB_NQ_CASE(18) TSB_NQ_CASE(19)
    TSB_NQ_CASE(20)
#undef TSB_NQ_CASE
  }
  return TSB_EINVAL;
}

}  // namespace

namespace {

// tile table of a round: pieces in logical order -> ExpandParams
int make_params(const std::vector<PoolExtent>& pieces, int tile_records, tsb::ExpandParams* prm) {
  if (pieces.empty() || pieces.size() > tsb::EXP_MAX_PIECES) return TSB_EINVAL;
  std::memset(prm, 0, sizeof(*prm));
  long long cum = 0;
  for (size_t i = 0; i < pieces.size(); i++) {
    const PoolExtent& x = pieces[i];
    const long long t0 = x.b / tile_records, t1 = (x.e + tile_records - 1) / tile_records;
    prm->piece[i].lo = x.b;
    prm->piece[i].hi = x.e;
    prm->piece[i].first_tile = t0;
    prm->piece[i].tile_cum = static_cast<int>(cum);
    cum += t1 - t0;
  }
  if (cum > INT_MAX / 2) return TSB_EINVAL;
  prm->n_pieces = static_cast<int>(pieces.size());
  prm->n_tiles = static_cast<int>(cum);
  return TSB_OK;
}

// one evaluate + generate_children round over `pieces` of `arena` (count, build); children packed at
// `children_d`.  Synchronous: the counts come back through the host-mapped result record.
// AUX: `aux` / `children_aux` are the side arrays of `arena` / `children_d` (nq_expand2.cuh)
template <int N, bool AUX>
int nq_expand_n(tsb_nq* h, const uint8_t* arena, const unsigned long long* aux, const std::vector<PoolExtent>& pieces,
                uint8_t* children_d, unsigned long long* children_aux, cudaStream_t s, unsigned long long* n_children,
                unsigned long long* n_solutions, bool early) {
  tsb::ExpandParams prm;
  int rc = make_params(pieces, tsb::NQ_TILE, &prm);
  if (rc != TSB_OK) return rc;
  ExpandCtx& ex = h->ex;
  const bool trace = !ex.attr_set && std::getenv("TSB200_TRACE");
  const auto tnow = [] { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
  const double tr0 = trace ? tnow() : 0;
  // (sized for the largest round up front: the items array is 1 KB * N per tile)
  rc = ex.reserve(std::max<long long>(prm.n_tiles, h->M_max / tsb::NQ_TILE + 2 * tsb::EXP_MAX_PIECES),
                  static_cast<long long>(tsb::NQ_TILE) * N * 2, s);
  if (rc != TSB_OK) return rc;
  auto k1 = tsb::nq_expand_count_kernel<N, AUX>;
  auto k3 = tsb::nq_expand_build_kernel<N, AUX>;
  const size_t smem1 = sizeof(tsb::NqCountSmem<AUX>) + 128, smem3 = sizeof(tsb::NqBuildSmem<AUX>) + 128;
  bool& attr_set = AUX ? ex.attr_set2 : ex.attr_set;
  if (!attr_set) {
    TSB_CUDA(cudaFuncSetAttribute(k1, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem1)));
    TSB_CUDA(cudaFuncSetAttribute(k3, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem3)));
    attr_set = true;
  }
  const long long recs = static_cast<long long>(prm.n_tiles) * tsb::NQ_TILE;
  int g1 = 1, g3 = 1;
  rc = grid_for(k1, tsb::NQ_THREADS, smem1, recs, tsb::NQ_TILE, h->di.sms, &g1, AUX ? &ex.occ_count2 : &ex.occ_count);
  if (rc != TSB_OK) return rc;
  rc = grid_for(k3, tsb::NQ_THREADS, smem3, recs, tsb::NQ_TILE, h->di.sms, &g3, AUX ? &ex.occ_build2 : &ex.occ_build);
  if (rc != TSB_OK) return rc;
  prm.epoch = ++ex.epoch;
  if ((prm.n_tiles + g3 - 1) / g3 > tsb::EXP_MAX_OWN) return TSB_EINVAL;  // (M_max * N < 2^31 keeps this far away)
  uint16_t* d_items = reinterpret_cast<uint16_t*>(ex.d_cmask);
  const double tr1 = trace ? tnow() : 0;
  k1<<<g1, tsb::NQ_THREADS, smem1, s>>>(arena, aux, prm, d_items, ex.d_tile, ex.d_st);
  k3<<<g3, tsb::NQ_THREADS, smem3, s>>>(arena, aux, prm, d_items, ex.d_tile, children_d, children_aux, ex.d_st, ex.d_res);
  TSB_CUDA(cudaGetLastError());
  h->launches += 2;
  const double tr2 = trace ? tnow() : 0;
  rc = ex.wait_result(prm.epoch, s, early);
  if (trace)
    std::fprintf(stderr, "[tsb200] first expand round: reserve+attributes %.2f ms, 2 launches %.2f ms, wait %.2f ms\n",
                 tr1 - tr0, tr2 - tr1, tnow() - tr2);
  if (rc != TSB_OK) {
    if (g_last_cuda_error.empty()) g_last_cuda_error = "expand kernels did not publish their result";
    return rc;
  }
  *n_children = ex.h_res->children;
  *n_solutions = ex.h_res->solutions;
  return TSB_OK;
}

int nq_expand_dispatch(tsb_nq* h, const uint8_t* arena, const std::vector<PoolExtent>& pieces, uint8_t* children_d,
                       cudaStream_t s, unsigned long long* nc, unsigned long long* ns, bool early = false,
                       const unsigned long long* aux = nullptr, unsigned long long* children_aux = nullptr) {
  switch (h->N) {
#define TSB_NQ_CASE(n)                                                                                   \
  case n:                                                                                                \
    return aux ? nq_expand_n<n, true>(h, arena, aux, pieces, children_d, children_aux, s, nc, ns, early) \
               : nq_expand_n<n, false>(h, arena, nullptr, pieces, children_d, nullptr, s, nc, ns, early);
    TSB_NQ_CASE(1) TSB_NQ_CASE(2) TSB_NQ_CASE(3) TSB_NQ_CASE(4) TSB_NQ_CASE(5) TSB_NQ_CASE(6) TSB_NQ_CASE(7)
    TSB_NQ_CASE(8) TSB_NQ_CASE(9) TSB_NQ_CASE(10) TSB_NQ_CASE(11) TSB_NQ_CASE(12) TSB_NQ_CASE(13)
    TSB_NQ_CASE(14) TSB_NQ_CASE(15) TSB_NQ_CASE(16) TSB_NQ_CASE(17) TSB_NQ_CASE(18) TSB_NQ_CASE(19)
    TSB_NQ_CASE(20)
#undef TSB_NQ_CASE
  }
  return TSB_EINVAL;
}

// the newest n nodes of a pool, as pieces in logical order
void pool_top_pieces(const DevicePool& p, long long n, std::vector<PoolExtent>* pieces) {
  pieces->clear();
  long long left = n;
  for (size_t i = p.ext.size(); i-- > 0 && left > 0;) {
    const long long t = std::min(left, p.ext[i].e - p.ext[i].b);
    pieces->insert(pieces->begin(), PoolExtent{p.ext[i].e - t, p.ext[i].e});
    left -= t;
  }
}
// drop the newest n nodes
void pool_pop(DevicePool& p, long long n) {
  long long left = n;
  while (left > 0 && !p.ext.empty()) {
    PoolExtent& x = p.ext.back();
    const long long t = std::min(left, x.e - x.b);
    x.e -= t;
    left -= t;
    if (x.e == x.b) p.ext.pop_back();
  }
  p.size -= n;
}

}  // namespace

namespace {
// Work stealing between device pools (SURVEY §8f row 3; the reference steals between its per-GPU host pools,
// nqueens_multigpu_chpl.chpl:255-312): the OLDEST half of the victim's pool (popFrontBulkFree,
// lib/commons/Pool_par.chpl:178-191: size / 2 nodes from the front, only if size >= 2 m) moves to the top of the
// thief's pool, device to device (cudaMemcpyPeerAsync: NVLink between two GPUs, a plain copy on one), order
// preserved.  Both pools must be quiescent (no round in flight); the caller serialises access to both handles.
int pool_steal_front(DevicePool& v, int vdev, cudaStream_t vs, DevicePool& t, int tdev, cudaStream_t ts, int m,
                     long long min_cap, long long* n_stolen) {
  *n_stolen = 0;
  if (v.size < 2LL * m) return TSB_OK;
  const long long want = v.size / 2;
  const bool trace = std::getenv("TSB200_TRACE") != nullptr;
  const auto tnow = [] { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
  const double tr0 = trace ? tnow() : 0;
  TSB_CUDA(cudaSetDevice(tdev));
  int rc = t.reserve(ts, want, min_cap);
  if (rc != TSB_OK) return rc;
  long long at = t.top();
  if (t.rec == sizeof(tsb_pfsp_node)) at = (at + 1) & ~1LL;  // PFSP extents start on a 16-byte boundary
  if (at + want > t.cap) {
    rc = t.compact(ts, std::max<long long>(2 * t.cap, t.size + want + 1024));
    if (rc != TSB_OK) return rc;
    at = t.top();
    if (t.rec == sizeof(tsb_pfsp_node)) at = (at + 1) & ~1LL;
  }
  TSB_CUDA(cudaSetDevice(vdev));
  long long left = want, dst = at;
  while (left > 0 && !v.ext.empty()) {
    PoolExtent& x = v.ext.front();
    const long long n = std::min(left, x.e - x.b);
    TSB_CUDA(cudaMemcpyPeerAsync(t.arena[t.cur] + dst * t.rec, tdev, v.arena[v.cur] + x.b * v.rec, vdev,
                                 static_cast<size_t>(n) * v.rec, vs));
    x.b += n;
    dst += n;
    left -= n;
    if (x.b == x.e) v.ext.erase(v.ext.begin());
  }
  TSB_CUDA(cudaStreamSynchronize(vs));
  const long long got = want - left;
  v.size -= got;
  if (got) {
    t.ext.push_back({at, at + got});
    t.size += got;
  }
  *n_stolen = got;
  if (trace)
    std::fprintf(stderr, "[tsb200] steal: %lld nodes (%.1f MB) device %d -> %d in %.2f ms (victim keeps %lld, thief has %lld)\n",
                 got, got * v.rec / 1e6, vdev, tdev, tnow() - tr0, v.size, t.size);
  return TSB_OK;
}
void enable_peer(int a, int b) {
  if (a == b) return;
  int can = 0;
  if (cudaDeviceCanAccessPeer(&can, a, b) == cudaSuccess && can) {
    cudaSetDevice(a);
    if (cudaDeviceEnablePeerAccess(b, 0) != cudaSuccess) (void)cudaGetLastError();  // (already enabled is fine)
  }
  (void)cudaGetLastError();
}
}  // namespace

// ============================================================================ PFSP
struct tsb_pfsp : Base {
  int jobs = 0, machines = 0, pairs = 0, mt = 0;  // mt = template machine count (5, 10 or 20)
  tsb::PfspLb1Tables* d_tab1 = nullptr;
  tsb::Lb2Const* lb2c = nullptr;  // packed Johnson tables, passed to the lb2 kernels by value (constant bank)
  tsb::Lb2ConstU* lb2u = nullptr; // <= 10 machines: address of the shared-memory-resident table (tsb::Lb2TabU)
  tsb::Lb2TabU* d_tabu = nullptr;
  bool attr_set[3] = {false, false, false};
  int occ[3] = {0, 0, 0};
  bool simd16 = false;  // lb1 / lb1_d children two per register (values < 2^16, min_tails non-increasing)
  bool wide = false;    // MAX_JOBS = 50 build: 208-byte nodes, the general kernels of pfsp_wide.cuh
  tsb::PfspWideTables* d_wtab = nullptr;
  bool wide_attr[3] = {false, false, false};
  int wide_occ[3] = {0, 0, 0};
  // fused expand + device-resident pool
  ExpandCtx ex;
  bool ex_attr[4] = {false, false, false, false};  // count lb1_d, lb1, lb2; build
  int ex_occ[4] = {0, 0, 0, 0};
  bool wex_attr[4] = {false, false, false, false};  // the same for the 208-byte kernels (pfsp_wide_expand.cuh)
  int wex_occ[4] = {0, 0, 0, 0};
  uint8_t* d_children = nullptr;
  size_t d_children_bytes = 0;
  DevicePool pool;
  uint64_t slow_rounds = 0;
  std::vector<tsb_pfsp_node> h_chunk, h_kids;  // slow path scratch
  std::vector<tsb_pfsp_node50> h_chunk50, h_kids50;
  size_t rec() const { return wide ? sizeof(tsb_pfsp_node50) : sizeof(tsb_pfsp_node); }  // bytes per node
  int tile() const { return wide ? tsb::PW_TILE : tsb::PF_TILE; }                        // parents per expand tile
  std::vector<int32_t> h_bounds;
};

namespace {

template <int KIND, int M, bool SIMD>
int launch_lb1_km(tsb_pfsp* h, const uint8_t* in, uint8_t* out, long long count, cudaStream_t s) {
  auto kernel = tsb::pfsp_lb1_kernel<KIND, M, SIMD>;
  const size_t smem = sizeof(tsb::Lb1Smem) + 128;
  if (!h->attr_set[KIND]) {
    TSB_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    h->attr_set[KIND] = true;
  }
  int grid = 1;
  int rc = grid_for(kernel, tsb::PF_THREADS, smem, count, tsb::PF_TILE, h->di.sms, &grid, &h->occ[KIND]);
  if (rc != TSB_OK) return rc;
  kernel<<<grid, tsb::PF_THREADS, smem, s>>>(in, out, count, h->d_tab1);
  TSB_CUDA(cudaGetLastError());
  h->launches++;
  return TSB_OK;
}

template <int M, typename CT>
int launch_lb2_mc(tsb_pfsp* h, const CT& C, const uint8_t* in, uint8_t* out, long long count, int best, cudaStream_t s) {
  auto kernel = tsb::pfsp_lb2_kernel<M, CT>;
  const size_t smem = sizeof(tsb::Lb2Smem<M>) + 128;
  if (!h->attr_set[2]) {
    TSB_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    h->attr_set[2] = true;
  }
  int grid = 1;
  int rc = grid_for(kernel, tsb::PF_THREADS, smem, count, tsb::LB2_TILE, h->di.sms, &grid, &h->occ[2]);
  if (rc != TSB_OK) return rc;
  kernel<<<grid, tsb::PF_THREADS, smem, s>>>(in, out, count, h->d_tab1, C, best);
  TSB_CUDA(cudaGetLastError());
  h->launches++;
  return TSB_OK;
}
template <int M>
int launch_lb2_m(tsb_pfsp* h, const uint8_t* in, uint8_t* out, long long count, int best, cudaStream_t s) {
  if constexpr (M <= 10) {
    if (h->lb2u) return launch_lb2_mc<M>(h, *h->lb2u, in, out, count, best, s);
  }
  return launch_lb2_mc<M>(h, *h->lb2c, in, out, count, best, s);
}

template <int KIND, int M>
int launch_wide_km(tsb_pfsp* h, const uint8_t* in, uint8_t* out, long long count, int best, cudaStream_t s) {
  auto kernel = tsb::pfsp_wide_kernel<KIND, M>;
  const size_t smem = sizeof(tsb::PfspWideSmem) + 128;
  if (!h->wide_attr[KIND]) {
    TSB_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    h->wide_attr[KIND] = true;
  }
  int grid = 1;
  int rc = grid_for(kernel, tsb::PW_THREADS, smem, count + tsb::PW_TILE - 1, tsb::PW_TILE, h->di.sms, &grid, &h->wide_occ[KIND]);
  if (rc != TSB_OK) return rc;
  kernel<<<grid, tsb::PW_THREADS, smem, s>>>(in, reinterpret_cast<int32_t*>(out), count, h->d_wtab, best);
  TSB_CUDA(cudaGetLastError());
  h->launches++;
  return TSB_OK;
}
template <int M>
int launch_wide_m(tsb_pfsp* h, int lb_kind, const uint8_t* in, uint8_t* out, long long count, int best, cudaStream_t s) {
  if (lb_kind == TSB_LB1_D) return launch_wide_km<0, M>(h, in, out, count, best, s);
  if (lb_kind == TSB_LB1) return launch_wide_km<1, M>(h, in, out, count, best, s);
  return launch_wide_km<2, M>(h, in, out, count, best, s);
}

int launch_pfsp(tsb_pfsp* h, int lb_kind, const uint8_t* in, uint8_t* out, long long count, int64_t best64,
                cudaStream_t s) {
  // bounds are int32 and `lb > best` can never hold for best >= INT32_MAX (Chapel's max(int) under --ub 0)
  const int best = best64 > INT_MAX ? INT_MAX : best64 < INT_MIN ? INT_MIN : static_cast<int>(best64);
  if (h->wide) {
    if (h->mt == 5) return launch_wide_m<5>(h, lb_kind, in, out, count, best, s);
    if (h->mt == 10) return launch_wide_m<10>(h, lb_kind, in, out, count, best, s);
    return launch_wide_m<20>(h, lb_kind, in, out, count, best, s);
  }
#define TSB_PF_DISPATCH(M)                                                                                      \
  if (lb_kind == TSB_LB1)                                                                                        \
    return h->simd16 ? launch_lb1_km<1, M, true>(h, in, out, count, s) : launch_lb1_km<1, M, false>(h, in, out, count, s); \
  if (lb_kind == TSB_LB1_D)                                                                                      \
    return h->simd16 ? launch_lb1_km<0, M, true>(h, in, out, count, s) : launch_lb1_km<0, M, false>(h, in, out, count, s); \
  return launch_lb2_m<M>(h, in, out, count, best, s);
  if (h->mt == 5) { TSB_PF_DISPATCH(5) }
  if (h->mt == 10) { TSB_PF_DISPATCH(10) }
  TSB_PF_DISPATCH(20)
#undef TSB_PF_DISPATCH
}

}  // namespace

namespace {

inline int clamp_best(int64_t best64) {
  return best64 > INT_MAX ? INT_MAX : best64 < INT_MIN ? INT_MIN : static_cast<int>(best64);
}

template <int M>
int pfsp_expand_m(tsb_pfsp* h, int lb_kind, const uint8_t* arena, const tsb::ExpandParams& prm, uint8_t* children_d,
                  cudaStream_t s) {
  ExpandCtx& ex = h->ex;
  const long long recs = static_cast<long long>(prm.n_tiles) * tsb::PF_TILE;
  auto k3 = tsb::pfsp_expand_build_kernel;
  const size_t smem3 = sizeof(tsb::PfBuildSmem) + 128;
  if (!h->ex_attr[3]) {
    TSB_CUDA(cudaFuncSetAttribute(k3, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem3)));
    h->ex_attr[3] = true;
  }
  int g1 = 1, g3 = 1;
  int rc = grid_for(k3, tsb::PF_THREADS, smem3, recs, tsb::PF_TILE, h->di.sms, &g3, &h->ex_occ[3]);
  if (rc != TSB_OK) return rc;
  if ((prm.n_tiles + g3 - 1) / g3 > tsb::EXP_MAX_OWN) return TSB_EINVAL;
  if (lb_kind == TSB_LB2) {
    const size_t smem1 = sizeof(tsb::Lb2CountSmem<M>) + 128;
    // (this kernel walks the round in half tiles and accumulates the tile counts)
    TSB_CUDA(cudaMemsetAsync(ex.d_tile, 0, static_cast<size_t>(prm.n_tiles) * sizeof(int), s));
    auto go = [&](auto k1, const auto& C) -> int {
      if (!h->ex_attr[2]) {
        TSB_CUDA(cudaFuncSetAttribute(k1, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem1)));
        h->ex_attr[2] = true;
      }
      int r2 = grid_for(k1, tsb::PF_THREADS, smem1, recs, tsb::LB2_TILE, h->di.sms, &g1, &h->ex_occ[2]);
      if (r2 != TSB_OK) return r2;
      k1<<<g1, tsb::PF_THREADS, smem1, s>>>(arena, prm, h->d_tab1, C, ex.d_cmask, ex.d_tile, ex.d_st);
      return TSB_OK;
    };
    bool done = false;
    if constexpr (M <= 10) {
      if (h->lb2u) {
        rc = go(tsb::pfsp_expand_count_lb2_kernel<M, tsb::Lb2ConstU>, *h->lb2u);
        done = true;
      }
    }
    if (!done) rc = go(tsb::pfsp_expand_count_lb2_kernel<M, tsb::Lb2Const>, *h->lb2c);
    if (rc != TSB_OK) return rc;
  } else if (lb_kind == TSB_LB1) {
    auto k1 = h->simd16 ? tsb::pfsp_expand_count_lb1_kernel<1, M, true> : tsb::pfsp_expand_count_lb1_kernel<1, M, false>;
    const size_t smem1 = sizeof(tsb::Lb1CountSmem) + 128;
    if (!h->ex_attr[1]) {
      TSB_CUDA(cudaFuncSetAttribute(k1, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem1)));
      h->ex_attr[1] = true;
    }
    rc = grid_for(k1, tsb::PF_THREADS, smem1, recs, tsb::PF_TILE, h->di.sms, &g1, &h->ex_occ[1]);
    if (rc != TSB_OK) return rc;
    k1<<<g1, tsb::PF_THREADS, smem1, s>>>(arena, prm, h->d_tab1, ex.d_cmask, ex.d_tile, ex.d_st);
  } else {
    auto k1 = h->simd16 ? tsb::pfsp_expand_count_lb1_kernel<0, M, true> : tsb::pfsp_expand_count_lb1_kernel<0, M, false>;
    const size_t smem1 = sizeof(tsb::Lb1CountSmem) + 128;
    if (!h->ex_attr[0]) {
      TSB_CUDA(cudaFuncSetAttribute(k1, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem1)));
      h->ex_attr[0] = true;
    }
    rc = grid_for(k1, tsb::PF_THREADS, smem1, recs, tsb::PF_TILE, h->di.sms, &g1, &h->ex_occ[0]);
    if (rc != TSB_OK) return rc;
    k1<<<g1, tsb::PF_THREADS, smem1, s>>>(arena, prm, h->d_tab1, ex.d_cmask, ex.d_tile, ex.d_st);
  }
  k3<<<g3, tsb::PF_THREADS, smem3, s>>>(arena, prm, ex.d_cmask, ex.d_tile, children_d, ex.d_st, ex.d_res);
  TSB_CUDA(cudaGetLastError());
  h->launches += 2;
  return TSB_OK;
}

// 208-byte nodes (pfsp_wide_expand.cuh): count + build, one template per (bound, machines)
template <int KIND, int M>
int pfsp_wide_expand_km(tsb_pfsp* h, const uint8_t* arena, const tsb::ExpandParams& prm, uint8_t* children_d,
                        cudaStream_t s) {
  ExpandCtx& ex = h->ex;
  const long long recs = static_cast<long long>(prm.n_tiles) * tsb::PW_TILE;
  auto k1 = tsb::pfsp_wide_expand_count_kernel<KIND, M>;
  auto k3 = tsb::pfsp_wide_expand_build_kernel;
  const size_t smem1 = sizeof(tsb::PwCountSmem) + 128, smem3 = sizeof(tsb::PwBuildSmem) + 128;
  if (!h->wex_attr[KIND]) {
    TSB_CUDA(cudaFuncSetAttribute(k1, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem1)));
    h->wex_attr[KIND] = true;
  }
  if (!h->wex_attr[3]) {
    TSB_CUDA(cudaFuncSetAttribute(k3, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem3)));
    h->wex_attr[3] = true;
  }
  int g1 = 1, g3 = 1;
  int rc = grid_for(k1, tsb::PW_THREADS, smem1, recs, tsb::PW_TILE, h->di.sms, &g1, &h->wex_occ[KIND]);
  if (rc == TSB_OK) rc = grid_for(k3, tsb::PW_THREADS, smem3, recs, tsb::PW_TILE, h->di.sms, &g3, &h->wex_occ[3]);
  if (rc != TSB_OK) return rc;
  if ((prm.n_tiles + g3 - 1) / g3 > tsb::EXP_MAX_OWN) return TSB_EINVAL;
  auto* cmask = reinterpret_cast<unsigned long long*>(ex.d_cmask);
  k1<<<g1, tsb::PW_THREADS, smem1, s>>>(arena, prm, h->d_wtab, cmask, ex.d_tile, ex.d_st);
  k3<<<g3, tsb::PW_THREADS, smem3, s>>>(arena, prm, cmask, ex.d_tile, children_d, ex.d_st, ex.d_res);
  TSB_CUDA(cudaGetLastError());
  h->launches += 2;
  return TSB_OK;
}
template <int M>
int pfsp_wide_expand_m(tsb_pfsp* h, int lb_kind, const uint8_t* arena, const tsb::ExpandParams& prm,
                       uint8_t* children_d, cudaStream_t s) {
  if (lb_kind == TSB_LB1_D) return pfsp_wide_expand_km<0, M>(h, arena, prm, children_d, s);
  if (lb_kind == TSB_LB1) return pfsp_wide_expand_km<1, M>(h, arena, prm, children_d, s);
  return pfsp_wide_expand_km<2, M>(h, arena, prm, children_d, s);
}

// generate_children of pfsp_gpu_chpl.chpl:273-303 on host arrays (the sequential rule, used by the slow path)
template <class Node>
void pfsp_generate_children_host(int jobs, const Node* parents, int size, const int32_t* bounds, int64_t* best,
                                 std::vector<Node>* kids, uint64_t* sol) {
  for (int i = 0; i < size; i++) {
    const Node& parent = parents[i];
    const int depth = parent.depth;
    for (int j = parent.limit1 + 1; j < jobs; j++) {
      const int32_t lb = bounds[j + static_cast<size_t>(i) * jobs];
      if (depth + 1 == jobs) {
        ++*sol;
        if (lb < *best) *best = lb;
      } else if (lb < *best) {
        Node c = parent;
        c.depth = depth + 1;
        c.limit1 = parent.limit1 + 1;
        std::swap(c.prmu[depth], c.prmu[j]);
        kids->push_back(c);
      }
    }
  }
}

// the host half of the slow path: the chunk (d_in) and its bounds (d_out) back, the sequential rule, the children
// to `children_d`
template <class Node>
int pfsp_slow_children(tsb_pfsp* h, std::vector<Node>& chunk, std::vector<Node>& kids, long long n,
                       uint8_t* children_d, cudaStream_t s, int64_t* best, unsigned long long* n_children,
                       unsigned long long* n_solutions) {
  chunk.resize(static_cast<size_t>(n));
  int rc = h->copy_d2h(chunk.data(), h->d_in, static_cast<size_t>(n) * sizeof(Node), s);
  if (rc == TSB_OK) rc = h->copy_d2h(h->h_bounds.data(), h->d_out, static_cast<size_t>(n) * h->jobs * 4, s);
  if (rc != TSB_OK) return rc;
  kids.clear();
  uint64_t sol = 0;
  pfsp_generate_children_host(h->jobs, chunk.data(), static_cast<int>(n), h->h_bounds.data(), best, &kids, &sol);
  rc = h->copy_h2d(children_d, kids.data(), kids.size() * sizeof(Node), s);
  if (rc != TSB_OK) return rc;
  *n_children = kids.size();
  *n_solutions = sol;
  return TSB_OK;
}

// One evaluate + generate_children round over `pieces` of `arena`; children packed at `children_d` (room for
// n * jobs nodes).  *best is read and updated with the reference's semantics.  Synchronous.
int pfsp_expand_round(tsb_pfsp* h, int lb_kind, const uint8_t* arena, const std::vector<PoolExtent>& pieces,
                      uint8_t* children_d, cudaStream_t s, int64_t* best, unsigned long long* n_children,
                      unsigned long long* n_solutions, bool early = false) {
  tsb::ExpandParams prm;
  const int tile = h->tile();
  int rc = make_params(pieces, tile, &prm);
  if (rc != TSB_OK) return rc;
  const int best_launch = clamp_best(*best);
  ExpandCtx& ex = h->ex;
  // side array: one child mask per parent, 32-bit for 20 jobs, 64-bit for 50
  rc = ex.reserve(std::max<long long>(prm.n_tiles, h->M_max / tile + 2 * tsb::EXP_MAX_PIECES),
                  static_cast<long long>(tile) * (h->wide ? 8 : 4), s);
  if (rc != TSB_OK) return rc;
  prm.epoch = ++ex.epoch;
  prm.best = best_launch;
  if (h->wide)
    rc = h->mt == 5 ? pfsp_wide_expand_m<5>(h, lb_kind, arena, prm, children_d, s)
         : h->mt == 10 ? pfsp_wide_expand_m<10>(h, lb_kind, arena, prm, children_d, s)
                       : pfsp_wide_expand_m<20>(h, lb_kind, arena, prm, children_d, s);
  else if (h->mt == 5)
    rc = pfsp_expand_m<5>(h, lb_kind, arena, prm, children_d, s);
  else if (h->mt == 10)
    rc = pfsp_expand_m<10>(h, lb_kind, arena, prm, children_d, s);
  else
    rc = pfsp_expand_m<20>(h, lb_kind, arena, prm, children_d, s);
  if (rc != TSB_OK) return rc;
  rc = ex.wait_result(prm.epoch, s, early);
  if (rc != TSB_OK) {
    if (g_last_cuda_error.empty()) g_last_cuda_error = "expand kernels did not publish their result";
    return rc;
  }
  if (ex.h_res->best >= best_launch) {  // no leaf of the chunk improved best: the launch-value masks are exact
    *n_children = ex.h_res->children;
    *n_solutions = ex.h_res->solutions;
    return TSB_OK;
  }
  // ---- slow path: a leaf lowered best inside this chunk, which changes what the rest of the chunk pushes
  // (sequential rule).  Redo the round: bounds through the evaluator, children on the host.
  ++h->slow_rounds;
  long long n = 0;
  for (const PoolExtent& x : pieces) n += x.e - x.b;
  if (n > h->M_max) return TSB_EINVAL;  // (cannot happen: every entry point checks count <= M_max first)
  const size_t rec = h->rec();
  long long at = 0;
  if (!(arena == h->d_in && pieces.size() == 1 && pieces[0].b == 0))
    for (const PoolExtent& x : pieces) {  // the chunk, contiguous
      TSB_CUDA(cudaMemcpyAsync(h->d_in + at * rec, arena + x.b * rec, static_cast<size_t>(x.e - x.b) * rec,
                               cudaMemcpyDeviceToDevice, s));
      at += x.e - x.b;
    }
  rc = launch_pfsp(h, lb_kind, h->d_in, h->d_out, n, *best, s);
  if (rc != TSB_OK) return rc;
  h->h_bounds.resize(static_cast<size_t>(n) * h->jobs);
  return h->wide ? pfsp_slow_children(h, h->h_chunk50, h->h_kids50, n, children_d, s, best, n_children, n_solutions)
                 : pfsp_slow_children(h, h->h_chunk, h->h_kids, n, children_d, s, best, n_children, n_solutions);
}

long long pfsp_pool_min_cap(const tsb_pfsp* h) {
  if (const long long c = env_pool_cap(); c > 0) return c;
  return std::max<long long>(1LL << 20, 4LL * h->M_max * h->jobs);
}
void pfsp_pool_setup(tsb_pfsp* h) {
  h->pool.rec = h->rec();
  h->pool.slack = static_cast<size_t>(h->tile()) * h->rec();
}

}  // namespace

__attribute__((visibility("hidden"))) int tsb_pfsp_handle_max_jobs(const tsb_pfsp* h) {
  return h && h->wide ? TSB_MAX_JOBS_WIDE : TSB_MAX_JOBS;
}

// ============================================================================ exported C ABI
extern "C" {

const char* tsb_version(void) { return "tsb200 0.1 (sm_100a)"; }

const char* tsb_strerror(int code) {
  switch (code) {
    case TSB_OK: return "ok";
    case TSB_EINVAL: return "invalid argument";
    case TSB_ECUDA: return "CUDA runtime error (see tsb_last_cuda_error)";
    case TSB_ENOMEM: return "out of memory";
    case TSB_ENODEV: return "no such CUDA device";
    case TSB_EALIGN: return "device pointer not 16-byte aligned";
    case TSB_EUNSUPPORTED: return "unsupported instance shape (jobs must be 20, machines 1..20)";
  }
  return "unknown error";
}
const char* tsb_last_cuda_error(void) { return g_last_cuda_error.c_str(); }

int tsb_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    (void)cudaGetLastError();
    return TSB_ENODEV;
  }
  return n;
}

// NUMA placement of a host thread that feeds one GPU (SCALE_r01: eight zero-copy streams through one socket's
// memory controllers and the inter-socket link cost half of the 8-GPU e2e throughput): pin the CALLING thread to
// the cores local to `device` (sysfs local_cpulist of its PCI function); pages the thread touches first afterwards
// — its chunk arrays, the library's pinned staging buffers — then live on that GPU's NUMA node.
int tsb_bind_thread_to_device(int device) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || device < 0 || device >= n) {
    (void)cudaGetLastError();
    return TSB_ENODEV;
  }
  char bus[64] = {0};
  TSB_CUDA(cudaDeviceGetPCIBusId(bus, sizeof(bus) - 1, device));
  for (char* c = bus; *c; ++c) *c = static_cast<char>(std::tolower(static_cast<unsigned char>(*c)));
  const std::string path = std::string("/sys/bus/pci/devices/") + bus + "/local_cpulist";
  std::FILE* f = std::fopen(path.c_str(), "r");
  if (!f) return TSB_EUNSUPPORTED;
  char line[4096] = {0};
  const bool got = std::fgets(line, sizeof(line) - 1, f) != nullptr;
  std::fclose(f);
  if (!got) return TSB_EUNSUPPORTED;
  cpu_set_t want, have;
  CPU_ZERO(&want);
  int count = 0;
  for (const char* p = line; *p;) {  // "0-31,64-95"
    char* end = nullptr;
    const long a = std::strtol(p, &end, 10);
    if (end == p) break;
    long b = a;
    p = end;
    if (*p == '-') {
      b = std::strtol(p + 1, &end, 10);
      p = end;
    }
    for (long c = a; c <= b && c < CPU_SETSIZE; c++) CPU_SET(static_cast<int>(c), &want);
    if (*p == ',') ++p;
  }
  if (sched_getaffinity(0, sizeof(have), &have) != 0) return TSB_EUNSUPPORTED;
  cpu_set_t both;
  CPU_AND(&both, &want, &have);  // never outside what the process was given (containers, taskset)
  count = CPU_COUNT(&both);
  if (count == 0) return TSB_EUNSUPPORTED;
  if (sched_setaffinity(0, sizeof(both), &both) != 0) return TSB_EUNSUPPORTED;
  return count;
}

int tsb_init_devices(int n) {
  int have = 0;
  if (cudaGetDeviceCount(&have) != cudaSuccess || have < 1) {
    (void)cudaGetLastError();
    return TSB_ENODEV;
  }
  for (int d = 0; d < n && d < have; d++) {
    TSB_CUDA(cudaSetDevice(d));
    TSB_CUDA(cudaFree(nullptr));
    // the library's kernels are loaded lazily, as one module, at the first launch (~15 ms): do it here, where
    // the Chapel runtime loads its own GPU code — at program start, outside the drivers' timers
    cudaFuncAttributes fa;
    TSB_CUDA(cudaFuncGetAttributes(&fa, tsb::nq_evaluate_kernel<1, 0>));
  }
  // peer access between the devices of a multi-GPU search, once and before any timer (the first
  // cudaDeviceEnablePeerAccess of a pair takes milliseconds): steals between device pools then go GPU to GPU
  // over NVLink instead of being staged through the host
  static std::mutex peer_mu;
  static bool peer_on[16][16] = {};
  std::lock_guard<std::mutex> lk(peer_mu);
  const int nd = std::min(std::min(n, have), 16);
  for (int a = 0; a < nd && nd > 1; a++)
    for (int b = 0; b < nd; b++)
      if (a != b && !peer_on[a][b]) {
        enable_peer(a, b);
        peer_on[a][b] = true;
      }
  return TSB_OK;
}

// ---------------------------------------------------------------- N-Queens
int tsb_nq_create(tsb_nq** out, int device, int N, int g, int M_max) {
  if (!out || N < 1 || N > TSB_MAX_QUEENS || g < 1 || M_max < 1) return TSB_EINVAL;
  tsb_nq* h = new (std::nothrow) tsb_nq();
  if (!h) return TSB_ENOMEM;
  h->N = N;
  h->g = g;
  if (const char* v = std::getenv("TSB200_NQ_VARIANT")) h->variant = std::atoi(v);
  if (const char* v = std::getenv("TSB200_NQ_TILE_THREADS")) h->tile_threads = std::atoi(v);
  int rc = h->init(device, M_max, sizeof(tsb_nq_node), static_cast<size_t>(N));
  if (rc != TSB_OK) {
    h->fini();
    delete h;
    return rc;
  }
  *out = h;
  return TSB_OK;
}

void tsb_nq_destroy(tsb_nq* h) {
  if (!h) return;
  for (tsb_nq*& x : h->sibling) {
    if (x) tsb_nq_destroy(x);
    x = nullptr;
  }
  cudaSetDevice(h->device);
  if (h->stream) cudaStreamSynchronize(h->stream);
  h->ex.release();
  h->rounds.release();
  if (h->d_children) cudaFree(h->d_children);
  h->pool.release();
  h->fini();
  delete h;
}

// ---- fused evaluate + generate_children, and the device-resident pool (SURVEY §8f rows 1, 3)
int tsb_nq_expand_device(tsb_nq* h, const void* parents_d, int count, void* children_d, uint64_t* n_children,
                         uint64_t* n_solutions, void* stream) {
  if (!h || count < 0 || !n_children || !n_solutions) return TSB_EINVAL;
  *n_children = *n_solutions = 0;
  if (count == 0) return TSB_OK;
  if (!parents_d || !children_d) return TSB_EINVAL;
  if (reinterpret_cast<uintptr_t>(parents_d) & 15) return TSB_EALIGN;
  TSB_CUDA(cudaSetDevice(h->device));
  unsigned long long nc = 0, ns = 0;
  const std::vector<PoolExtent> pieces{{0, count}};
  int rc = nq_expand_dispatch(h, static_cast<const uint8_t*>(parents_d), pieces, static_cast<uint8_t*>(children_d),
                              stream ? static_cast<cudaStream_t>(stream) : h->stream, &nc, &ns);
  *n_children = nc;
  *n_solutions = ns;
  return rc;
}

int tsb_nq_expand(tsb_nq* h, const void* parents, int count, void* children, uint64_t capacity, uint64_t* n_children,
                  uint64_t* n_solutions) {
  if (!h || count < 0 || count > h->M_max || !n_children || !n_solutions) return TSB_EINVAL;
  *n_children = *n_solutions = 0;
  if (count == 0) return TSB_OK;
  if (!parents || !children) return TSB_EINVAL;
  TSB_CUDA(cudaSetDevice(h->device));
  const size_t need = static_cast<size_t>(h->M_max) * h->N * sizeof(tsb_nq_node) + 64;
  if (h->d_children_bytes < need) {
    if (h->d_children) cudaFree(h->d_children);
    h->d_children = nullptr;
    h->d_children_bytes = 0;
    TSB_CUDA(cudaMalloc(&h->d_children, need));
    h->d_children_bytes = need;
  }
  int rc = h->copy_h2d(h->d_in, parents, sizeof(tsb_nq_node) * static_cast<size_t>(count), h->stream);
  if (rc != TSB_OK) return rc;
  unsigned long long nc = 0, ns = 0;
  const std::vector<PoolExtent> pieces{{0, count}};
  rc = nq_expand_dispatch(h, h->d_in, pieces, h->d_children, h->stream, &nc, &ns);
  if (rc != TSB_OK) return rc;
  *n_children = nc;
  *n_solutions = ns;
  if (nc > capacity) return TSB_ENOMEM;  // the caller's children array is too small; counts are valid
  return h->copy_d2h(children, h->d_children, nc * sizeof(tsb_nq_node), h->stream);
}

}  // extern "C"
namespace {
// arena capacity a handle starts with: four worst-case rounds (every slot of every parent survives)
long long nq_pool_min_cap(const tsb_nq* h) {
  if (const long long c = env_pool_cap(); c > 0) return c;
  return std::max<long long>(1LL << 22, 4LL * h->M_max * h->N);
}
// A/B experiment, off by default (TSB200_AUX=1 turns it on): one side word per node (nq_expand2.cuh).  Measured on
// the N = 17 search at M = 4 Mi: count 36.8 us + build 59.9 us per round against 44.6 + 51.5 us without — the
// instructions it saves in the count kernel are paid back as 38 % more bytes per node.
bool env_aux() {
  static const bool v = [] {
    const char* e = std::getenv("TSB200_AUX");
    return e && *e && *e != '0';
  }();
  return v;
}
void nq_pool_setup(tsb_nq* h) {
  h->pool.rec = sizeof(tsb_nq_node);
  h->pool.slack = static_cast<size_t>(tsb::NQ_TILE) * sizeof(tsb_nq_node);  // full-tile loads may run past the top
  if (env_aux()) {
    h->pool.side_rec = sizeof(unsigned long long);
    h->pool.side_slack = static_cast<size_t>(tsb::NQ_TILE) * sizeof(unsigned long long);
  }
}
template <int N>
int nq_aux_fill_n(tsb_nq* h, long long lo, long long hi) {
  if (hi <= lo) return TSB_OK;
  const long long blocks = std::min<long long>((hi - lo + 255) / 256, 64LL * h->di.sms);
  tsb::nq_aux_fill_kernel<N><<<static_cast<unsigned>(blocks), 256, 0, h->stream>>>(
      h->pool.arena[h->pool.cur], reinterpret_cast<unsigned long long*>(h->pool.side[h->pool.cur]), lo, hi);
  TSB_CUDA(cudaGetLastError());
  h->launches++;
  return TSB_OK;
}
int nq_aux_fill(tsb_nq* h, long long lo, long long hi) {
  switch (h->N) {
#define TSB_NQ_CASE(n) \
  case n:              \
    return nq_aux_fill_n<n>(h, lo, hi);
    TSB_NQ_CASE(1) TSB_NQ_CASE(2) TSB_NQ_CASE(3) TSB_NQ_CASE(4) TSB_NQ_CASE(5) TSB_NQ_CASE(6) TSB_NQ_CASE(7)
    TSB_NQ_CASE(8) TSB_NQ_CASE(9) TSB_NQ_CASE(10) TSB_NQ_CASE(11) TSB_NQ_CASE(12) TSB_NQ_CASE(13)
    TSB_NQ_CASE(14) TSB_NQ_CASE(15) TSB_NQ_CASE(16) TSB_NQ_CASE(17) TSB_NQ_CASE(18) TSB_NQ_CASE(19)
    TSB_NQ_CASE(20)
#undef TSB_NQ_CASE
  }
  return TSB_EINVAL;
}
// side words for every node of the pool (after host pushes into a pool whose words were stale, a steal, the
// persistent kernel's export)
int nq_aux_ensure(tsb_nq* h) {
  if (h->aux_ok || !h->pool.side_rec) return TSB_OK;
  for (const PoolExtent& x : h->pool.ext)
    if (int rc = nq_aux_fill(h, x.b, x.e); rc != TSB_OK) return rc;
  h->aux_ok = true;
  return TSB_OK;
}
}  // namespace
extern "C" {

int tsb_nq_pool_push(tsb_nq* h, const void* nodes, int64_t n) {
  if (!h || n < 0 || (n && !nodes)) return TSB_EINVAL;
  TSB_CUDA(cudaSetDevice(h->device));
  nq_pool_setup(h);
  int rc = nq_materialize(h);
  if (rc != TSB_OK) return rc;
  h->rounds.aux_valid = 0;  // (the side words of the persistent kernel describe the pool it left behind)
  rc = h->pool.reserve(h->stream, n, nq_pool_min_cap(h));
  if (rc != TSB_OK) return rc;
  if (n == 0) return TSB_OK;
  const long long at = h->pool.top();
  // (on the handle's non-blocking stream, which the kernels of the next round are ordered after)
  rc = h->copy_h2d(h->pool.arena[h->pool.cur] + at * sizeof(tsb_nq_node), nodes,
                   static_cast<size_t>(n) * sizeof(tsb_nq_node), h->stream);
  if (rc != TSB_OK) return rc;
  if (h->pool.size == 0) h->aux_ok = true;  // (nothing else to describe)
  if (h->pool.ext.empty())
    h->pool.ext.push_back({at, at + n});
  else
    h->pool.ext.back().e += n;
  h->pool.size += n;
  if (h->aux_ok && h->pool.side_rec) return nq_aux_fill(h, at, at + n);  // (ordered after the copy on the handle's stream)
  return TSB_OK;
}

int64_t tsb_nq_pool_size(const tsb_nq* h) { return h ? h->pool.size : -1; }

int tsb_nq_pool_step(tsb_nq* h, int m, int M, int64_t* n_parents, uint64_t* n_children, uint64_t* n_solutions) {
  if (!h || m < 1 || M < 1 || M > h->M_max || !n_parents || !n_children || !n_solutions) return TSB_EINVAL;
  *n_parents = 0;
  *n_children = *n_solutions = 0;
  DevicePool& p = h->pool;
  if (p.size < m) return TSB_OK;  // popBackBulk returns 0 below m (lib/commons/Pool.chpl:50-59)
  TSB_CUDA(cudaSetDevice(h->device));
  int rc = nq_materialize(h);
  if (rc != TSB_OK) return rc;
  h->rounds.aux_valid = 0;
  const long long n = std::min<long long>(p.size, M);
  // room above the top for the worst case (every slot of every parent survives); the chunk itself is read
  // in place, as the newest pieces of the extent stack
  std::vector<PoolExtent> pieces;
  pool_top_pieces(p, n, &pieces);
  if (pieces.size() > tsb::EXP_MAX_PIECES)
    rc = p.compact(h->stream, p.cap);
  if (rc == TSB_OK) rc = p.reserve(h->stream, n * h->N, nq_pool_min_cap(h));
  if (rc != TSB_OK) return rc;
  pool_top_pieces(p, n, &pieces);  // (positions change when the pool was compacted)
  const long long top = p.top();
  unsigned long long nc = 0, ns = 0;
  uint8_t* arena = p.arena[p.cur];
  if (p.side_rec) {  // every node evaluated once, when it is built (nq_expand2.cuh)
    rc = nq_aux_ensure(h);
    if (rc != TSB_OK) return rc;
    unsigned long long* side = reinterpret_cast<unsigned long long*>(p.side[p.cur]);
    rc = nq_expand_dispatch(h, arena, pieces, arena + top * sizeof(tsb_nq_node), h->stream, &nc, &ns, /*early=*/true, side,
                            side + top);
  } else {
    rc = nq_expand_dispatch(h, arena, pieces, arena + top * sizeof(tsb_nq_node), h->stream, &nc, &ns, /*early=*/true);
  }
  if (rc != TSB_OK) return rc;
  pool_pop(p, n);
  if (nc) {
    p.ext.push_back({top, top + static_cast<long long>(nc)});
    p.size += static_cast<long long>(nc);
  }
  *n_parents = n;
  *n_children = nc;
  *n_solutions = ns;
  return TSB_OK;
}

}  // extern "C"
namespace {
template <int N, int T>
int nq_rounds_launch_nt(tsb_nq* h, const tsb::RoundsParams& prm, int grid, cudaStream_t s) {
  auto kernel = tsb::nq_rounds_kernel<N, T>;
  const size_t smem = sizeof(tsb::RoundsSmem<T>) + 128;
  if (!h->rounds.attr_set) {
    TSB_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    h->rounds.attr_set = true;
  }
  void* args[] = {const_cast<tsb::RoundsParams*>(&prm)};
  // cooperative: all CTAs co-resident (they exchange flags through L2), or the launch fails
  TSB_CUDA(cudaLaunchCooperativeKernel(reinterpret_cast<void*>(kernel), dim3(grid), dim3(T), args, smem, s));
  h->launches++;
  return TSB_OK;
}
template <int N>
int nq_rounds_launch_n(tsb_nq* h, const tsb::RoundsParams& prm, int grid, cudaStream_t s) {
  if (h->rounds.threads == 256) return nq_rounds_launch_nt<N, 256>(h, prm, grid, s);
  return nq_rounds_launch_nt<N, 512>(h, prm, grid, s);
}
int nq_rounds_launch(tsb_nq* h, const tsb::RoundsParams& prm, int grid, cudaStream_t s) {
  switch (h->N) {
#define TSB_NQ_CASE(n) \
  case n:              \
    return nq_rounds_launch_n<n>(h, prm, grid, s);
    TSB_NQ_CASE(1) TSB_NQ_CASE(2) TSB_NQ_CASE(3) TSB_NQ_CASE(4) TSB_NQ_CASE(5) TSB_NQ_CASE(6) TSB_NQ_CASE(7)
    TSB_NQ_CASE(8) TSB_NQ_CASE(9) TSB_NQ_CASE(10) TSB_NQ_CASE(11) TSB_NQ_CASE(12) TSB_NQ_CASE(13)
    TSB_NQ_CASE(14) TSB_NQ_CASE(15) TSB_NQ_CASE(16) TSB_NQ_CASE(17) TSB_NQ_CASE(18) TSB_NQ_CASE(19)
    TSB_NQ_CASE(20)
#undef TSB_NQ_CASE
  }
  return TSB_EINVAL;
}
template <int N>
int nq_ll_launch_n(tsb_nq* h, const tsb::LlMultiParams& prm, int grid, int pools, int ppt, cudaStream_t s) {
  // (one pool: the 160-register build, one CTA per SM; several: capped at 128 registers for two CTAs per SM; three
  // or four pools: 74 CTAs per pool with 768 parents each, see ll_slice)
  // ppt > 10: the three-CTAs-per-SM build (80 registers, 64 KB of shared memory) with ppt - 10 parents per thread
  const int var = pools == 1 ? 0 : ppt == 2 ? 1 : ppt == 3 ? 2 : 3;
  auto kernel = var == 0   ? tsb::nq_rounds_ll_kernel<N, tsb::LL_T, 1, 2>
                : var == 1 ? tsb::nq_rounds_ll_kernel<N, tsb::LL_T, 2, 2>
                : var == 2 ? tsb::nq_rounds_ll_kernel<N, tsb::LL_T, 2, 3>
                           : tsb::nq_rounds_ll_kernel<N, tsb::LL_T, 3, 2>;
  const size_t smem = (var == 0   ? sizeof(tsb::LlSmem<tsb::LL_T, 2, 1>)
                       : var == 1 ? sizeof(tsb::LlSmem<tsb::LL_T, 2, 2>)
                       : var == 2 ? sizeof(tsb::LlSmem<tsb::LL_T, 3, 2>)
                                  : sizeof(tsb::LlSmem<tsb::LL_T, 2, 3>)) + 128;
  bool& attr = h->rounds.attr_llv[var];
  if (!attr) {
    TSB_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    attr = true;
  }
  void* args[] = {const_cast<tsb::LlMultiParams*>(&prm)};
  // cooperative: all CTAs of all pools co-resident (two per SM when there are two pools), or the launch fails
  TSB_CUDA(cudaLaunchCooperativeKernel(reinterpret_cast<void*>(kernel), dim3(grid, pools), dim3(tsb::LL_T), args, smem, s));
  h->launches++;
  return TSB_OK;
}
template <int N>
int nq_ll_import_n(tsb_nq* h, long long size, cudaStream_t s) {
  if (size > 0) {
    tsb::nq_fat_import_kernel<N><<<static_cast<unsigned>((size + 255) / 256), 256, 0, s>>>(
        h->pool.arena[h->pool.cur], h->rounds.d_fat, size, h->rounds.epoch);
    TSB_CUDA(cudaGetLastError());
    h->launches++;
  }
  return TSB_OK;
}
int nq_ll_launch(tsb_nq* h, const tsb::LlMultiParams& prm, int grid, int pools, int ppt, cudaStream_t s) {
  switch (h->N) {
#define TSB_NQ_CASE(n) \
  case n:              \
    return nq_ll_launch_n<n>(h, prm, grid, pools, ppt, s);
    TSB_NQ_CASE(1) TSB_NQ_CASE(2) TSB_NQ_CASE(3) TSB_NQ_CASE(4) TSB_NQ_CASE(5) TSB_NQ_CASE(6) TSB_NQ_CASE(7)
    TSB_NQ_CASE(8) TSB_NQ_CASE(9) TSB_NQ_CASE(10) TSB_NQ_CASE(11) TSB_NQ_CASE(12) TSB_NQ_CASE(13)
    TSB_NQ_CASE(14) TSB_NQ_CASE(15) TSB_NQ_CASE(16) TSB_NQ_CASE(17) TSB_NQ_CASE(18) TSB_NQ_CASE(19)
    TSB_NQ_CASE(20)
#undef TSB_NQ_CASE
  }
  return TSB_EINVAL;
}
int nq_ll_import(tsb_nq* h, long long size, cudaStream_t s) {
  switch (h->N) {
#define TSB_NQ_CASE(n) \
  case n:              \
    return nq_ll_import_n<n>(h, size, s);
    TSB_NQ_CASE(1) TSB_NQ_CASE(2) TSB_NQ_CASE(3) TSB_NQ_CASE(4) TSB_NQ_CASE(5) TSB_NQ_CASE(6) TSB_NQ_CASE(7)
    TSB_NQ_CASE(8) TSB_NQ_CASE(9) TSB_NQ_CASE(10) TSB_NQ_CASE(11) TSB_NQ_CASE(12) TSB_NQ_CASE(13)
    TSB_NQ_CASE(14) TSB_NQ_CASE(15) TSB_NQ_CASE(16) TSB_NQ_CASE(17) TSB_NQ_CASE(18) TSB_NQ_CASE(19)
    TSB_NQ_CASE(20)
#undef TSB_NQ_CASE
  }
  return TSB_EINVAL;
}
// the pool back in the plain 21-byte arena (whoever needs the node records calls this first)
int nq_materialize(tsb_nq* h) {
  if (!h->rounds.in_fat) return TSB_OK;
  TSB_CUDA(cudaSetDevice(h->device));
  const long long size = h->pool.size;
  if (size > 0) {
    tsb::nq_fat_export_kernel<<<static_cast<unsigned>((size + 255) / 256), 256, 0, h->stream>>>(
        h->rounds.d_fat, h->pool.arena[h->pool.cur], size);
    TSB_CUDA(cudaGetLastError());
    h->launches++;
    TSB_CUDA(cudaStreamSynchronize(h->stream));
  }
  h->rounds.in_fat = false;
  h->aux_ok = false;  // (the exported nodes carry no side words)
  return TSB_OK;
}
bool env_no_rounds() {
  const char* v = std::getenv("TSB200_NO_ROUNDS");
  return v && *v && *v != '0';
}
// grid (CTAs per pool) of the persistent kernel for chunks of up to M parents when one launch serves `pools` pools;
// 0: M is too large for it.  Measured on the N = 17 search at M = 50000 (B200, 148 SMs): one pool: best at 128 CTAs
// (one per SM); two pools: 148 + 148 (two CTAs per SM; 128 + 128: 6 % slower); four pools: 74 CTAs each.
// *ppt: parents per thread of the kernel variant to launch (2, or 3 when the pool's CTAs would not cover M with 2).
int nq_ll_grid(const tsb_nq* h, int M, int pools, int* ppt = nullptr) {
  if (!h->di.coop || env_no_rounds() || pools < 1 || pools > tsb::LL_MAX_POOLS) return 0;
  const int sms = std::min(h->di.sms, static_cast<int>(tsb::RND_MAX_CTAS));
  int most = pools == 1 ? sms : 2 * sms / pools;  // two CTAs per SM in all
  int per = static_cast<long long>(most) * tsb::ll_slice(2) >= M ? 2 : 3;
  if (pools > 1 && h->rounds.ppt == 3) per = 3;
  bool occ3 = false;
  if (pools > 1 && h->rounds.occ == 3 && static_cast<long long>(3 * sms / pools) * tsb::ll_slice(2) >= M) {
    most = 3 * sms / pools;  // three CTAs per SM in all, 512 parents per CTA
    per = 2;
    occ3 = true;
  }
  const int slice = tsb::ll_slice(per);
  int grid = pools == 1 ? std::max(1, (sms * 7 / 8) & ~1) : most;
  if (h->rounds.ctas > 0) grid = std::min(most, h->rounds.ctas);
  while (static_cast<long long>(grid) * slice < M && grid < most) ++grid;  // (M decides)
  if (ppt) *ppt = occ3 ? 12 : per;
  return static_cast<long long>(M) <= static_cast<long long>(grid) * slice && (pools > 1 || per == 2) ? grid : 0;
}
// Up to `max_rounds` rounds of EACH of the K pools (handles on one device, same N) in launches of the persistent
// kernel that serve all pools that still have work: grid (grid, pools).  out[4 i ..] += {rounds, parents, children,
// solutions} of pool i.  A pool leaves the launch on its own (done, round budget, arena full, layer table full); the
// launch ends when every pool has left, the pools that stopped for room grow and go again.
int nq_ll_run_multi(tsb_nq* const* hs, int K, int m, int M, int64_t max_rounds, uint64_t* out) {
  int64_t left[tsb::LL_MAX_POOLS];
  bool active[tsb::LL_MAX_POOLS];
  for (int i = 0; i < K; i++) {
    left[i] = max_rounds;
    active[i] = true;
    nq_pool_setup(hs[i]);
    int rc = hs[i]->rounds.ensure(hs[i]->stream);
    if (rc != TSB_OK) return rc;
  }
  const bool prof = std::getenv("TSB200_ROUNDS_PROF") != nullptr;
  for (;;) {
    tsb::LlMultiParams mp;
    std::memset(&mp, 0, sizeof(mp));
    int map[tsb::LL_MAX_POOLS], n_act = 0;
    long long need_of[tsb::LL_MAX_POOLS];
    for (int i = 0; i < K; i++) {
      tsb_nq* h = hs[i];
      DevicePool& p = h->pool;
      if (!active[i] || p.size < m || left[i] <= 0) {
        active[i] = false;
        continue;
      }
      const long long n = std::min<long long>(p.size, M);
      const long long need = p.size - n + n * h->N;
      int rc = TSB_OK;
      if (h->rounds.in_fat && need > p.cap) rc = nq_materialize(h);  // (grows below and imports again)
      if (rc != TSB_OK) return rc;
      if (!h->rounds.in_fat) {
        // the plain pool as ONE contiguous stack [0, size) with room for the worst case of the next round
        if (need > p.cap)
          rc = p.compact(h->stream, std::max<long long>(2 * p.cap, need + need / 2));
        else if (p.ext.size() != 1 || p.ext[0].b != 0)
          rc = p.compact(h->stream, p.cap);
        if (rc == TSB_OK) rc = h->rounds.ensure_fat(p.cap, h->stream);
        if (rc == TSB_OK) rc = nq_ll_import(h, p.size, h->stream);
        if (rc != TSB_OK) return rc;
        h->rounds.in_fat = true;
        if (n_act > 0) TSB_CUDA(cudaStreamSynchronize(h->stream));  // (the launch goes on the first pool's stream)
      }
      tsb::LlParams& prm = mp.pool[n_act];
      prm.fat = h->rounds.d_fat;
      prm.cap = std::min(p.cap, h->rounds.fat_cap);
      prm.size0 = p.size;
      prm.epoch0 = h->rounds.epoch;
      prm.m = m;
      prm.M = M;
      prm.max_rounds = left[i];
      prm.prof = prof;
      prm.sync = h->rounds.d_ll;
      prm.state = h->rounds.d_state;
      h->rounds.h_state->exit_code = -1;
      need_of[n_act] = need;
      map[n_act++] = i;
    }
    if (n_act == 0) break;
    tsb_nq* h0 = hs[map[0]];
    // (variant and grid follow the number of pools that still run: a lone survivor gets the one-pool kernel)
    int ppt = 2;
    const int grid = nq_ll_grid(h0, M, n_act, &ppt);
    if (grid == 0) return TSB_EINVAL;  // (checked by the callers for K pools, and fewer pools fit a fortiori)
    int rc = nq_ll_launch(h0, mp, grid, n_act, ppt, h0->stream);
    if (rc != TSB_OK) return rc;
    TSB_CUDA(cudaStreamSynchronize(h0->stream));
    for (int a = 0; a < n_act; a++) {
      const int i = map[a];
      tsb_nq* h = hs[i];
      DevicePool& p = h->pool;
      const tsb::RoundsState st = *h->rounds.h_state;
      if (st.exit_code < 0 || st.exit_code == tsb::RND_EXIT_ABORT) {
        g_last_cuda_error = "nq_rounds_ll_kernel: watchdog abort (a flag exchange or a node poll did not complete)";
        return TSB_ECUDA;
      }
      if (prof)
        std::fprintf(stderr, "[tsb200] LL rounds kernel (pool %d of %d): %llu rounds; CTA 0 cycles per round: build %.0f | fence-check %.0f "
                     "poll-nodes %.0f scan+items %.0f gather-wait %.0f store %.0f signal %.0f\n", a, n_act,
                     static_cast<unsigned long long>(st.rounds), 1.0 * st.prof[6] / std::max<unsigned long long>(1, st.rounds),
                     1.0 * st.prof[0] / std::max<unsigned long long>(1, st.rounds), 1.0 * st.prof[1] / std::max<unsigned long long>(1, st.rounds),
                     1.0 * st.prof[2] / std::max<unsigned long long>(1, st.rounds), 1.0 * st.prof[3] / std::max<unsigned long long>(1, st.rounds),
                     1.0 * st.prof[4] / std::max<unsigned long long>(1, st.rounds), 1.0 * st.prof[5] / std::max<unsigned long long>(1, st.rounds));
      h->rounds.epoch = st.epoch;
      p.size = st.size;
      p.ext.clear();
      if (p.size) p.ext.push_back({0, p.size});
      out[4 * i + 0] += st.rounds;
      out[4 * i + 1] += st.parents;
      out[4 * i + 2] += st.children;
      out[4 * i + 3] += st.solutions;
      left[i] -= static_cast<int64_t>(st.rounds);
      if (st.exit_code == tsb::RND_EXIT_SPACE) {
        if (st.rounds == 0 && need_of[a] <= p.cap) return TSB_ENOMEM;  // (cannot happen)
        rc = nq_materialize(h);  // back to the plain arena, which then grows
        if (rc != TSB_OK) return rc;
      } else if (st.exit_code != tsb::RND_EXIT_RELAUNCH) {  // (layer table full: a fresh launch trusts the whole pool)
        active[i] = false;                                    // DONE or PAUSE
      }
    }
  }
  return TSB_OK;
}
}  // namespace
extern "C" {

int tsb_nq_pool_run(tsb_nq* h, int m, int M, int64_t max_rounds, uint64_t* n_rounds, uint64_t* n_parents,
                    uint64_t* n_children, uint64_t* n_solutions) {
  if (!h || m < 1 || M < 1 || M > h->M_max || max_rounds < 0 || !n_rounds || !n_parents || !n_children || !n_solutions)
    return TSB_EINVAL;
  *n_rounds = *n_parents = *n_children = *n_solutions = 0;
  DevicePool& p = h->pool;
  TSB_CUDA(cudaSetDevice(h->device));
  int rc = h->rounds.ensure(h->stream);
  if (rc != TSB_OK) return rc;
  int grid = std::min(h->di.sms, static_cast<int>(tsb::RND_MAX_CTAS));
  if (h->rounds.version == 3)  // measured best at 128 of 148 SMs
    grid = h->rounds.ctas > 0 ? std::min(grid, h->rounds.ctas) : std::max(1, (grid * 7 / 8) & ~1);
  else
    grid = h->rounds.ctas > 0 ? std::min(grid, h->rounds.ctas) : std::max(1, 2 * grid / 3);
  while (static_cast<long long>(grid) * h->rounds.threads * tsb::RND_PPT < M && grid < h->di.sms) ++grid;  // (M decides)
  const bool persistent = static_cast<long long>(M) <= static_cast<long long>(grid) * h->rounds.threads * tsb::RND_PPT &&
                          h->di.coop && !env_no_rounds();
  if (!persistent) {  // large chunks: one round = two bandwidth-bound kernels (tsb_nq_pool_step)
    while (static_cast<int64_t>(*n_rounds) < max_rounds) {
      int64_t np = 0;
      uint64_t nc = 0, ns = 0;
      int rc = tsb_nq_pool_step(h, m, M, &np, &nc, &ns);
      if (rc != TSB_OK) return rc;
      if (np == 0) break;
      ++*n_rounds;
      *n_parents += static_cast<uint64_t>(np);
      *n_children += nc;
      *n_solutions += ns;
    }
    return TSB_OK;
  }
  nq_pool_setup(h);
  if (h->rounds.version == 3 && nq_ll_grid(h, M, 1) > 0) {
    // ---- the fence-free kernel on the fat arena (nq_rounds_ll.cuh)
    uint64_t out[4] = {0, 0, 0, 0};
    tsb_nq* one[1] = {h};
    rc = nq_ll_run_multi(one, 1, m, M, max_rounds, out);
    *n_rounds = out[0];
    *n_parents = out[1];
    *n_children = out[2];
    *n_solutions = out[3];
    return rc;
  }
  nq_pool_setup(h);
  while (p.size >= m && static_cast<int64_t>(*n_rounds) < max_rounds) {
    // the kernel works on ONE contiguous stack [0, size) with room for the worst case of the next round
    const long long n = std::min<long long>(p.size, M);
    const long long need = p.size - n + n * h->N;
    if (need > p.cap) {
      rc = p.compact(h->stream, std::max<long long>(2 * p.cap, need + need / 2));
      h->rounds.aux_valid = 0;
    } else if (p.ext.size() != 1 || p.ext[0].b != 0) {
      rc = p.compact(h->stream, p.cap);
      h->rounds.aux_valid = 0;
    }
    if (rc == TSB_OK) rc = h->rounds.ensure_aux(p.cap);
    if (rc != TSB_OK) return rc;
    tsb::RoundsParams prm;
    prm.aux = h->rounds.d_aux;
    prm.aux_valid = std::min(h->rounds.aux_valid, p.size);
    prm.arena = p.arena[p.cur];
    prm.cap = p.cap;
    prm.size0 = p.size;
    prm.epoch0 = h->rounds.epoch;
    prm.m = m;
    prm.M = M;
    prm.max_rounds = max_rounds - static_cast<int64_t>(*n_rounds);
    prm.prof = std::getenv("TSB200_ROUNDS_PROF") != nullptr;
    prm.sync = h->rounds.d_sync;
    prm.state = h->rounds.d_state;
    h->rounds.h_state->exit_code = -1;
    rc = nq_rounds_launch(h, prm, grid, h->stream);
    if (rc != TSB_OK) return rc;
    TSB_CUDA(cudaStreamSynchronize(h->stream));
    const tsb::RoundsState st = *h->rounds.h_state;
    if (st.exit_code < 0 || st.exit_code == tsb::RND_EXIT_ABORT) {
      g_last_cuda_error = "nq_rounds_kernel: watchdog abort (a flag exchange did not complete)";
      return TSB_ECUDA;
    }
    if (prm.prof)
      std::fprintf(stderr, "[tsb200] rounds kernel: %llu rounds; CTA 0 cycles per round: wait-done %.0f load %.0f eval+scan %.0f "
                   "gather %.0f build+store %.0f release %.0f\n", static_cast<unsigned long long>(st.rounds),
                   1.0 * st.prof[0] / std::max<unsigned long long>(1, st.rounds), 1.0 * st.prof[1] / std::max<unsigned long long>(1, st.rounds),
                   1.0 * st.prof[2] / std::max<unsigned long long>(1, st.rounds), 1.0 * st.prof[3] / std::max<unsigned long long>(1, st.rounds),
                   1.0 * st.prof[4] / std::max<unsigned long long>(1, st.rounds), 1.0 * st.prof[5] / std::max<unsigned long long>(1, st.rounds));
    h->rounds.epoch = st.epoch;
    h->aux_ok = false;
    h->rounds.aux_valid = st.size;
    p.size = st.size;
    p.ext.clear();
    if (p.size) p.ext.push_back({0, p.size});
    *n_rounds += st.rounds;
    *n_parents += st.parents;
    *n_children += st.children;
    *n_solutions += st.solutions;
    if (st.exit_code == tsb::RND_EXIT_SPACE && st.rounds == 0 && need <= p.cap) return TSB_ENOMEM;  // (cannot happen)
    if (st.exit_code != tsb::RND_EXIT_SPACE) break;  // DONE or PAUSE
  }
  return TSB_OK;
}

int tsb_nq_sibling(tsb_nq* h, int index, tsb_nq** sibling) {
  if (!h || !sibling || index < 1 || index >= tsb::LL_MAX_POOLS) return TSB_EINVAL;
  if (!h->sibling[index - 1]) {
    int rc = tsb_nq_create(&h->sibling[index - 1], h->device, h->N, h->g, h->M_max);
    if (rc != TSB_OK) return rc;
  }
  *sibling = h->sibling[index - 1];
  return TSB_OK;
}

int tsb_nq_pools_per_launch(const tsb_nq* h, int M) {
  if (!h || M < 1 || M > h->M_max || h->rounds.version != 3) return 1;
  for (int pools = tsb::LL_MAX_POOLS; pools > 1; pools--)
    if (nq_ll_grid(h, M, pools) > 0) return pools;
  return 1;
}

int tsb_nq_pool_run_multi(tsb_nq* const* handles, int n_pools, int m, int M, int64_t max_rounds, uint64_t* out) {
  if (!handles || n_pools < 1 || n_pools > tsb::LL_MAX_POOLS || m < 1 || M < 1 || max_rounds < 0 || !out) return TSB_EINVAL;
  for (int i = 0; i < n_pools; i++) {
    const tsb_nq* h = handles[i];
    if (!h || M > h->M_max || h->device != handles[0]->device || h->N != handles[0]->N) return TSB_EINVAL;
    for (int j = 0; j < i; j++)
      if (handles[j] == h) return TSB_EINVAL;
  }
  std::memset(out, 0, sizeof(uint64_t) * 4 * n_pools);
  TSB_CUDA(cudaSetDevice(handles[0]->device));
  const int grid = handles[0]->rounds.version == 3 ? nq_ll_grid(handles[0], M, n_pools) : 0;
  if (grid == 0) {  // chunks too large for the persistent kernel with this many pools: one pool after the other
    for (int i = 0; i < n_pools; i++) {
      int rc = tsb_nq_pool_run(handles[i], m, M, max_rounds, &out[4 * i], &out[4 * i + 1], &out[4 * i + 2], &out[4 * i + 3]);
      if (rc != TSB_OK) return rc;
    }
    return TSB_OK;
  }
  return nq_ll_run_multi(handles, n_pools, m, M, max_rounds, out);
}

int tsb_nq_pool_steal(tsb_nq* victim, tsb_nq* thief, int m, int64_t* n_stolen) {
  if (!victim || !thief || victim == thief || m < 1 || !n_stolen || victim->N != thief->N) return TSB_EINVAL;
  nq_pool_setup(victim);
  nq_pool_setup(thief);
  long long n = 0;
  if (victim->pool.size < 2LL * m) {
    *n_stolen = 0;
    return TSB_OK;
  }
  int rc = nq_materialize(victim);
  if (rc == TSB_OK) rc = nq_materialize(thief);
  if (rc != TSB_OK) return rc;
  victim->rounds.aux_valid = 0;
  thief->rounds.aux_valid = 0;
  rc = pool_steal_front(victim->pool, victim->device, victim->stream, thief->pool, thief->device, thief->stream, m,
                            nq_pool_min_cap(thief), &n);
  *n_stolen = n;
  if (n) thief->aux_ok = false;  // (the stolen nodes arrive without side words: filled before the thief's next round)
  return rc;
}

// diagnostics: cycles per round of the bare flag-exchange skeleton of the persistent kernel (nq_rounds.cuh)
int tsb_debug_flag_exchange(int device, int rounds, int variant, int ctas, double* cycles_per_round) {
  if (!cycles_per_round || rounds < 1) return TSB_EINVAL;
  DeviceInfo di;
  int rc = query_device(device, di);
  if (rc != TSB_OK) return rc;
  if (!di.coop) return TSB_EUNSUPPORTED;
  tsb::RoundsSync* sy = nullptr;
  uint4* scratch = nullptr;
  long long* d_out = nullptr;
  int grid = std::min(di.sms, static_cast<int>(tsb::RND_MAX_CTAS));
  if (ctas > 0 && ctas < grid) grid = ctas;
  TSB_CUDA(cudaMalloc(&sy, sizeof(*sy)));
  const size_t scratch_bytes = std::max<size_t>((static_cast<size_t>(grid) * tsb::RND_THREADS + 2) * sizeof(uint4), 2 * 256 * 256 * 4);
  TSB_CUDA(cudaMalloc(&scratch, scratch_bytes));
  TSB_CUDA(cudaMemset(scratch, 0, scratch_bytes));
  TSB_CUDA(cudaMalloc(&d_out, sizeof(long long)));
  TSB_CUDA(cudaMemset(sy, 0, sizeof(*sy)));
  unsigned epoch0 = 0;
  void* args[] = {&sy, &epoch0, &rounds, &variant, &scratch, &d_out};
  cudaError_t e = cudaLaunchCooperativeKernel(reinterpret_cast<void*>(tsb::rounds_sync_bench_kernel), dim3(grid),
                                              dim3(tsb::RND_THREADS), args, 0, nullptr);
  if (e == cudaSuccess) e = cudaDeviceSynchronize();
  long long cyc = 0;
  if (e == cudaSuccess) e = cudaMemcpy(&cyc, d_out, sizeof(cyc), cudaMemcpyDeviceToHost);
  cudaFree(sy);
  cudaFree(scratch);
  cudaFree(d_out);
  if (e != cudaSuccess) {
    g_last_cuda_error = std::string("flag exchange bench: ") + cudaGetErrorString(e);
    (void)cudaGetLastError();
    return TSB_ECUDA;
  }
  *cycles_per_round = static_cast<double>(cyc) / rounds;
  return TSB_OK;
}

int tsb_nq_pool_drain(tsb_nq* h, void* nodes, int64_t capacity, int64_t* n) {
  if (!h || !n || capacity < 0) return TSB_EINVAL;
  DevicePool& p = h->pool;
  *n = p.size;
  if (p.size > capacity) return TSB_ENOMEM;
  TSB_CUDA(cudaSetDevice(h->device));
  if (int rc = nq_materialize(h); rc != TSB_OK) return rc;
  long long at = 0;
  for (const PoolExtent& x : p.ext) {  // extents are the pool in logical (oldest first) order
    int rc = h->copy_d2h(static_cast<uint8_t*>(nodes) + at * sizeof(tsb_nq_node),
                         p.arena[p.cur] + x.b * sizeof(tsb_nq_node),
                         static_cast<size_t>(x.e - x.b) * sizeof(tsb_nq_node), h->stream);
    if (rc != TSB_OK) return rc;
    at += x.e - x.b;
  }
  p.ext.clear();
  p.size = 0;
  return TSB_OK;
}

int tsb_nq_evaluate(tsb_nq* h, const void* parents, int count, uint8_t* labels) {
  if (!h || count < 0 || count > h->M_max) return TSB_EINVAL;
  if (count == 0) return TSB_OK;
  if (!parents || !labels) return TSB_EINVAL;
  TSB_CUDA(cudaSetDevice(h->device));
  return h->evaluate_host(parents, count, labels, [h](const uint8_t* in, uint8_t* out, int n, cudaStream_t s) {
    return launch_nq(h, in, out, n, s);
  });
}

int tsb_nq_evaluate_device(tsb_nq* h, const void* parents_d, int count, uint8_t* labels_d, void* stream) {
  if (!h || count < 0) return TSB_EINVAL;
  if (count == 0) return TSB_OK;
  if (!parents_d || !labels_d) return TSB_EINVAL;
  if ((reinterpret_cast<uintptr_t>(parents_d) | reinterpret_cast<uintptr_t>(labels_d)) & 15) return TSB_EALIGN;
  TSB_CUDA(cudaSetDevice(h->device));
  cudaStream_t s = stream ? static_cast<cudaStream_t>(stream) : h->stream;
  return launch_nq(h, static_cast<const uint8_t*>(parents_d), labels_d, count, s);
}

int tsb_nq_register_host(tsb_nq* h, void* ptr, size_t bytes) {
  if (!h) return TSB_EINVAL;
  TSB_CUDA(cudaSetDevice(h->device));
  return h->reg.add(ptr, bytes);
}
int tsb_nq_unregister_host(tsb_nq* h, void* ptr) {
  if (!h) return TSB_EINVAL;
  TSB_CUDA(cudaSetDevice(h->device));
  return h->reg.remove(ptr);
}

int tsb_nq_set_xfer(tsb_nq* h, int mode) {
  if (!h || mode < 0 || mode > 2) return TSB_EINVAL;
  h->xfer = mode;
  return TSB_OK;
}
uint64_t tsb_nq_kernel_launches(const tsb_nq* h) {
  if (!h) return 0;
  uint64_t n = h->launches;
  for (const tsb_nq* x : h->sibling)
    if (x) n += x->launches;
  return n;
}
void* tsb_nq_stream(const tsb_nq* h) { return h ? static_cast<void*>(h->stream) : nullptr; }

// ---------------------------------------------------------------- PFSP
int tsb_pfsp_create(tsb_pfsp** out, int device, int jobs, int machines, int M_max, const int32_t* p_times,
                    const int32_t* min_heads, const int32_t* min_tails, int nb_pairs, const int32_t* johnson,
                    const int32_t* lags, const int32_t* mp0, const int32_t* mp1, const int32_t* mp_order) {
  if (!out || !p_times || !min_heads || !min_tails || M_max < 1 || nb_pairs < 0) return TSB_EINVAL;
  if (nb_pairs > 0 && (!johnson || !lags || !mp0 || !mp1 || !mp_order)) return TSB_EINVAL;
  if (jobs != TSB_MAX_JOBS || machines < 1 || machines > TSB_MAX_MACHINES || nb_pairs > TSB_MAX_PAIRS)
    return TSB_EUNSUPPORTED;
  tsb_pfsp* h = new (std::nothrow) tsb_pfsp();
  if (!h) return TSB_ENOMEM;
  h->jobs = jobs;
  h->machines = machines;
  h->pairs = nb_pairs;
  h->mt = machines <= 5 ? 5 : machines <= 10 ? 10 : 20;
  int rc = h->init(device, M_max, sizeof(tsb_pfsp_node), static_cast<size_t>(jobs) * 4);
  // tables -> device blob (zero padding up to the template machine count is value-neutral:
  // the reference itself evaluates 20-wide zero-padded tuples, lib/pfsp/Bound_simple.chpl:125-135)
  std::vector<tsb::PfspLb1Tables> t1v(1);
  tsb::PfspLb1Tables& t1 = t1v[0];
  std::memset(&t1, 0, sizeof(t1));
  const int mp = tsb::row_stride(h->mt);
  t1.jobs = jobs;
  t1.machines = machines;
  t1.pairs = nb_pairs;
  t1.mp = mp;
  long long sum_all = 0, max_head = 0, max_tail = 0;
  bool nonneg = true, tails_monotone = true;
  const int hs = tsb::half_stride(h->mt);
  for (int k = 0; k < machines; k++) {
    t1.min_heads[k] = min_heads[k];
    t1.min_tails[k] = min_tails[k];
    max_head = std::max<long long>(max_head, min_heads[k]);
    max_tail = std::max<long long>(max_tail, min_tails[k]);
    nonneg &= min_heads[k] >= 0 && min_tails[k] >= 0;
    if (k > 0) tails_monotone &= min_tails[k] <= min_tails[k - 1];
    for (int j = 0; j < jobs; j++) {
      const int32_t pv = p_times[k * jobs + j];
      t1.total[k] += pv;
      t1.pj[j * mp + k] = pv;
      nonneg &= pv >= 0;
      sum_all += pv;
      t1.ph[j * hs + (k >> 1)] |= static_cast<uint32_t>(pv & 0xFFFF) << (16 * (k & 1));
    }
  }
  // every intermediate of the bounds is <= sum of all processing times + largest head + largest tail
  h->simd16 = nonneg && tails_monotone && sum_all + max_head + max_tail < 65536 && !std::getenv("TSB200_NO_SIMD16");
  // lb2: packed Johnson tables in machine_pair_order (tsb::Lb2Const); value ranges checked, indices checked
  bool bad = false, wide = false;
  if (nb_pairs > 0) {
    h->lb2c = new (std::nothrow) tsb::Lb2Const();
    if (!h->lb2c) rc = TSB_ENOMEM;
  }
  for (int l = 0; l < nb_pairs && h->lb2c; l++) {
    const int i = mp_order[l];
    if (i < 0 || i >= nb_pairs) {
      bad = true;
      continue;
    }
    const int a = mp0[i], b = mp1[i];
    if (a < 0 || a >= machines || b < 0 || b >= machines) {
      bad = true;
      continue;
    }
    wide |= min_tails[a] < 0 || min_tails[a] > 2047 || min_tails[b] < 0 || min_tails[b] > 2047;
    h->lb2c->pair[l] = static_cast<uint32_t>(a) | static_cast<uint32_t>(b) << 5 |
                       static_cast<uint32_t>(min_tails[a] & 2047) << 10 | static_cast<uint32_t>(min_tails[b] & 2047) << 21;
    for (int j = 0; j < jobs; j++) {
      const int job = johnson[i * jobs + j];
      if (job < 0 || job >= jobs) {
        bad = true;
        continue;
      }
      const int pa = p_times[a * jobs + job], pb = p_times[b * jobs + job], lg = lags[i * jobs + job];
      wide |= pa < 0 || pa > 127 || pb < 0 || pb > 127 || lg < 0 || lg > 8191;
      h->lb2c->jp[l * tsb::PF_MAXJ + j] = static_cast<uint32_t>(job) | static_cast<uint32_t>(pa & 127) << 5 |
                                          static_cast<uint32_t>(pb & 127) << 12 | static_cast<uint32_t>(lg & 8191) << 19;
    }
  }
  // one-word-per-use table for the lb2 kernels of instances with <= 10 machines (env TSB200_NO_LB2U=1 disables)
  std::vector<tsb::Lb2TabU> tuv;
  const char* no_u = std::getenv("TSB200_NO_LB2U");
  if (rc == TSB_OK && !bad && !wide && nb_pairs > 0 && nb_pairs <= tsb::LB2U_PAIRS && h->mt <= 10 && h->simd16 &&
      !(no_u && *no_u && *no_u != '0')) {
    tuv.resize(1);
    tsb::Lb2TabU& tu = tuv[0];
    std::memset(&tu, 0, sizeof(tu));
    for (int l = 0; l < nb_pairs; l++) {
      const int i = mp_order[l], a = mp0[i], b = mp1[i];
      tu.mach[l] = static_cast<uint32_t>(a) | static_cast<uint32_t>(b) << 8;
      tu.tails[l] = static_cast<uint32_t>(min_tails[a]) | static_cast<uint32_t>(min_tails[b]) << 16;
      for (int j = 0; j < jobs; j++) {
        const int job = johnson[i * jobs + j];
        const int pa = p_times[a * jobs + job], pb = p_times[b * jobs + job], lg = lags[i * jobs + job];
        tu.e[l * tsb::PF_MAXJ + j] = make_uint4(1u << job, static_cast<uint32_t>(pa + lg),
                                                 static_cast<uint32_t>(pa - pb), 0u);
      }
    }
  }
  if (rc == TSB_OK && bad) rc = TSB_EINVAL;
  if (rc == TSB_OK && wide) {  // processing times > 127 / lags > 8191 (outside the Taillard range): no lb2 on this handle
    delete h->lb2c;
    h->lb2c = nullptr;
    h->pairs = 0;
  }
  auto upload = [&]() -> int {
    TSB_CUDA(cudaMalloc(&h->d_tab1, sizeof(t1)));
    TSB_CUDA(cudaMemcpyAsync(h->d_tab1, &t1, sizeof(t1), cudaMemcpyHostToDevice, h->stream));
    if (!tuv.empty()) {
      TSB_CUDA(cudaMalloc(&h->d_tabu, sizeof(tsb::Lb2TabU)));
      TSB_CUDA(cudaMemcpyAsync(h->d_tabu, tuv.data(), sizeof(tsb::Lb2TabU), cudaMemcpyHostToDevice, h->stream));
      h->lb2u = new (std::nothrow) tsb::Lb2ConstU{h->d_tabu};
    }
    TSB_CUDA(cudaStreamSynchronize(h->stream));
    return TSB_OK;
  };
  if (rc == TSB_OK) rc = upload();
  if (rc != TSB_OK) {
    tsb_pfsp_destroy(h);
    return rc;
  }
  *out = h;
  return TSB_OK;
}

// The reference built with MAX_JOBS = max_jobs (lib/pfsp/PFSP_node.chpl:7): 20 = tsb_pfsp_create; 50 = 208-byte nodes,
// jobs == 50 instances (ta031..ta060), evaluated by the general kernels of pfsp_wide.cuh; the fused expand and the
// device pool run the 208-byte kernels of pfsp_wide_expand.cuh
int tsb_pfsp_create_wide(tsb_pfsp** out, int device, int max_jobs, int jobs, int machines, int M_max, const int32_t* p_times,
                         const int32_t* min_heads, const int32_t* min_tails, int nb_pairs, const int32_t* johnson,
                         const int32_t* lags, const int32_t* mp0, const int32_t* mp1, const int32_t* mp_order) {
  if (max_jobs == TSB_MAX_JOBS)
    return tsb_pfsp_create(out, device, jobs, machines, M_max, p_times, min_heads, min_tails, nb_pairs, johnson, lags, mp0,
                           mp1, mp_order);
  if (!out || !p_times || !min_heads || !min_tails || M_max < 1 || nb_pairs < 0) return TSB_EINVAL;
  if (nb_pairs > 0 && (!johnson || !lags || !mp0 || !mp1 || !mp_order)) return TSB_EINVAL;
  if (max_jobs != TSB_MAX_JOBS_WIDE || jobs != max_jobs || machines < 1 || machines > TSB_MAX_MACHINES ||
      nb_pairs > TSB_MAX_PAIRS)
    return TSB_EUNSUPPORTED;
  tsb_pfsp* h = new (std::nothrow) tsb_pfsp();
  if (!h) return TSB_ENOMEM;
  h->jobs = jobs;
  h->machines = machines;
  h->pairs = nb_pairs;
  h->wide = true;
  h->mt = machines <= 5 ? 5 : machines <= 10 ? 10 : 20;
  int rc = h->init(device, M_max, tsb::PW_REC, static_cast<size_t>(jobs) * 4);
  std::vector<tsb::PfspWideTables> tv(1);
  tsb::PfspWideTables& t = tv[0];
  std::memset(&t, 0, sizeof(t));
  t.jobs = jobs;
  t.machines = machines;
  t.pairs = nb_pairs;
  bool bad = false, wide_values = false;
  for (int k = 0; k < machines; k++) {
    t.min_heads[k] = min_heads[k];
    t.min_tails[k] = min_tails[k];
    for (int j = 0; j < jobs; j++) {
      const int32_t pv = p_times[k * jobs + j];
      t.total[k] += pv;
      t.pj[j * tsb::PW_PSTRIDE + k] = pv;
    }
  }
  for (int l = 0; l < nb_pairs; l++) {
    const int i = mp_order[l];
    if (i < 0 || i >= nb_pairs) {
      bad = true;
      continue;
    }
    const int a = mp0[i], b = mp1[i];
    if (a < 0 || a >= machines || b < 0 || b >= machines) {
      bad = true;
      continue;
    }
    wide_values |= min_tails[a] < 0 || min_tails[a] > 2047 || min_tails[b] < 0 || min_tails[b] > 2047;
    t.pair[l] = static_cast<uint32_t>(a) | static_cast<uint32_t>(b) << 5 | static_cast<uint32_t>(min_tails[a] & 2047) << 10 |
                static_cast<uint32_t>(min_tails[b] & 2047) << 21;
    for (int j = 0; j < jobs; j++) {
      const int job = johnson[i * jobs + j];
      if (job < 0 || job >= jobs) {
        bad = true;
        continue;
      }
      const int pa = p_times[a * jobs + job], pb = p_times[b * jobs + job], lg = lags[i * jobs + job];
      wide_values |= pa < 0 || pa > 127 || pb < 0 || pb > 127 || lg < 0 || lg > 4095;
      t.jp[l * jobs + j] = static_cast<uint32_t>(job) | static_cast<uint32_t>(pa & 127) << 6 | static_cast<uint32_t>(pb & 127) << 13 |
                           static_cast<uint32_t>(lg & 4095) << 20;
    }
  }
  if (rc == TSB_OK && bad) rc = TSB_EINVAL;
  if (rc == TSB_OK && wide_values) h->pairs = 0;  // values outside the Taillard range: no lb2 on this handle
  auto upload = [&]() -> int {
    TSB_CUDA(cudaMalloc(&h->d_wtab, sizeof(t)));
    TSB_CUDA(cudaMemcpyAsync(h->d_wtab, &t, sizeof(t), cudaMemcpyHostToDevice, h->stream));
    TSB_CUDA(cudaStreamSynchronize(h->stream));
    return TSB_OK;
  };
  if (rc == TSB_OK) rc = upload();
  if (rc != TSB_OK) {
    tsb_pfsp_destroy(h);
    return rc;
  }
  *out = h;
  return TSB_OK;
}

void tsb_pfsp_destroy(tsb_pfsp* h) {
  if (!h) return;
  cudaSetDevice(h->device);
  if (h->stream) cudaStreamSynchronize(h->stream);
  if (h->d_tab1) cudaFree(h->d_tab1);
  if (h->d_wtab) cudaFree(h->d_wtab);
  delete h->lb2c;
  delete h->lb2u;
  if (h->d_tabu) cudaFree(h->d_tabu);
  h->ex.release();
  if (h->d_children) cudaFree(h->d_children);
  h->pool.release();
  h->fini();
  delete h;
}

int tsb_pfsp_evaluate(tsb_pfsp* h, int lb_kind, const void* parents, int count, int64_t best, int32_t* bounds) {
  if (!h || count < 0 || count > h->M_max || lb_kind < 0 || lb_kind > 2) return TSB_EINVAL;
  if (lb_kind == TSB_LB2 && h->pairs == 0) return TSB_EINVAL;
  if (count == 0) return TSB_OK;
  if (!parents || !bounds) return TSB_EINVAL;
  TSB_CUDA(cudaSetDevice(h->device));
  return h->evaluate_host(parents, count, bounds,
                          [h, lb_kind, best](const uint8_t* in, uint8_t* out, int n, cudaStream_t s) {
                            return launch_pfsp(h, lb_kind, in, out, n, best, s);
                          });
}

int tsb_pfsp_evaluate_device(tsb_pfsp* h, int lb_kind, const void* parents_d, int count, int64_t best,
                             int32_t* bounds_d, void* stream) {
  if (!h || count < 0 || lb_kind < 0 || lb_kind > 2) return TSB_EINVAL;
  if (lb_kind == TSB_LB2 && h->pairs == 0) return TSB_EINVAL;
  if (count == 0) return TSB_OK;
  if (!parents_d || !bounds_d) return TSB_EINVAL;
  if ((reinterpret_cast<uintptr_t>(parents_d) | reinterpret_cast<uintptr_t>(bounds_d)) & 15) return TSB_EALIGN;
  TSB_CUDA(cudaSetDevice(h->device));
  cudaStream_t s = stream ? static_cast<cudaStream_t>(stream) : h->stream;
  return launch_pfsp(h, lb_kind, static_cast<const uint8_t*>(parents_d), reinterpret_cast<uint8_t*>(bounds_d),
                     count, best, s);
}

int tsb_pfsp_register_host(tsb_pfsp* h, void* ptr, size_t bytes) {
  if (!h) return TSB_EINVAL;
  TSB_CUDA(cudaSetDevice(h->device));
  return h->reg.add(ptr, bytes);
}
int tsb_pfsp_unregister_host(tsb_pfsp* h, void* ptr) {
  if (!h) return TSB_EINVAL;
  TSB_CUDA(cudaSetDevice(h->device));
  return h->reg.remove(ptr);
}

int tsb_pfsp_set_xfer(tsb_pfsp* h, int mode) {
  if (!h || mode < 0 || mode > 2) return TSB_EINVAL;
  h->xfer = mode;
  return TSB_OK;
}
uint64_t tsb_pfsp_kernel_launches(const tsb_pfsp* h) { return h ? h->launches : 0; }
void* tsb_pfsp_stream(const tsb_pfsp* h) { return h ? static_cast<void*>(h->stream) : nullptr; }

uint64_t tsb_pfsp_slow_rounds(const tsb_pfsp* h) { return h ? h->slow_rounds : 0; }

int tsb_pfsp_expand_device(tsb_pfsp* h, int lb_kind, const void* parents_d, int count, int64_t* best,
                           void* children_d, uint64_t* n_children, uint64_t* n_solutions, void* stream) {
  if (!h || count < 0 || lb_kind < 0 || lb_kind > 2 || !best || !n_children || !n_solutions) return TSB_EINVAL;
  if (lb_kind == TSB_LB2 && h->pairs == 0) return TSB_EINVAL;
  *n_children = *n_solutions = 0;
  if (count == 0) return TSB_OK;
  if (!parents_d || !children_d || count > h->M_max) return TSB_EINVAL;
  // (208-byte children are written by whole-image TMA stores: 16-byte aligned like the parents)
  if ((reinterpret_cast<uintptr_t>(parents_d) & 15) || (reinterpret_cast<uintptr_t>(children_d) & (h->wide ? 15 : 7)))
    return TSB_EALIGN;
  TSB_CUDA(cudaSetDevice(h->device));
  unsigned long long nc = 0, ns = 0;
  const std::vector<PoolExtent> pieces{{0, count}};
  int rc = pfsp_expand_round(h, lb_kind, static_cast<const uint8_t*>(parents_d), pieces,
                             static_cast<uint8_t*>(children_d), stream ? static_cast<cudaStream_t>(stream) : h->stream,
                             best, &nc, &ns);
  *n_children = nc;
  *n_solutions = ns;
  return rc;
}

int tsb_pfsp_expand(tsb_pfsp* h, int lb_kind, const void* parents, int count, int64_t* best, void* children,
                    uint64_t capacity, uint64_t* n_children, uint64_t* n_solutions) {
  if (!h || count < 0 || count > h->M_max || lb_kind < 0 || lb_kind > 2 || !best || !n_children || !n_solutions)
    return TSB_EINVAL;
  if (lb_kind == TSB_LB2 && h->pairs == 0) return TSB_EINVAL;
  *n_children = *n_solutions = 0;
  if (count == 0) return TSB_OK;
  if (!parents || !children) return TSB_EINVAL;
  TSB_CUDA(cudaSetDevice(h->device));
  const size_t rec = h->rec();
  const size_t need = static_cast<size_t>(h->M_max) * h->jobs * rec + 64;
  if (h->d_children_bytes < need) {
    if (h->d_children) cudaFree(h->d_children);
    h->d_children = nullptr;
    h->d_children_bytes = 0;
    TSB_CUDA(cudaMalloc(&h->d_children, need));
    h->d_children_bytes = need;
  }
  int rc = h->copy_h2d(h->d_in, parents, rec * static_cast<size_t>(count), h->stream);
  if (rc != TSB_OK) return rc;
  unsigned long long nc = 0, ns = 0;
  const std::vector<PoolExtent> pieces{{0, count}};
  rc = pfsp_expand_round(h, lb_kind, h->d_in, pieces, h->d_children, h->stream, best, &nc, &ns);
  if (rc != TSB_OK) return rc;
  *n_children = nc;
  *n_solutions = ns;
  if (nc > capacity) return TSB_ENOMEM;
  return h->copy_d2h(children, h->d_children, nc * rec, h->stream);
}

int tsb_pfsp_pool_push(tsb_pfsp* h, const void* nodes, int64_t n) {
  if (!h || n < 0 || (n && !nodes)) return TSB_EINVAL;
  TSB_CUDA(cudaSetDevice(h->device));
  pfsp_pool_setup(h);
  int rc = h->pool.reserve(h->stream, n, pfsp_pool_min_cap(h));
  if (rc != TSB_OK) return rc;
  if (n == 0) return TSB_OK;
  const long long at = h->pool.top();
  rc = h->copy_h2d(h->pool.arena[h->pool.cur] + at * h->rec(), nodes, static_cast<size_t>(n) * h->rec(), h->stream);
  if (rc != TSB_OK) return rc;
  if (h->pool.ext.empty())
    h->pool.ext.push_back({at, at + n});
  else
    h->pool.ext.back().e += n;
  h->pool.size += n;
  return TSB_OK;
}

int64_t tsb_pfsp_pool_size(const tsb_pfsp* h) { return h ? h->pool.size : -1; }

int tsb_pfsp_pool_step(tsb_pfsp* h, int lb_kind, int m, int M, int64_t* best, int64_t* n_parents,
                       uint64_t* n_children, uint64_t* n_solutions) {
  if (!h || lb_kind < 0 || lb_kind > 2 || m < 1 || M < 1 || M > h->M_max || !best || !n_parents || !n_children ||
      !n_solutions)
    return TSB_EINVAL;
  if (lb_kind == TSB_LB2 && h->pairs == 0) return TSB_EINVAL;
  *n_parents = 0;
  *n_children = *n_solutions = 0;
  DevicePool& p = h->pool;
  if (p.size < m) return TSB_OK;  // popBackBulk returns 0 below m (lib/commons/Pool.chpl:50-59)
  TSB_CUDA(cudaSetDevice(h->device));
  const long long n = std::min<long long>(p.size, M);
  std::vector<PoolExtent> pieces;
  pool_top_pieces(p, n, &pieces);
  int rc = TSB_OK;
  if (pieces.size() > tsb::EXP_MAX_PIECES) rc = p.compact(h->stream, p.cap);
  if (rc == TSB_OK) rc = p.reserve(h->stream, n * h->jobs + 2, pfsp_pool_min_cap(h));
  if (rc != TSB_OK) return rc;
  pool_top_pieces(p, n, &pieces);
  // children start on a 16-byte boundary (88-byte records: an even position; 208 = 13 * 16: any position)
  const long long top = h->wide ? p.top() : (p.top() + 1) & ~1LL;
  unsigned long long nc = 0, ns = 0;
  uint8_t* arena = p.arena[p.cur];
  rc = pfsp_expand_round(h, lb_kind, arena, pieces, arena + top * h->rec(), h->stream, best, &nc, &ns,
                         /*early=*/true);
  if (rc != TSB_OK) return rc;
  pool_pop(p, n);
  if (nc) {
    p.ext.push_back({top, top + static_cast<long long>(nc)});
    p.size += static_cast<long long>(nc);
  }
  *n_parents = n;
  *n_children = nc;
  *n_solutions = ns;
  return TSB_OK;
}

int tsb_pfsp_pool_steal(tsb_pfsp* victim, tsb_pfsp* thief, int m, int64_t* n_stolen) {
  if (!victim || !thief || victim == thief || m < 1 || !n_stolen || victim->jobs != thief->jobs) return TSB_EINVAL;
  pfsp_pool_setup(victim);
  pfsp_pool_setup(thief);
  long long n = 0;
  int rc = pool_steal_front(victim->pool, victim->device, victim->stream, thief->pool, thief->device, thief->stream, m,
                            pfsp_pool_min_cap(thief), &n);
  *n_stolen = n;
  return rc;
}

int tsb_pfsp_pool_drain(tsb_pfsp* h, void* nodes, int64_t capacity, int64_t* n) {
  if (!h || !n || capacity < 0) return TSB_EINVAL;
  DevicePool& p = h->pool;
  *n = p.size;
  if (p.size > capacity) return TSB_ENOMEM;
  TSB_CUDA(cudaSetDevice(h->device));
  long long at = 0;
  for (const PoolExtent& x : p.ext) {
    int rc = h->copy_d2h(static_cast<uint8_t*>(nodes) + at * h->rec(), p.arena[p.cur] + x.b * h->rec(),
                         static_cast<size_t>(x.e - x.b) * h->rec(), h->stream);
    if (rc != TSB_OK) return rc;
    at += x.e - x.b;
  }
  p.ext.clear();
  p.size = 0;
  return TSB_OK;
}

}  // extern "C"
