// tsb_host.cpp — host side of libtsb200: the CPU logic the reference keeps in Chapel, restated in
// C++ only because no Chapel compiler exists on the build / bench hosts (SURVEY.md fact 1):
//   * Taillard instance generator and PFSP table precompute (lib/pfsp/Taillard.chpl,
//     fill_* in lib/pfsp/Bound_simple.chpl / Bound_johnson.chpl) -> tsb_pfsp_tables_build
//   * the 3-step search drivers (nqueens_gpu_chpl.chpl, nqueens_multigpu_chpl.chpl,
//     pfsp_gpu_chpl.chpl, pfsp_multigpu_chpl.chpl) with the same Pool contract
//     (lib/commons/Pool.chpl) and the same --m / --M / --D meaning -> tsb_nq_search, tsb_pfsp_search
// The offload step of those drivers calls tsb_*_evaluate, i.e. exactly the C ABI a patched Chapel
// driver would call (INTEGRATION.md).  Nothing here touches the GPU directly and nothing here
// uses oracle/.
#include <algorithm>
#include <chrono>
#include <climits>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <atomic>
#include <condition_variable>
#include <mutex>
#include <thread>
#include <vector>

#include "tsb200.h"

// MAX_JOBS of the build a handle emulates: 20 or 50 (tsb200_api.cu; internal to the library)
__attribute__((visibility("hidden"))) int tsb_pfsp_handle_max_jobs(const tsb_pfsp* h);

namespace {

// ---- Taillard benchmark data (seeds and best-known makespans of ta001..ta120, Taillard 1993;
// the values the reference tabulates in lib/pfsp/Taillard.chpl:3-27, :56-67) ----
const int64_t kSeeds[120] = {
    873654221,  379008056,  1866992158, 216771124,  495070989,  402959317,  1369363414, 2021925980,
    573109518,  88325120,   587595453,  1401007982, 873136276,  268827376,  1634173168, 691823909,
    73807235,   1273398721, 2065119309, 1672900551, 479340445,  268827376,  1958948863, 918272953,
    555010963,  2010851491, 1519833303, 1748670931, 1923497586, 1829909967, 1328042058, 200382020,
    496319842,  1203030903, 1730708564, 450926852,  1303135678, 1273398721, 587288402,  248421594,
    1958948863, 575633267,  655816003,  1977864101, 93805469,   1803345551, 49612559,   1899802599,
    2013025619, 578962478,  1539989115, 691823909,  655816003,  1315102446, 1949668355, 1923497586,
    1805594913, 1861070898, 715643788,  464843328,  896678084,  1179439976, 1122278347, 416756875,
    267829958,  1835213917, 1328833962, 1418570761, 161033112,  304212574,  1539989115, 655816003,
    960914243,  1915696806, 2013025619, 1168140026, 1923497586, 167698528,  1528387973, 993794175,
    450926852,  1462772409, 1021685265, 83696007,   508154254,  1861070898, 26482542,   444956424,
    2115448041, 118254244,  471503978,  1215892992, 135346136,  1602504050, 160037322,  551454346,
    519485142,  383947510,  1968171878, 540872513,  2013025619, 475051709,  914834335,  810642687,
    1019331795, 2056065863, 1342855162, 1325809384, 1988803007, 765656702,  1368624604, 450181436,
    1927888393, 1759567256, 606425239,  19268348,   1298201670, 2041736264, 379756761,  28837162};
const int32_t kBestUb[120] = {
    1278,  1359,  1081,  1293,  1235,  1195,  1234,  1206,  1230,  1108,  1582,  1659,  1496,  1377,  1419,
    1397,  1484,  1538,  1593,  1591,  2297,  2099,  2326,  2223,  2291,  2226,  2273,  2200,  2237,  2178,
    2724,  2834,  2621,  2751,  2863,  2829,  2725,  2683,  2552,  2782,  2991,  2867,  2839,  3063,  2976,
    3006,  3093,  3037,  2897,  3065,  3846,  3699,  3640,  3719,  3610,  3679,  3704,  3691,  3741,  3755,
    5493,  5268,  5175,  5014,  5250,  5135,  5246,  5094,  5448,  5322,  5770,  5349,  5676,  5781,  5467,
    5303,  5595,  5617,  5871,  5845,  6173,  6183,  6252,  6254,  6285,  6331,  6223,  6372,  6247,  6404,
    10862, 10480, 10922, 10889, 10524, 10329, 10854, 10730, 10438, 10675, 11158, 11160, 11281, 11275, 11259,
    11176, 11337, 11301, 11146, 11284, 26040, 26500, 26371, 26456, 26334, 26469, 26389, 26560, 26005, 26457};

double now_s() {
  return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

// growable deque with the reference pool's interface (lib/commons/Pool.chpl:12-73)
template <class Node>
struct Pool {
  std::vector<Node> el;
  size_t front = 0, size = 0;
  Pool() { el.resize(1024); }
  void pushBack(const Node& n) {
    if (front + size >= el.size()) el.resize(el.size() * 2);
    el[front + size] = n;
    ++size;
  }
  bool popBack(Node& n) {
    if (!size) return false;
    n = el[front + --size];
    return true;
  }
  bool popFront(Node& n) {
    if (!size) return false;
    n = el[front++];
    --size;
    return true;
  }
  // Pool.chpl:50-59: nothing below m; otherwise the newest min(size, M) nodes, order preserved
  int popBackBulk(int m, int M, Node* parents) {
    if (size < static_cast<size_t>(m)) return 0;
    const size_t n = std::min(size, static_cast<size_t>(M));
    size -= n;
    std::memcpy(parents, &el[front + size], n * sizeof(Node));
    return static_cast<int>(n);
  }
};

// ------------------------------------------------------------------ N-Queens CPU twin
// isSafe / decompose of the drivers' CPU steps 1 and 3 (nqueens_gpu_chpl.chpl:51-89)
inline bool nq_safe(const tsb_nq_node& p, int depth, int row_pos) {
  for (int i = 0; i < depth; i++) {
    const int d = depth - i, o = p.board[i];
    if (o == row_pos - d || o == row_pos + d) return false;
  }
  return true;
}
void nq_decompose(int N, const tsb_nq_node& parent, uint64_t& tree, uint64_t& sol, Pool<tsb_nq_node>& pool) {
  const int depth = parent.depth;
  if (depth == N) {
    ++sol;
    return;
  }
  for (int j = depth; j < N; j++)
    if (nq_safe(parent, depth, parent.board[j])) {
      tsb_nq_node c = parent;
      c.depth = static_cast<uint8_t>(depth + 1);
      std::swap(c.board[depth], c.board[j]);
      pool.pushBack(c);
      ++tree;
    }
}
// nqueens_gpu_chpl.chpl:126-149
void nq_generate_children(int N, const tsb_nq_node* parents, int size, const uint8_t* labels, uint64_t& tree,
                          uint64_t& sol, Pool<tsb_nq_node>& pool) {
  for (int i = 0; i < size; i++) {
    const tsb_nq_node& parent = parents[i];
    const int depth = parent.depth;
    if (depth == N) {
      ++sol;
      continue;
    }
    const uint8_t* lab = labels + static_cast<size_t>(i) * N;
    for (int j = depth; j < N; j++)
      if (lab[j] == 1) {
        tsb_nq_node c = parent;
        c.depth = static_cast<uint8_t>(depth + 1);
        std::swap(c.board[depth], c.board[j]);
        pool.pushBack(c);
        ++tree;
      }
  }
}

struct GpuTaskResult {
  uint64_t tree = 0, sol = 0, offloads = 0, parents = 0, launches = 0;
  int64_t best = 0;
  int rc = 0;
};

// one GPU task's offload loop (nqueens_gpu_chpl.chpl:197-215; nqueens_multigpu_chpl.chpl:234-253)
inline void bind_task(int device, bool multi) {  // one host thread per GPU: next to its GPU (env TSB200_NO_NUMA=1: no)
  if (multi && !std::getenv("TSB200_NO_NUMA")) (void)tsb_bind_thread_to_device(device);
}

void nq_gpu_task(int device, int N, int g, int m, int M, Pool<tsb_nq_node>& pool, GpuTaskResult& r) {
  tsb_nq* h = nullptr;
  r.rc = tsb_nq_create(&h, device, N, g, M);
  if (r.rc != TSB_OK) return;
  std::vector<tsb_nq_node> parents(M);
  std::vector<uint8_t> labels(static_cast<size_t>(M) * N);
  // the chunk arrays live for the whole step 2 (nqueens_gpu_chpl.chpl:191-192): page-lock them once
  tsb_nq_register_host(h, parents.data(), parents.size() * sizeof(tsb_nq_node));
  tsb_nq_register_host(h, labels.data(), labels.size());
  for (;;) {
    const int n = pool.popBackBulk(m, M, parents.data());
    if (n <= 0) break;
    r.rc = tsb_nq_evaluate(h, parents.data(), n, labels.data());
    if (r.rc != TSB_OK) break;
    ++r.offloads;
    r.parents += static_cast<uint64_t>(n);
    nq_generate_children(N, parents.data(), n, labels.data(), r.tree, r.sol, pool);
  }
  r.launches = tsb_nq_kernel_launches(h);
  tsb_nq_destroy(h);
}

// ---- intra-node work stealing between the tasks' DEVICE pools (the reference steals between its per-GPU host
// pools: nqueens_multigpu_chpl.chpl:255-312, pfsp_multigpu_chpl.chpl:438-495).  A task that runs out of work
// (pool below m) asks the task with the fullest pool; the victim serves the request between two of its launches
// (its pool is on its GPU and only it may touch it while kernels run): the oldest half of its pool moves to the
// thief's GPU over NVLink (tsb_*_pool_steal = popFrontBulkFree, Pool_par.chpl:178-191).  Termination: all tasks
// idle (util.chpl:16-30).  Counts are split-invariant for N-Queens and for PFSP with --ub 1, so stealing changes
// the per-GPU shares, never the totals.
struct StealBoard {
  explicit StealBoard(int D_) : D(D_), size(D_, 0), request(D_, -1), reply(D_, 0), handle(D_, nullptr), failed(false) {}
  const int D;
  std::mutex mu;
  std::condition_variable cv;
  std::vector<long long> size;  // pool size every task last published
  std::vector<int> request;     // request[v] = thief waiting for victim v, or -1
  std::vector<int> reply;       // reply[thief]: 0 pending, 1 granted, -1 denied
  std::vector<void*> handle;    // the tasks' library handles
  bool failed;                  // a task could not create its handle: nobody steals
  int idle = 0;
  bool done = false;
  uint64_t steals = 0;
  // every task's handle exists before anybody steals
  void publish_handle(int me, void* h, long long my_size) {
    std::unique_lock<std::mutex> lk(mu);
    handle[me] = h;
    size[me] = my_size;
    if (!h) failed = true;
    cv.notify_all();
    cv.wait(lk, [&] {
      if (failed) return true;
      for (void* x : handle)
        if (!x) return false;
      return true;
    });
  }
};

// what a device-pool task does between two launches: publish its pool size, serve a pending steal request
// smallest pool worth stealing from: the reference's 2 m (Pool_par.chpl:178-191) for the small chunks of the
// persistent kernel; with large chunks a pool below 2 M is one or two bandwidth-bound rounds of work — splitting
// it costs more (arena reservation on the thief, under-filled launches on both) than it saves: on 8 GPUs the
// N=17 search at M = 4 Mi went from 0.06 s (static split) to 0.18 s when every idle task stole half of such pools
inline long long steal_floor(int m, int M) { return M <= 75776 ? 2LL * m : std::max<long long>(2LL * m, 2LL * M); }

template <class StealFn>
int board_service(StealBoard* sb, int me, long long my_size, long long floor_, StealFn&& steal) {
  if (!sb) return TSB_OK;
  int thief = -1;
  {
    std::lock_guard<std::mutex> lk(sb->mu);
    sb->size[me] = my_size;
    thief = sb->request[me];
    sb->request[me] = -1;
  }
  if (thief < 0) return TSB_OK;
  int64_t got = 0;
  int rc = TSB_OK;
  if (my_size >= floor_ && !sb->failed) rc = steal(sb->handle[me], sb->handle[thief], &got);
  {
    std::lock_guard<std::mutex> lk(sb->mu);
    sb->reply[thief] = (rc == TSB_OK && got > 0) ? 1 : -1;
    sb->size[me] = my_size - got;
    if (got > 0) ++sb->steals;
  }
  sb->cv.notify_all();
  return rc;
}
// out of work: true = stole something (keep going), false = everybody is idle (terminate)
inline bool board_acquire(StealBoard* sb, int me, long long my_size, long long floor_) {
  if (!sb) return false;
  std::unique_lock<std::mutex> lk(sb->mu);
  sb->size[me] = my_size;
  const auto deny_mine = [&] {  // I have nothing to give
    if (sb->request[me] >= 0) {
      sb->reply[sb->request[me]] = -1;
      sb->request[me] = -1;
      sb->cv.notify_all();
    }
  };
  deny_mine();
  ++sb->idle;
  for (;;) {
    if (sb->idle == sb->D) {
      sb->done = true;
      sb->cv.notify_all();
      return false;
    }
    if (sb->done) return false;
    int v = -1;
    for (int i = 0; i < sb->D && !sb->failed; i++)  // the fullest pool nobody is already asking
      if (i != me && sb->request[i] < 0 && sb->size[i] >= floor_ && (v < 0 || sb->size[i] > sb->size[v])) v = i;
    if (v < 0) {
      deny_mine();
      sb->cv.wait_for(lk, std::chrono::microseconds(200));
      continue;
    }
    sb->request[v] = me;
    sb->reply[me] = 0;
    --sb->idle;  // waiting for a victim is not being idle: the victim may hand over half of its pool
    sb->cv.wait(lk, [&] { return sb->reply[me] != 0 || sb->done; });
    if (sb->reply[me] > 0) return true;
    if (sb->done) return false;
    ++sb->idle;
    sb->size[v] = std::min<long long>(sb->size[v], floor_ - 1);  // (it publishes again after its next launch)
  }
}

// a task leaves on an error: nobody may wait for it any more
inline void board_abort(StealBoard* sb, int me) {
  if (!sb) return;
  std::lock_guard<std::mutex> lk(sb->mu);
  sb->failed = sb->done = true;
  if (sb->request[me] >= 0) sb->reply[sb->request[me]] = -1;
  sb->request[me] = -1;
  sb->cv.notify_all();
}

template <class Node>
void static_split(Pool<Node>& pool, int D, std::vector<Pool<Node>>& multi);

// rounds per library call when other tasks may want to steal (a victim serves requests between calls)
inline int64_t rounds_per_call(const StealBoard* sb, int M) { return !sb ? INT64_MAX : M <= 75776 ? 256 : 4; }

// the offload loop with the task's pool resident on the device (tsb_nq_pool_*): all rounds of step 2 inside the
// library (one persistent kernel for small M, two kernels per round otherwise); the host only reads counters
void nq_devpool_rounds(tsb_nq* h, int m, int M, StealBoard* sb, int me, GpuTaskResult& r) {
  const auto steal = [m](void* v, void* t, int64_t* got) {
    return tsb_nq_pool_steal(static_cast<tsb_nq*>(v), static_cast<tsb_nq*>(t), m, got);
  };
  while (r.rc == TSB_OK) {
    uint64_t nr = 0, np = 0, nc = 0, ns = 0;
    r.rc = tsb_nq_pool_run(h, m, M, rounds_per_call(sb, M), &nr, &np, &nc, &ns);
    if (r.rc != TSB_OK) break;
    r.tree += nc;
    r.sol += ns;
    r.offloads += nr;
    r.parents += np;
    const long long size = tsb_nq_pool_size(h);
    if (size >= m) {
      r.rc = board_service(sb, me, size, steal_floor(m, M), steal);
      continue;
    }
    if (!board_acquire(sb, me, size, steal_floor(m, M))) break;
  }
  if (r.rc != TSB_OK) board_abort(sb, me);
}
// Several pools per task (TSB200_POOLS=1 turns it off, =2 caps it at two): for chunks that fit the persistent kernel a
// round is a chain of L2 round trips with ~1 us of work in between, so the task's share of the warm-up pool is split
// once more — the reference's own strided split (static_split) — into P device pools (P = tsb_nq_pools_per_launch: 4
// on a B200 for M <= 56832) whose rounds run in ONE launch (tsb_nq_pool_run_multi), two CTAs of different pools on
// every SM filling each other's waits.  Each pool follows the reference's rule on its own nodes: for D tasks the
// chunk sequence is that of a 2-level split into P D pools, the totals are split-invariant.  A pool of the group
// that runs dry takes the oldest half of the fullest one (as between tasks).
inline int nq_pools_wanted(int M) {  // (decides the warm-up size, before any handle exists)
  int cap = 4;
  if (const char* v = std::getenv("TSB200_POOLS")) cap = std::max(1, std::min(4, std::atoi(v)));
  // the persistent kernel's ranges on 148 SMs: 768 parents x 74 CTAs (four pools), 768 x 98 (three), 512 x 148 (two)
  const int fit = M <= 56832 ? 4 : M <= 75264 ? 3 : M <= 75776 ? 2 : 1;
  return std::min(cap, fit);
}
inline int nq_pools_of(tsb_nq* h, int M) { return std::min(nq_pools_wanted(M), tsb_nq_pools_per_launch(h, M)); }
void nq_devpool_multi_rounds(std::vector<tsb_nq*>& hs, int m, int M, StealBoard* sb, int me, GpuTaskResult& r) {
  const bool no_steal = [] {
    const char* v = std::getenv("TSB200_NO_STEAL");
    return v && *v && *v != '0';
  }();
  const int P = static_cast<int>(hs.size());
  const auto fullest = [&] {
    int v = 0;
    for (int i = 1; i < P; i++)
      if (tsb_nq_pool_size(hs[i]) > tsb_nq_pool_size(hs[v])) v = i;
    return v;
  };
  // a thief task is served from the fullest pool of the group
  const auto steal = [&](void*, void* t, int64_t* got) {
    return tsb_nq_pool_steal(hs[fullest()], static_cast<tsb_nq*>(t), m, got);
  };
  const long long floor_ = steal_floor(m, M);
  std::vector<uint64_t> out(4 * P);
  while (r.rc == TSB_OK) {
    if (!no_steal) {  // balance inside the group: every dry pool takes half of the fullest one
      for (int i = 0; i < P && r.rc == TSB_OK; i++) {
        if (tsb_nq_pool_size(hs[i]) >= m) continue;
        const int v = fullest();
        if (v == i || tsb_nq_pool_size(hs[v]) < floor_) break;
        int64_t got = 0;
        r.rc = tsb_nq_pool_steal(hs[v], hs[i], m, &got);
      }
      if (r.rc != TSB_OK) break;
    }
    long long most = 0, total = 0;
    for (tsb_nq* x : hs) {
      most = std::max<long long>(most, tsb_nq_pool_size(x));
      total += tsb_nq_pool_size(x);
    }
    if (most < m) {
      if (!board_acquire(sb, me, total, floor_)) break;
      continue;
    }
    r.rc = tsb_nq_pool_run_multi(hs.data(), P, m, M, sb ? rounds_per_call(sb, M) : 2048, out.data());
    if (r.rc != TSB_OK) break;
    for (int i = 0; i < P; i++) {
      r.offloads += out[4 * i];
      r.parents += out[4 * i + 1];
      r.tree += out[4 * i + 2];
      r.sol += out[4 * i + 3];
    }
    r.rc = board_service(sb, me, tsb_nq_pool_size(hs[fullest()]), floor_, steal);
  }
  if (r.rc != TSB_OK) board_abort(sb, me);
}
// pool -> device, all rounds, leftovers (fewer than m nodes) back to the host pool for step 3
void nq_devpool_on(tsb_nq* h, int m, int M, Pool<tsb_nq_node>& pool, GpuTaskResult& r, StealBoard* sb = nullptr,
                   int me = 0) {
  const uint64_t l0 = tsb_nq_kernel_launches(h);
  if (const int P = nq_pools_of(h, M); P > 1) {
    std::vector<tsb_nq*> hs{h};
    for (int i = 1; i < P && r.rc == TSB_OK; i++) {
      tsb_nq* sib = nullptr;
      r.rc = tsb_nq_sibling(h, i, &sib);
      hs.push_back(sib);
    }
    std::vector<Pool<tsb_nq_node>> part;
    if (r.rc == TSB_OK) static_split(pool, P, part);
    long long most = 0;
    for (int i = 0; i < P && r.rc == TSB_OK; i++) {
      r.rc = tsb_nq_pool_push(hs[i], &part[i].el[part[i].front], static_cast<int64_t>(part[i].size));
      most = std::max<long long>(most, tsb_nq_pool_size(hs[i]));
    }
    if (sb) sb->publish_handle(me, r.rc == TSB_OK ? h : nullptr, most);
    if (r.rc == TSB_OK) nq_devpool_multi_rounds(hs, m, M, sb, me, r);
    for (tsb_nq* x : hs) {
      if (r.rc != TSB_OK) break;
      const int64_t left = tsb_nq_pool_size(x);
      std::vector<tsb_nq_node> rest(static_cast<size_t>(left) + 1);
      int64_t n = 0;
      r.rc = tsb_nq_pool_drain(x, rest.data(), left, &n);
      for (int64_t i = 0; i < n && r.rc == TSB_OK; i++) pool.pushBack(rest[i]);
    }
    r.launches = tsb_nq_kernel_launches(h) - l0;
    return;
  }
  r.rc = tsb_nq_pool_push(h, &pool.el[pool.front], static_cast<int64_t>(pool.size));
  pool.front = 0;
  pool.size = 0;
  if (sb) sb->publish_handle(me, r.rc == TSB_OK ? h : nullptr, tsb_nq_pool_size(h));
  if (r.rc == TSB_OK) nq_devpool_rounds(h, m, M, sb, me, r);
  if (r.rc == TSB_OK) {
    const int64_t left = tsb_nq_pool_size(h);
    std::vector<tsb_nq_node> rest(static_cast<size_t>(left) + 1);
    int64_t n = 0;
    r.rc = tsb_nq_pool_drain(h, rest.data(), left, &n);
    for (int64_t i = 0; i < n && r.rc == TSB_OK; i++) pool.pushBack(rest[i]);
  }
  r.launches = tsb_nq_kernel_launches(h) - l0;
}
// Handles of the device-pool drivers are kept between searches (per device, N, g, M): a handle with its sibling
// pools, arenas and fat arenas is ~1.4 GB of cudaMalloc / cudaFree per GPU, which at 8 GPUs cost more than the N = 17
// search itself.  (The Chapel drivers declare their device arrays once, outside the search loop, as well.)
// At most two idle handles are kept per device; tsb_release_cached_handles frees them all.
struct NqHandleCache {
  struct Entry {
    int device, N, g, M;
    tsb_nq* h;
  };
  std::mutex mu;
  std::vector<Entry> idle;
  tsb_nq* acquire(int device, int N, int g, int M, int* rc) {
    {
      std::lock_guard<std::mutex> lk(mu);
      for (size_t i = 0; i < idle.size(); i++)
        if (idle[i].device == device && idle[i].N == N && idle[i].g == g && idle[i].M == M) {
          tsb_nq* h = idle[i].h;
          idle.erase(idle.begin() + static_cast<long>(i));
          *rc = TSB_OK;
          return h;
        }
    }
    tsb_nq* h = nullptr;
    *rc = tsb_nq_create(&h, device, N, g, M);
    return *rc == TSB_OK ? h : nullptr;
  }
  void release(tsb_nq* h, int device, int N, int g, int M, bool healthy) {
    if (!h) return;
    if (!healthy || std::getenv("TSB200_NO_HANDLE_CACHE")) {
      tsb_nq_destroy(h);
      return;
    }
    // at most two idle handles per device (a handle with four pools holds ~1.4 GB): the oldest one goes
    tsb_nq* evict = nullptr;
    {
      std::lock_guard<std::mutex> lk(mu);
      idle.push_back({device, N, g, M, h});
      int on_device = 0;
      for (const Entry& e : idle) on_device += e.device == device;
      if (on_device > 2)
        for (size_t i = 0; i < idle.size(); i++)
          if (idle[i].device == device) {
            evict = idle[i].h;
            idle.erase(idle.begin() + static_cast<long>(i));
            break;
          }
    }
    if (evict) tsb_nq_destroy(evict);
  }
  void clear() {
    std::lock_guard<std::mutex> lk(mu);
    for (Entry& e : idle) tsb_nq_destroy(e.h);
    idle.clear();
  }
};
NqHandleCache& nq_handle_cache() {
  static NqHandleCache* c = new NqHandleCache();  // (never destroyed: no CUDA calls at process exit)
  return *c;
}

void nq_devpool_task(int device, int N, int g, int m, int M, Pool<tsb_nq_node>& pool, GpuTaskResult& r,
                     StealBoard* sb = nullptr, int me = 0) {
  tsb_nq* h = nullptr;
  const bool trace = std::getenv("TSB200_TRACE") != nullptr;
  const double tt0 = now_s();
  h = nq_handle_cache().acquire(device, N, g, M, &r.rc);
  if (r.rc != TSB_OK) {
    if (sb) sb->publish_handle(me, nullptr, 0);
    return;
  }
  const double tt1 = now_s();
  nq_devpool_on(h, m, M, pool, r, sb, me);
  const double tt2 = now_s();
  nq_handle_cache().release(h, device, N, g, M, r.rc == TSB_OK);
  if (trace) std::fprintf(stderr, "[tsb200] device %d: create %.1f ms, %llu rounds in %.1f ms, destroy %.1f ms\n", device,
                          (tt1 - tt0) * 1e3, static_cast<unsigned long long>(r.offloads), (tt2 - tt1) * 1e3,
                          (now_s() - tt2) * 1e3);
}

// static strided split of the warm-up pool (nqueens_multigpu_chpl.chpl:199-226)
template <class Node>
void static_split(Pool<Node>& pool, int D, std::vector<Pool<Node>>& multi) {
  const size_t poolSize = pool.size, c = poolSize / D, l = poolSize - (D - 1) * c, f = pool.front;
  multi.resize(D);
  for (int g = 0; g < D; g++) {
    for (size_t i = 0; i < c; i++) multi[g].pushBack(pool.el[g + f + i * D]);
    if (g == D - 1)
      for (size_t i = 0; i < l - c; i++) multi[g].pushBack(pool.el[D * c + f + i]);
  }
  pool.front = 0;
  pool.size = 0;
}

// ------------------------------------------------------------------ PFSP CPU twin
int64_t unif(int64_t& seed, int64_t low, int64_t high) {  // lib/pfsp/Taillard.chpl:72-84
  const int64_t m = 2147483647, a = 16807, b = 127773, c = 2836;
  const int64_t k = seed / b;
  seed = a * (seed % b) - k * c;
  if (seed < 0) seed += m;
  const double v = static_cast<double>(seed) / static_cast<double>(m);
  return low + static_cast<int64_t>(v * static_cast<double>(high - low + 1));
}

// the two builds of the reference: MAX_JOBS = 20 (tsb_pfsp_tables, 88-byte nodes) and MAX_JOBS = 50
// (tsb_pfsp_tables50, 208-byte nodes, ta031..ta060)
template <class Node>
constexpr int max_jobs_of() {
  return static_cast<int>(sizeof(Node::prmu) / sizeof(int32_t));
}
inline int pfsp_tables_for(tsb_pfsp_tables* t, int inst) { return tsb_pfsp_tables_build(t, inst); }
inline int pfsp_tables_for(tsb_pfsp_tables50* t, int inst) { return tsb_pfsp_tables50_build(t, inst, TSB_LB2_FULL); }
inline int pfsp_create_for(tsb_pfsp** h, int device, int M, const tsb_pfsp_tables* t) {
  return tsb_pfsp_create_from_tables(h, device, M, t);
}
inline int pfsp_create_for(tsb_pfsp** h, int device, int M, const tsb_pfsp_tables50* t) {
  return tsb_pfsp_create50_from_tables(h, device, M, t);
}

template <class Tables>
struct HostBounds {  // CPU bounds used by decompose in steps 1 and 3 (pfsp_gpu_chpl.chpl:88-189)
  const Tables& t;
  explicit HostBounds(const Tables& tt) : t(tt) {}
  void front_of(const int32_t* prmu, int limit1, int32_t* F) const {  // schedule_front
    const int N = t.jobs, M = t.machines;
    if (limit1 == -1) {
      for (int j = 0; j < M; j++) F[j] = t.min_heads[j];
      return;
    }
    std::fill(F, F + M, 0);
    for (int i = 0; i <= limit1; i++) {
      const int job = prmu[i];
      F[0] += t.p_times[job];
      for (int j = 1; j < M; j++) F[j] = std::max(F[j - 1], F[j]) + t.p_times[j * N + job];
    }
  }
  void remain_of(const int32_t* prmu, int limit1, int32_t* R) const {  // sum_unscheduled
    const int N = t.jobs, M = t.machines;
    std::fill(R, R + M, 0);
    for (int k = limit1 + 1; k < N; k++)
      for (int j = 0; j < M; j++) R[j] += t.p_times[j * N + prmu[k]];
  }
  int32_t lb1(const int32_t* prmu, int limit1) const {  // lb1_bound
    const int M = t.machines;
    int32_t F[TSB_MAX_MACHINES], R[TSB_MAX_MACHINES];
    front_of(prmu, limit1, F);
    remain_of(prmu, limit1, R);
    int32_t tmp0 = F[0] + R[0], lb = tmp0 + t.min_tails[0];
    for (int i = 1; i < M; i++) {
      const int32_t tmp1 = std::max(tmp0, F[i] + R[i]);
      lb = std::max(lb, tmp1 + t.min_tails[i]);
      tmp0 = tmp1;
    }
    return lb;
  }
  void lb1_children(const int32_t* prmu, int limit1, int32_t* lb_begin) const {  // lb1_children_bounds
    const int N = t.jobs, M = t.machines;
    int32_t F[TSB_MAX_MACHINES], R[TSB_MAX_MACHINES];
    front_of(prmu, limit1, F);
    remain_of(prmu, limit1, R);
    std::fill(lb_begin, lb_begin + N, 0);
    for (int i = limit1 + 1; i < N; i++) {
      const int job = prmu[i];
      int32_t lb = F[0] + R[0] + t.min_tails[0], tmp0 = F[0] + t.p_times[job];
      for (int k = 1; k < M; k++) {
        const int32_t tmp1 = std::max(tmp0, F[k]);
        lb = std::max(lb, tmp1 + R[k] + t.min_tails[k]);
        tmp0 = tmp1 + t.p_times[k * N + job];
      }
      lb_begin[job] = lb;
    }
  }
  int32_t lb2(const int32_t* prmu, int limit1, int64_t best) const {  // lb2_bound
    const int N = t.jobs;
    int32_t F[TSB_MAX_MACHINES];
    front_of(prmu, limit1, F);
    uint64_t sched = 0;  // (64-bit: jobs up to 50)
    for (int j = 0; j <= limit1; j++) sched |= 1ull << prmu[j];
    int32_t lb = 0;
    for (int l = 0; l < t.pairs; l++) {
      const int i = t.mp_order[l], a = t.mp0[i], b = t.mp1[i];
      int32_t t0 = F[a], t1 = F[b];
      for (int j = 0; j < N; j++) {
        const int job = t.johnson[i * N + j];
        if (!((sched >> job) & 1ull)) {
          t0 += t.p_times[a * N + job];
          t1 = std::max(t1, t0 + t.lags[i * N + job]) + t.p_times[b * N + job];
        }
      }
      lb = std::max(lb, std::max(t1 + t.min_tails[b], t0 + t.min_tails[a]));
      if (static_cast<int64_t>(lb) > best) break;
    }
    return lb;
  }
};

template <class Node>
inline void pfsp_child(const Node& parent, int i, Node& c) {
  c = parent;
  c.depth = parent.depth + 1;
  c.limit1 = parent.limit1 + 1;
  std::swap(c.prmu[parent.depth], c.prmu[i]);
}

// decompose (pfsp_gpu_chpl.chpl:88-189)
template <class Tables, class Node>
void pfsp_decompose(const HostBounds<Tables>& hb, int lb_kind, const Node& parent, uint64_t& tree, uint64_t& sol,
                    int64_t& best, Pool<Node>& pool) {
  const int jobs = hb.t.jobs;
  int32_t lb_begin[max_jobs_of<Node>()];
  if (lb_kind == TSB_LB1_D) hb.lb1_children(parent.prmu, parent.limit1, lb_begin);
  for (int i = parent.limit1 + 1; i < jobs; i++) {
    Node c;
    pfsp_child(parent, i, c);
    const int32_t lb = lb_kind == TSB_LB1_D ? lb_begin[parent.prmu[i]]
                       : lb_kind == TSB_LB1 ? hb.lb1(c.prmu, c.limit1)
                                            : hb.lb2(c.prmu, c.limit1, best);
    if (c.depth == jobs) {
      ++sol;
      if (lb < best) best = lb;
    } else if (lb < best) {
      pool.pushBack(c);
      ++tree;
    }
  }
}

// generate_children (pfsp_gpu_chpl.chpl:273-303)
template <class Node>
void pfsp_generate_children(int jobs, const Node* parents, int size, const int32_t* bounds, uint64_t& tree,
                            uint64_t& sol, int64_t& best, Pool<Node>& pool) {
  for (int i = 0; i < size; i++) {
    const Node& parent = parents[i];
    const int depth = parent.depth;
    for (int j = parent.limit1 + 1; j < jobs; j++) {
      const int32_t lb = bounds[j + static_cast<size_t>(i) * jobs];
      if (depth + 1 == jobs) {
        ++sol;
        if (lb < best) best = lb;
      } else if (lb < best) {
        Node c;
        pfsp_child(parent, j, c);
        pool.pushBack(c);
        ++tree;
      }
    }
  }
}

template <class Tables, class Node>
void pfsp_gpu_task(int device, const Tables& t, int lb_kind, int m, int M, Pool<Node>& pool, GpuTaskResult& r) {
  tsb_pfsp* h = nullptr;
  r.rc = pfsp_create_for(&h, device, M, &t);
  if (r.rc != TSB_OK) return;
  const int jobs = t.jobs;
  std::vector<Node> parents(M);
  std::vector<int32_t> bounds(static_cast<size_t>(M) * jobs);
  // the chunk arrays live for the whole step 2 (pfsp_gpu_chpl.chpl:355-356): page-lock them once
  tsb_pfsp_register_host(h, parents.data(), parents.size() * sizeof(Node));
  tsb_pfsp_register_host(h, bounds.data(), bounds.size() * sizeof(int32_t));
  for (;;) {
    const int n = pool.popBackBulk(m, M, parents.data());
    if (n <= 0) break;
    r.rc = tsb_pfsp_evaluate(h, lb_kind, parents.data(), n, r.best, bounds.data());
    if (r.rc != TSB_OK) break;
    ++r.offloads;
    r.parents += static_cast<uint64_t>(n);
    pfsp_generate_children(jobs, parents.data(), n, bounds.data(), r.tree, r.sol, r.best, pool);
  }
  r.launches = tsb_pfsp_kernel_launches(h);
  tsb_pfsp_destroy(h);
}

// the same loop with the task's pool resident on the device (tsb_pfsp_pool_*)
template <class Node>
void pfsp_devpool_on(tsb_pfsp* h, int lb_kind, int m, int M, Pool<Node>& pool, GpuTaskResult& r,
                     StealBoard* sb = nullptr, int me = 0) {
  const uint64_t l0 = tsb_pfsp_kernel_launches(h);
  r.rc = tsb_pfsp_pool_push(h, &pool.el[pool.front], static_cast<int64_t>(pool.size));
  pool.front = 0;
  pool.size = 0;
  if (sb) sb->publish_handle(me, r.rc == TSB_OK ? h : nullptr, tsb_pfsp_pool_size(h));
  const auto steal = [m](void* v, void* t, int64_t* got) {
    return tsb_pfsp_pool_steal(static_cast<tsb_pfsp*>(v), static_cast<tsb_pfsp*>(t), m, got);
  };
  int since_service = 0;
  while (r.rc == TSB_OK) {
    int64_t np = 0;
    uint64_t nc = 0, ns = 0;
    r.rc = tsb_pfsp_pool_step(h, lb_kind, m, M, &r.best, &np, &nc, &ns);
    if (r.rc != TSB_OK) break;
    if (np == 0) {
      if (!board_acquire(sb, me, tsb_pfsp_pool_size(h), steal_floor(m, M))) break;
      continue;
    }
    r.tree += nc;
    r.sol += ns;
    ++r.offloads;
    r.parents += static_cast<uint64_t>(np);
    if (sb && ++since_service >= 2) {  // publish the pool size / serve thieves every other round
      since_service = 0;
      r.rc = board_service(sb, me, tsb_pfsp_pool_size(h), steal_floor(m, M), steal);
    }
  }
  if (r.rc != TSB_OK) board_abort(sb, me);
  if (r.rc == TSB_OK) {
    const int64_t left = tsb_pfsp_pool_size(h);
    std::vector<Node> rest(static_cast<size_t>(left) + 1);
    int64_t n = 0;
    r.rc = tsb_pfsp_pool_drain(h, rest.data(), left, &n);
    for (int64_t i = 0; i < n && r.rc == TSB_OK; i++) pool.pushBack(rest[i]);
  }
  r.launches = tsb_pfsp_kernel_launches(h) - l0;
}
template <class Tables, class Node>
void pfsp_devpool_task(int device, const Tables& t, int lb_kind, int m, int M, Pool<Node>& pool, GpuTaskResult& r,
                       StealBoard* sb = nullptr, int me = 0) {
  tsb_pfsp* h = nullptr;
  r.rc = pfsp_create_for(&h, device, M, &t);
  if (r.rc != TSB_OK) {
    if (sb) sb->publish_handle(me, nullptr, 0);
    return;
  }
  pfsp_devpool_on(h, lb_kind, m, M, pool, r, sb, me);
  tsb_pfsp_destroy(h);
}
template <class Tables, class Node>
void pfsp_gpu_task_nosteal(int device, const Tables& t, int lb_kind, int m, int M, Pool<Node>& pool, GpuTaskResult& r,
                           StealBoard*, int) {
  pfsp_gpu_task(device, t, lb_kind, m, M, pool, r);
}

}  // namespace

// ====================================================================== exported
extern "C" {

int tsb_taillard_nb_jobs(int id) {
  return id > 110 ? 500 : id > 90 ? 200 : id > 60 ? 100 : id > 30 ? 50 : 20;
}
int tsb_taillard_nb_machines(int id) {
  static const int m[12] = {5, 10, 20, 5, 10, 20, 5, 10, 20, 10, 20, 20};  // per group of ten instances
  if (id < 1 || id > 120) return -1;
  return m[(id - 1) / 10];
}
int64_t tsb_taillard_best_ub(int id) { return (id < 1 || id > 120) ? -1 : kBestUb[id - 1]; }

}  // extern "C"
namespace {
// lbound1 / lbound2 of a Taillard instance (pfsp_gpu_chpl.chpl:325-332) into either table struct
template <class T, int MAXJ>
int build_tables(T* t, int inst, int variant) {
  if (!t || inst < 1 || inst > 120 || variant < 0 || variant > 3) return TSB_EINVAL;
  std::memset(t, 0, sizeof(*t));
  const int N = t->jobs = tsb_taillard_nb_jobs(inst);
  const int M = t->machines = tsb_taillard_nb_machines(inst);
  if (N > MAXJ) return TSB_EUNSUPPORTED;  // MAX_JOBS (lib/pfsp/PFSP_node.chpl:7): 20, or 50 for the wide tables
  int64_t seed = kSeeds[inst - 1];
  for (int i = 0; i < M; i++)  // lib/pfsp/Taillard.chpl:86-97
    for (int j = 0; j < N; j++) t->p_times[i * N + j] = static_cast<int32_t>(unif(seed, 1, 99));
  // fill_min_heads_tails, lib/pfsp/Bound_simple.chpl:254-289.  Chapel's line 271 assigns
  // min(max(int(32)), tmp0): min_heads ends as the head times of the LAST job (SURVEY A.1);
  // the Chapel program is the parity target, so that is what is reproduced here.
  t->min_heads[0] = 0;
  {
    int32_t acc = t->p_times[N - 1];
    for (int k = 1; k < M; k++) {
      t->min_heads[k] = acc;
      acc += t->p_times[k * N + (N - 1)];
    }
  }
  for (int k = 0; k < M; k++) t->min_tails[k] = INT32_MAX;
  t->min_tails[M - 1] = 0;
  for (int i = 0; i < N; i++) {
    int32_t acc = t->p_times[(M - 1) * N + i];
    for (int k = M - 2; k >= 0; k--) {
      t->min_tails[k] = std::min(t->min_tails[k], acc);
      acc += t->p_times[k * N + i];
    }
  }
  // fill_machine_pairs (Bound_johnson.chpl:50-87: LB2_FULL / LB2_LEARN = all pairs, the branch the reference
  // compiles; LB2_NABESHIMA = adjacent machines, LB2_LAGEWEG = each machine with the last) + fill_lags (:89-104)
  int c = 0;
  const auto add_pair = [&](int a, int b) {
    t->mp0[c] = a;
    t->mp1[c] = b;
    t->mp_order[c] = c;
    for (int j = 0; j < N; j++) {
      int32_t s = 0;
      for (int k = a + 1; k < b; k++) s += t->p_times[k * N + j];
      t->lags[c * N + j] = s;
    }
    ++c;
  };
  if (variant == TSB_LB2_NABESHIMA) {
    for (int a = 0; a < M - 1; a++) add_pair(a, a + 1);
  } else if (variant == TSB_LB2_LAGEWEG) {
    for (int a = 0; a < M - 1; a++) add_pair(a, M - 1);
  } else {
    for (int a = 0; a < M - 1; a++)
      for (int b = a + 1; b < M; b++) add_pair(a, b);
  }
  t->pairs = c;
  // fill_johnson_schedules (:145-177): Johnson's rule per pair on (p_a + lag, p_b + lag)
  for (int k = 0; k < t->pairs; k++) {
    const int a = t->mp0[k], b = t->mp1[k];
    int order[MAXJ];
    int32_t k1[MAXJ], k2[MAXJ];
    for (int j = 0; j < N; j++) {
      order[j] = j;
      k1[j] = t->p_times[a * N + j] + t->lags[k * N + j];
      k2[j] = t->p_times[b * N + j] + t->lags[k * N + j];
    }
    std::stable_sort(order, order + N, [&](int x, int y) {
      const bool px = k1[x] < k2[x], py = k1[y] < k2[y];  // partition 0 (k1 < k2) first
      if (px != py) return px;
      return px ? k1[x] < k1[y] : k2[x] > k2[y];
    });
    for (int j = 0; j < N; j++) t->johnson[k * N + j] = order[j];
  }
  return TSB_OK;
}
}  // namespace
extern "C" {

int tsb_pfsp_tables_build(tsb_pfsp_tables* t, int inst) { return tsb_pfsp_tables_build_variant(t, inst, TSB_LB2_FULL); }
int tsb_pfsp_tables_build_variant(tsb_pfsp_tables* t, int inst, int variant) {
  return build_tables<tsb_pfsp_tables, TSB_MAX_JOBS>(t, inst, variant);
}
int tsb_pfsp_tables50_build(tsb_pfsp_tables50* t, int inst, int variant) {
  return build_tables<tsb_pfsp_tables50, TSB_MAX_JOBS_WIDE>(t, inst, variant);
}
int tsb_pfsp_create50_from_tables(tsb_pfsp** h, int device, int M_max, const tsb_pfsp_tables50* t) {
  if (!t) return TSB_EINVAL;
  return tsb_pfsp_create_wide(h, device, TSB_MAX_JOBS_WIDE, t->jobs, t->machines, M_max, t->p_times, t->min_heads,
                              t->min_tails, t->pairs, t->johnson, t->lags, t->mp0, t->mp1, t->mp_order);
}

int tsb_pfsp_create_from_tables(tsb_pfsp** h, int device, int M_max, const tsb_pfsp_tables* t) {
  if (!t) return TSB_EINVAL;
  return tsb_pfsp_create(h, device, t->jobs, t->machines, M_max, t->p_times, t->min_heads, t->min_tails,
                         t->pairs, t->johnson, t->lags, t->mp0, t->mp1, t->mp_order);
}

int tsb_nq_search(int N, int g, int m, int M, int D, tsb_search_stats* out) {
  if (!out || N < 1 || N > TSB_MAX_QUEENS || g < 1 || m < 1 || M < 1 || D < 1 || D > 8) return TSB_EINVAL;
  std::memset(out, 0, sizeof(*out));
  if (int rc = tsb_init_devices(D); rc != TSB_OK) return rc;  // contexts exist before the timers start
  Pool<tsb_nq_node> pool;
  tsb_nq_node root{};
  for (int i = 0; i < N; i++) root.board[i] = static_cast<uint8_t>(i);
  pool.pushBack(root);
  uint64_t tree = 0, sol = 0;
  tsb_nq_node parent;
  double t0 = now_s();
  while (pool.size < static_cast<size_t>(D) * m) {  // step 1 (nqueens_multigpu_chpl.chpl:173-179)
    if (!pool.popFront(parent)) break;
    nq_decompose(N, parent, tree, sol, pool);
  }
  double t1 = now_s();
  out->t_step1 = t1 - t0;
  std::vector<GpuTaskResult> res(D);  // step 2
  // task g drives GPU g; with fewer than D GPUs present the tasks wrap around (g % ndev): the
  // per-task pools stay independent, so counts are unchanged — used to test D > 1 on one GPU
  const int ndev = std::max(1, tsb_device_count());
  if (D == 1) {
    nq_gpu_task(0, N, g, m, M, pool, res[0]);
  } else {
    std::vector<Pool<tsb_nq_node>> multi;
    static_split(pool, D, multi);
    std::vector<std::thread> th;
    for (int gid = 0; gid < D; gid++)
      th.emplace_back([&, gid] {
        bind_task(gid % ndev, true);
        nq_gpu_task(gid % ndev, N, g, m, M, multi[gid], res[gid]);
      });
    for (auto& x : th) x.join();
    for (int gid = 0; gid < D; gid++)  // leftovers back to the global pool (:315-320)
      while (multi[gid].popBack(parent)) pool.pushBack(parent);
  }
  for (int gid = 0; gid < D; gid++) {
    if (res[gid].rc != TSB_OK) return res[gid].rc;
    tree += res[gid].tree;
    sol += res[gid].sol;
    out->offloads += res[gid].offloads;
    out->offloaded_parents += res[gid].parents;
    out->kernel_launches += res[gid].launches;
    out->per_gpu_tree[gid] = res[gid].tree;
  }
  double t2 = now_s();
  out->t_step2 = t2 - t1;
  while (pool.popBack(parent)) nq_decompose(N, parent, tree, sol, pool);  // step 3
  out->t_step3 = now_s() - t2;
  out->explored_tree = tree;
  out->explored_sol = sol;
  return TSB_OK;
}

// part < 0: the whole search.  part >= 0: only task `part` of the D-way static split, on `device` (one rank of a
// process-per-GPU launch): the step-1 tree is credited to part 0 and every part drains its own leftovers, so the
// per-part counts add up to the whole search's.  `on` != nullptr: D = 1 on a handle the caller created (set-up
// outside the search's timers, as the Chapel drivers' `on device var` declarations are).
static int nq_search_device_impl(int N, int g, int m, int M, int D, int part, int device, tsb_nq* on,
                                 tsb_search_stats* out) {
  if (!out || N < 1 || N > TSB_MAX_QUEENS || g < 1 || m < 1 || M < 1 || D < 1 || D > 8 || part >= D) return TSB_EINVAL;
  std::memset(out, 0, sizeof(*out));
  if (!on)
    if (int rc = tsb_init_devices(part < 0 ? D : device + 1); rc != TSB_OK) return rc;
  Pool<tsb_nq_node> pool;
  tsb_nq_node root{};
  for (int i = 0; i < N; i++) root.board[i] = static_cast<uint8_t>(i);
  pool.pushBack(root);
  uint64_t tree = 0, sol = 0;
  tsb_nq_node parent;
  double t0 = now_s();
  // step 1 on the CPU, as in the reference: m nodes for every pool (two per task in pair mode, see nq_pair_mode)
  while (pool.size < static_cast<size_t>(D) * m * nq_pools_wanted(M)) {
    if (!pool.popFront(parent)) break;
    nq_decompose(N, parent, tree, sol, pool);
  }
  double t1 = now_s();
  out->t_step1 = t1 - t0;
  // step 2: every task's pool moves to its device and stays there (same static split as tsb_nq_search); tasks
  // that run dry steal from the fullest device pool over NVLink
  std::vector<GpuTaskResult> res(D);
  const int ndev = std::max(1, tsb_device_count());
  if (on) {
    nq_devpool_on(on, m, M, pool, res[0]);
  } else if (part >= 0) {
    if (part != 0) tree = sol = 0;  // step 1 is credited to part 0
    std::vector<Pool<tsb_nq_node>> multi;
    if (D == 1) {
      multi.resize(1);
      std::swap(multi[0], pool);
    } else {
      static_split(pool, D, multi);
    }
    nq_devpool_task(device, N, g, m, M, multi[part], res[part]);
    while (multi[part].popBack(parent)) pool.pushBack(parent);
  } else if (D == 1) {
    nq_devpool_task(0, N, g, m, M, pool, res[0]);
  } else {
    std::vector<Pool<tsb_nq_node>> multi;
    static_split(pool, D, multi);
    StealBoard board(D);
    StealBoard* sb = std::getenv("TSB200_NO_STEAL") ? nullptr : &board;
    std::vector<std::thread> th;
    for (int gid = 0; gid < D; gid++)
      th.emplace_back([&, gid] {
        bind_task(gid % ndev, true);
        nq_devpool_task(gid % ndev, N, g, m, M, multi[gid], res[gid], sb, gid);
      });
    for (auto& x : th) x.join();
    for (int gid = 0; gid < D; gid++)
      while (multi[gid].popBack(parent)) pool.pushBack(parent);
    out->steals = board.steals;
  }
  for (int gid = 0; gid < D; gid++) {
    if (res[gid].rc != TSB_OK) return res[gid].rc;
    tree += res[gid].tree;
    sol += res[gid].sol;
    out->offloads += res[gid].offloads;
    out->offloaded_parents += res[gid].parents;
    out->kernel_launches += res[gid].launches;
    out->per_gpu_tree[gid] = res[gid].tree;
  }
  double t2 = now_s();
  out->t_step2 = t2 - t1;
  while (pool.popBack(parent)) nq_decompose(N, parent, tree, sol, pool);  // step 3
  out->t_step3 = now_s() - t2;
  out->explored_tree = tree;
  out->explored_sol = sol;
  return TSB_OK;
}

}  // extern "C"

// Tables / Node: the build of the reference the search emulates (tsb_pfsp_tables + tsb_pfsp_node: MAX_JOBS = 20;
// tsb_pfsp_tables50 + tsb_pfsp_node50: MAX_JOBS = 50)
template <class Tables, class Node>
static int pfsp_search_impl(int inst, int lb_kind, int ub, int m, int M, int D, bool devpool, int part, int device,
                            tsb_pfsp* on, tsb_search_stats* out) {
  if (!out || lb_kind < 0 || lb_kind > 2 || (ub != 0 && ub != 1) || m < 1 || M < 1 || D < 1 || D > 8 || part >= D)
    return TSB_EINVAL;
  std::memset(out, 0, sizeof(*out));
  std::vector<Tables> tv(1);
  Tables& t = tv[0];
  int rc = pfsp_tables_for(&t, inst);
  if (rc != TSB_OK) return rc;
  if (!on)
    if (rc = tsb_init_devices(part < 0 ? D : device + 1); rc != TSB_OK) return rc;  // contexts exist before the timers start
  HostBounds<Tables> hb(t);
  int64_t best = ub == 1 ? tsb_taillard_best_ub(inst) : INT64_MAX;  // pfsp_gpu_chpl.chpl:37
  Pool<Node> pool;
  Node root{};
  root.limit1 = -1;
  for (int i = 0; i < t.jobs; i++) root.prmu[i] = i;
  pool.pushBack(root);
  uint64_t tree = 0, sol = 0;
  Node parent;
  double t0 = now_s();
  while (pool.size < static_cast<size_t>(D) * m) {
    if (!pool.popFront(parent)) break;
    pfsp_decompose(hb, lb_kind, parent, tree, sol, best, pool);
  }
  double t1 = now_s();
  out->t_step1 = t1 - t0;
  std::vector<GpuTaskResult> res(D);
  const int ndev = std::max(1, tsb_device_count());
  for (auto& r : res) r.best = best;  // per-task best_l = best (pfsp_multigpu_chpl.chpl:384)
  auto task = devpool ? pfsp_devpool_task<Tables, Node> : pfsp_gpu_task_nosteal<Tables, Node>;
  if (on) {
    pfsp_devpool_on(on, lb_kind, m, M, pool, res[0]);
  } else if (part >= 0) {  // one task of the split (see nq_search_device_impl)
    if (part != 0) tree = sol = 0;
    std::vector<Pool<Node>> multi;
    if (D == 1) {
      multi.resize(1);
      std::swap(multi[0], pool);
    } else {
      static_split(pool, D, multi);
    }
    task(device, t, lb_kind, m, M, multi[part], res[part], nullptr, 0);
    while (multi[part].popBack(parent)) pool.pushBack(parent);
  } else if (D == 1) {
    task(0, t, lb_kind, m, M, pool, res[0], nullptr, 0);
  } else {
    std::vector<Pool<Node>> multi;
    static_split(pool, D, multi);
    StealBoard board(D);
    // (stealing keeps the counts only when `best` is constant: --ub 1, SURVEY A.6)
    StealBoard* sb = (devpool && ub == 1 && !std::getenv("TSB200_NO_STEAL")) ? &board : nullptr;
    std::vector<std::thread> th;
    for (int gid = 0; gid < D; gid++)
      th.emplace_back([&, gid] {
        bind_task(gid % ndev, true);
        task(gid % ndev, t, lb_kind, m, M, multi[gid], res[gid], sb, gid);
      });
    for (auto& x : th) x.join();
    for (int gid = 0; gid < D; gid++)
      while (multi[gid].popBack(parent)) pool.pushBack(parent);
    out->steals = board.steals;
  }
  for (int gid = 0; gid < D; gid++) {
    if (res[gid].rc != TSB_OK) return res[gid].rc;
    tree += res[gid].tree;
    sol += res[gid].sol;
    best = std::min(best, res[gid].best);  // min reduce (pfsp_multigpu_chpl.chpl:520)
    out->offloads += res[gid].offloads;
    out->offloaded_parents += res[gid].parents;
    out->kernel_launches += res[gid].launches;
    out->per_gpu_tree[gid] = res[gid].tree;
  }
  double t2 = now_s();
  out->t_step2 = t2 - t1;
  while (pool.popBack(parent)) pfsp_decompose(hb, lb_kind, parent, tree, sol, best, pool);
  out->t_step3 = now_s() - t2;
  out->explored_tree = tree;
  out->explored_sol = sol;
  out->best = best;
  return TSB_OK;
}

extern "C" {

// step 1 of the drivers alone (nqueens_gpu_chpl.chpl:169-175): breadth-first from the root until the pool holds
// min_size nodes; the pool, in order, and what was explored on the way
void tsb_release_cached_handles(void) { nq_handle_cache().clear(); }

int tsb_nq_warmup(int N, int min_size, void* nodes, int64_t capacity, int64_t* n, uint64_t* tree, uint64_t* sol) {
  if (N < 1 || N > TSB_MAX_QUEENS || min_size < 1 || !n || !tree || !sol || (capacity && !nodes)) return TSB_EINVAL;
  Pool<tsb_nq_node> pool;
  tsb_nq_node root{}, parent;
  for (int i = 0; i < N; i++) root.board[i] = static_cast<uint8_t>(i);
  pool.pushBack(root);
  *tree = *sol = 0;
  while (pool.size < static_cast<size_t>(min_size)) {
    if (!pool.popFront(parent)) break;
    nq_decompose(N, parent, *tree, *sol, pool);
  }
  *n = static_cast<int64_t>(pool.size);
  if (*n > capacity) return TSB_ENOMEM;
  if (pool.size) std::memcpy(nodes, &pool.el[pool.front], pool.size * sizeof(tsb_nq_node));
  return TSB_OK;
}

int tsb_nq_search_device(int N, int g, int m, int M, int D, tsb_search_stats* out) {
  return nq_search_device_impl(N, g, m, M, D, -1, 0, nullptr, out);
}
int tsb_nq_search_device_part(int N, int g, int m, int M, int D, int part, int device, tsb_search_stats* out) {
  if (part < 0) return TSB_EINVAL;
  return nq_search_device_impl(N, g, m, M, D, part, device, nullptr, out);
}
int tsb_nq_search_on(tsb_nq* h, int N, int m, int M, tsb_search_stats* out) {
  if (!h) return TSB_EINVAL;
  return nq_search_device_impl(N, 1, m, M, 1, -1, 0, h, out);
}
int tsb_pfsp_search(int inst, int lb_kind, int ub, int m, int M, int D, tsb_search_stats* out) {
  return pfsp_search_impl<tsb_pfsp_tables, tsb_pfsp_node>(inst, lb_kind, ub, m, M, D, false, -1, 0, nullptr, out);
}
int tsb_pfsp_search_device(int inst, int lb_kind, int ub, int m, int M, int D, tsb_search_stats* out) {
  return pfsp_search_impl<tsb_pfsp_tables, tsb_pfsp_node>(inst, lb_kind, ub, m, M, D, true, -1, 0, nullptr, out);
}
int tsb_pfsp_search_device_part(int inst, int lb_kind, int ub, int m, int M, int D, int part, int device,
                                tsb_search_stats* out) {
  if (part < 0) return TSB_EINVAL;
  return pfsp_search_impl<tsb_pfsp_tables, tsb_pfsp_node>(inst, lb_kind, ub, m, M, D, true, part, device, nullptr, out);
}
int tsb_pfsp_search_on(tsb_pfsp* h, int inst, int lb_kind, int ub, int m, int M, tsb_search_stats* out) {
  if (!h) return TSB_EINVAL;
  if (tsb_pfsp_handle_max_jobs(h) == TSB_MAX_JOBS_WIDE) {
    if (inst < 1 || inst > 120) return TSB_EINVAL;
    if (tsb_taillard_nb_jobs(inst) != TSB_MAX_JOBS_WIDE) return TSB_EUNSUPPORTED;  // the handle's build takes 50 jobs
    return pfsp_search_impl<tsb_pfsp_tables50, tsb_pfsp_node50>(inst, lb_kind, ub, m, M, 1, true, -1, 0, h, out);
  }
  return pfsp_search_impl<tsb_pfsp_tables, tsb_pfsp_node>(inst, lb_kind, ub, m, M, 1, true, -1, 0, h, out);
}

// the search as a build of the reference with MAX_JOBS = max_jobs runs it: 20 = tsb_pfsp_search[_device]; 50 =
// 208-byte nodes, ta031..ta060.  Everything is validated before any device is touched.
static int pfsp_search_wide(int max_jobs, int inst, int lb_kind, int ub, int m, int M, int D, bool devpool,
                            tsb_search_stats* out) {
  if (max_jobs == TSB_MAX_JOBS)
    return pfsp_search_impl<tsb_pfsp_tables, tsb_pfsp_node>(inst, lb_kind, ub, m, M, D, devpool, -1, 0, nullptr, out);
  if (max_jobs != TSB_MAX_JOBS_WIDE) return TSB_EUNSUPPORTED;
  if (inst < 1 || inst > 120) return TSB_EINVAL;
  if (tsb_taillard_nb_jobs(inst) != TSB_MAX_JOBS_WIDE) return TSB_EUNSUPPORTED;  // (jobs == MAX_JOBS, as for handles)
  return pfsp_search_impl<tsb_pfsp_tables50, tsb_pfsp_node50>(inst, lb_kind, ub, m, M, D, devpool, -1, 0, nullptr, out);
}
int tsb_pfsp_search_wide(int max_jobs, int inst, int lb_kind, int ub, int m, int M, int D, tsb_search_stats* out) {
  return pfsp_search_wide(max_jobs, inst, lb_kind, ub, m, M, D, false, out);
}
int tsb_pfsp_search_device_wide(int max_jobs, int inst, int lb_kind, int ub, int m, int M, int D,
                                tsb_search_stats* out) {
  return pfsp_search_wide(max_jobs, inst, lb_kind, ub, m, M, D, true, out);
}

}  // extern "C"
