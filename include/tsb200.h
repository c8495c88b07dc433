/*
 * tsb200.h — C ABI of libtsb200.so, the B200-native (sm_100a) batch node-evaluation engine.
 *
 * Drop-in boundary for the GPU offload step of the reference's Chapel drivers
 * (Guillaume-Helbecque/GPU-accelerated-tree-search-Chapel).  Paths below are relative to the
 * reference root.  Every entry point takes plain pointers and sizes, returns an int status
 * (0 = TSB_OK, negative = TSB_E*), never throws, never calls exit(), and calls
 * cudaSetDevice(handle->device) first (Chapel tasks share OS worker threads).
 *
 * One handle per (task, device); distinct handles are fully concurrent, a handle is not
 * re-entrant.  The library owns all device and pinned staging memory; caller pointers are
 * never retained past return.  A caller that keeps its chunk arrays for the whole search (the
 * Chapel drivers allocate `parents` / `labels` once, nqueens_gpu_chpl.chpl:191-192) may hand them
 * to tsb_*_register_host(): the range is page-locked + mapped (cudaHostRegister) and
 * tsb_*_evaluate then works on it in place (zero-copy over PCIe).  Registration is explicit and
 * the caller owns the lifetime: a registered array must stay allocated until it is unregistered
 * or the handle is destroyed.  Arrays that were never registered go through the handle's pinned
 * staging buffers.  (env TSB200_NO_REGISTER=1 turns registration into a no-op.)
 *
 * Node wire formats (must match the Chapel records bit for bit):
 *   N-Queens  lib/nqueens/NQueens_node.chpl:9-11   { uint8 depth; uint8 board[20]; }   21 B, align 1
 *   PFSP      lib/pfsp/PFSP_node.chpl:9-12         { int32 depth; int32 limit1; int32 prmu[20]; } 88 B
 *
 * Output contract (same as the reference kernels): only slots k >= depth (N-Queens) /
 * k >= limit1+1 (PFSP) are defined; the slots below the live range are unspecified (the reference
 * leaves them stale and its consumer never reads them, nqueens_gpu_chpl.chpl:137-138,
 * pfsp_gpu_chpl.chpl:280-281).  N-Queens boards must hold values < 32 (they are permutations
 * of 0..N-1 in every node the drivers create, lib/nqueens/NQueens_node.chpl:17-20).
 */
#ifndef TSB200_H
#define TSB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TSB_MAX_QUEENS 20
#define TSB_MAX_JOBS 20
#define TSB_MAX_MACHINES 20
#define TSB_MAX_PAIRS 190
#define TSB_MAX_JOBS_WIDE 50 /* the reference built with `-sMAX_JOBS=50` (lib/pfsp/PFSP_node.chpl:7): ta031..ta060 */

typedef struct {
  uint8_t depth;
  uint8_t board[TSB_MAX_QUEENS];
} tsb_nq_node; /* 21 bytes */

typedef struct {
  int32_t depth;
  int32_t limit1;
  int32_t prmu[TSB_MAX_JOBS];
} tsb_pfsp_node; /* 88 bytes */

typedef struct {
  int32_t depth;
  int32_t limit1;
  int32_t prmu[TSB_MAX_JOBS_WIDE];
} tsb_pfsp_node50; /* 208 bytes: PFSP Node of a MAX_JOBS = 50 build */

enum {
  TSB_OK = 0,
  TSB_EINVAL = -1,   /* bad argument (NULL handle, N out of 1..20, count > M_max, unknown lb_kind ...) */
  TSB_ECUDA = -2,    /* a CUDA runtime call failed; tsb_last_cuda_error() has the text */
  TSB_ENOMEM = -3,   /* host or device allocation failed */
  TSB_ENODEV = -4,   /* no such CUDA device / no CUDA driver */
  TSB_EALIGN = -5,   /* device pointer passed to *_evaluate_device is not 16-byte aligned */
  TSB_EUNSUPPORTED = -6 /* instance shape outside jobs <= 20, machines in 1..20 */
};

/* lower-bound selector: integer encoding of baselines/pfsp/pfsp_c.c:86-88 and
 * baselines/pfsp/lib/evaluate.cu:93-115 (Chapel spells them "lb1_d" | "lb1" | "lb2",
 * pfsp_gpu_chpl.chpl:15,257-270) */
enum { TSB_LB1_D = 0, TSB_LB1 = 1, TSB_LB2 = 2 };

/* host<->device transfer strategy of the host-buffer entry points */
enum {
  TSB_XFER_AUTO = 0,    /* pick per call (default; env TSB200_XFER=memcpy|zerocopy overrides) */
  TSB_XFER_MEMCPY = 1,  /* cudaMemcpyAsync of the live prefix, kernel, cudaMemcpyAsync back */
  TSB_XFER_ZEROCOPY = 2 /* the kernel's TMA engine reads/writes page-locked host memory over PCIe */
};

const char* tsb_strerror(int code);
const char* tsb_last_cuda_error(void); /* thread-local text of the last failing CUDA call */
int tsb_device_count(void);            /* >= 0, or TSB_ENODEV */
/* create the CUDA context of devices 0..n-1 now (the Chapel runtime does this at program start); the
 * emulation drivers call it before starting their timers */
int tsb_init_devices(int n);
/* pin the CALLING host thread to the CPU cores local to `device` (its PCI function's NUMA node), so that the
 * arrays the thread allocates afterwards and the library's staging buffers sit next to the GPU they feed: call it
 * at the top of every per-GPU task (Chapel: first statement inside the `coforall gpuID`, with one qthreads worker
 * per task).  Returns the number of cores (> 0), TSB_EUNSUPPORTED where sysfs does not tell, TSB_ENODEV. */
int tsb_bind_thread_to_device(int device);
const char* tsb_version(void);

/* ------------------------------------------------------------------ N-Queens ------------- */
typedef struct tsb_nq tsb_nq;

/* Replaces the `on device var parents_d, labels_d` declarations, nqueens_gpu_chpl.chpl:194-195
 * (multi-GPU: nqueens_multigpu_chpl.chpl:231-232).  N in 1..20, g >= 1 (results do not depend
 * on g: the reference's inner `for _g` loop ANDs the same boolean g times, :115-118),
 * M_max = the driver's --M (largest chunk). */
int tsb_nq_create(tsb_nq** h, int device, int N, int g, int M_max);
void tsb_nq_destroy(tsb_nq* h);

/* Replaces the three statements of one offload round, nqueens_gpu_chpl.chpl:203-205
 *   parents_d = parents;  on device do evaluate_gpu(parents_d, N*count, labels_d);  labels = labels_d;
 * parents: count x 21 B host records; labels: count x N host bytes, labels[p*N + k] = 1 iff the
 * queen board[k] can be placed on row `depth` (evaluate_gpu, nqueens_gpu_chpl.chpl:97-123).
 * Synchronous; count == 0 is a no-op; only the live prefix moves (unlike Chapel's whole-array copy). */
int tsb_nq_evaluate(tsb_nq* h, const void* parents, int count, uint8_t* labels);

/* Device-resident form: evaluate_gpu itself (nqueens_gpu_chpl.chpl:97-123) on caller-owned device
 * arrays (16-byte aligned), asynchronous on `stream` (a cudaStream_t; NULL = the handle's own
 * stream).  count is not limited by M_max. */
int tsb_nq_evaluate_device(tsb_nq* h, const void* parents_d, int count, uint8_t* labels_d, void* stream);

/* ---- beyond the drop-in: fused evaluate + generate_children on the device (SURVEY §8f row 1) ----
 * evaluate_gpu (nqueens_gpu_chpl.chpl:97-123) followed by generate_children (:126-149) in one call: the
 * children of the chunk come back packed, in the reference's order (parents in order, slots j ascending);
 * *n_solutions = parents with depth == N.  `children` must hold count*N nodes in the worst case; if it is
 * smaller than the actual number, TSB_ENOMEM is returned with the counts set.  Synchronous. */
int tsb_nq_expand(tsb_nq* h, const void* parents, int count, void* children, uint64_t capacity_nodes,
                  uint64_t* n_children, uint64_t* n_solutions);
int tsb_nq_expand_device(tsb_nq* h, const void* parents_d /*16-B aligned*/, int count,
                         void* children_d /*any alignment*/, uint64_t* n_children, uint64_t* n_solutions,
                         void* stream);

/* ---- device-resident pool (SURVEY §8f row 3): the reference's SinglePool (lib/commons/Pool.chpl) kept in
 * HBM.  push = pushBack of host nodes; step = one offload round of nqueens_gpu_chpl.chpl:197-215 done
 * entirely on the device (two kernels: count + build): popBackBulk(m, M) (nothing below m, else the newest min(size, M)
 * nodes, order preserved, read in place), evaluate, generate_children appended to the pool; drain = move what
 * is left to the host (logical order).  The pool's logical content after every round is byte-identical to
 * the reference's host pool. */
int tsb_nq_pool_push(tsb_nq* h, const void* nodes, int64_t n);
int64_t tsb_nq_pool_size(const tsb_nq* h);
int tsb_nq_pool_step(tsb_nq* h, int m, int M, int64_t* n_parents, uint64_t* n_children, uint64_t* n_solutions);
int tsb_nq_pool_drain(tsb_nq* h, void* nodes, int64_t capacity_nodes, int64_t* n);
/* rounds until the pool holds fewer than m nodes (or max_rounds are done): exactly the sequence of
 * tsb_nq_pool_step rounds — the same chunks, the same pool after every round — but for chunk sizes up to
 * 512 x #SMs (the reference's default --M 50000) the whole loop of nqueens_gpu_chpl.chpl:197-215 runs inside ONE
 * persistent cooperative kernel (two flag exchanges through L2 per round instead of two launches and a host
 * round trip); larger M falls back to one tsb_nq_pool_step per round.  Totals over the rounds come back. */
/* work stealing between two device pools (the reference steals between its per-GPU host pools,
 * nqueens_multigpu_chpl.chpl:255-312): if the victim holds >= 2 m nodes, the oldest size / 2 of them
 * (popFrontBulkFree, lib/commons/Pool_par.chpl:178-191) move to the top of the thief's pool, device to device
 * (NVLink between two GPUs).  No round may be in flight on either handle; the caller serialises the two. */
int tsb_nq_pool_steal(tsb_nq* victim, tsb_nq* thief, int m, int64_t* n_stolen);
int tsb_nq_pool_run(tsb_nq* h, int m, int M, int64_t max_rounds, uint64_t* n_rounds, uint64_t* n_parents,
                    uint64_t* n_children, uint64_t* n_solutions);

/* The same for up to 4 INDEPENDENT pools (handles on one device, same N) served by ONE launch of the persistent
 * kernel: the CTAs of pool i run pool i's rounds and never look at another pool; with two pools every SM hosts one CTA
 * of each and the L2 round trips that order one pool's rounds (count exchange, store -> poll) are filled with the
 * other pool's work.  Each pool follows, on its own nodes, exactly the sequence tsb_nq_pool_run produces — this is the
 * reference's multi-GPU static split (nqueens_multigpu_chpl.chpl:200-224: D tasks, D pools) with several of the D
 * pools living on one GPU.  out[4 i .. 4 i + 3] = {rounds, parents, children, solutions} of pool i.  Chunks too large
 * for the persistent kernel: the pools are run one after the other. */
int tsb_nq_pool_run_multi(tsb_nq* const* handles, int n_pools, int m, int M, int64_t max_rounds, uint64_t* out);
/* Further independent pools on the same device (index 1..3), created on first use and owned by `h` (destroyed with
 * it; their launches are included in h's tsb_nq_kernel_launches count): what a driver groups with `h` in
 * tsb_nq_pool_run_multi. */
int tsb_nq_sibling(tsb_nq* h, int index, tsb_nq** sibling);
/* How many pools one launch of the persistent kernel serves best for chunks of up to M parents on h's device: 4
 * (74 CTAs of 768 parents per pool on a B200), 2 (148 + 148 CTAs of 512), or 1 (M beyond the persistent kernel). */
int tsb_nq_pools_per_launch(const tsb_nq* h, int M);

/* page-lock + map a caller-owned host array for the lifetime of the handle (see the header comment);
 * TSB_EINVAL if the range partly overlaps a registered one / was not registered */
int tsb_nq_register_host(tsb_nq* h, void* ptr, size_t bytes);
int tsb_nq_unregister_host(tsb_nq* h, void* ptr);
int tsb_nq_set_xfer(tsb_nq* h, int mode);
uint64_t tsb_nq_kernel_launches(const tsb_nq* h); /* kernels launched through this handle so far */
void* tsb_nq_stream(const tsb_nq* h); /* the handle's cudaStream_t: the pool / expand / host-buffer entry points launch
                                        * on it (to bracket them with CUDA events) */

/* diagnostics: SM cycles per round of the bare two-flag-exchange skeleton of the persistent multi-round kernel
 * (no evaluation, no children) — the floor under a round of tsb_nq_pool_run; variant bits: 1 = no release fence,
 * 2 = no acquire fence, 4 = 16 bytes per thread stored before the release, 8 = weak L2 polls, 16 = one exchange */
int tsb_debug_flag_exchange(int device, int rounds, int variant, int ctas /* 0 = one per SM */, double* cycles_per_round);

/* ------------------------------------------------------------------ PFSP ----------------- */
typedef struct tsb_pfsp tsb_pfsp;

/* Replaces the device table set-up pfsp_gpu_chpl.chpl:359-371 (lbound1_d / lbound2_d); all
 * tables are copied.  Layouts as in lb1_bound_data (lib/pfsp/Bound_simple.chpl:6-27) and
 * lb2_bound_data (lib/pfsp/Bound_johnson.chpl:11-48):
 *   p_times[machines*jobs] machine-major (k*jobs + job); min_heads/min_tails[machines];
 *   johnson[nb_pairs*jobs], lags[nb_pairs*jobs]; mp0/mp1/mp_order[nb_pairs].
 * jobs <= 20 (the reference's MAX_JOBS), machines <= 20, nb_pairs <= 190. */
int tsb_pfsp_create(tsb_pfsp** h, int device, int jobs, int machines, int M_max, const int32_t* p_times,
                    const int32_t* min_heads, const int32_t* min_tails, int nb_pairs,
                    const int32_t* johnson, const int32_t* lags, const int32_t* mp0, const int32_t* mp1,
                    const int32_t* mp_order);
/* SURVEY §8(f4): the reference built with MAX_JOBS = max_jobs.  max_jobs == 20: tsb_pfsp_create.  max_jobs == 50:
 * nodes are 208-byte tsb_pfsp_node50 records, jobs must be 50 (ta031..ta060), bounds[p*50 + k].  Every PFSP entry
 * point below works on such a handle with 208-byte records in place of 88-byte ones: evaluate / evaluate_device
 * (general kernels, csrc/pfsp_wide.cuh), the fused expand and the device pool (csrc/pfsp_wide_expand.cuh).
 * Table layouts as for tsb_pfsp_create with jobs = 50. */
int tsb_pfsp_create_wide(tsb_pfsp** h, int device, int max_jobs, int jobs, int machines, int M_max, const int32_t* p_times,
                         const int32_t* min_heads, const int32_t* min_tails, int nb_pairs, const int32_t* johnson,
                         const int32_t* lags, const int32_t* mp0, const int32_t* mp1, const int32_t* mp_order);
void tsb_pfsp_destroy(tsb_pfsp* h);

/* Replaces pfsp_gpu_chpl.chpl:384-386
 *   parents_d = parents; on device do evaluate_gpu(parents_d, jobs*count, best, lbound1_d, lbound2_d, bounds_d);
 *   bounds = bounds_d;
 * bounds[p*jobs + k] for k >= limit1+1 = lower bound of the child that schedules prmu[k] next:
 * lb_kind TSB_LB1 -> evaluate_gpu_lb1 (:192-208), TSB_LB1_D -> evaluate_gpu_lb1_d (:216-235),
 * TSB_LB2 -> evaluate_gpu_lb2 (:238-254) including its early exit against `best` (the value at
 * launch for the whole chunk; Chapel int = int64, max(int) under --ub 0). */
int tsb_pfsp_evaluate(tsb_pfsp* h, int lb_kind, const void* parents, int count, int64_t best, int32_t* bounds);
int tsb_pfsp_evaluate_device(tsb_pfsp* h, int lb_kind, const void* parents_d, int count, int64_t best,
                             int32_t* bounds_d, void* stream);
/* ---- beyond the drop-in: fused evaluate + generate_children on the device (SURVEY §8f row 1), the PFSP twin
 * of tsb_nq_expand*: evaluate_gpu (pfsp_gpu_chpl.chpl:192-270) followed by generate_children (:273-303) of one
 * chunk.  *best is the incumbent: read at entry, lowered to the smallest leaf bound of the chunk exactly as
 * the reference's sequential generate_children does (a round in which a leaf improves *best is redone through
 * the evaluate entry point and the sequential rule, so the children are the reference's in every case).
 * *n_solutions = evaluated leaf children (:283-288).  children come back packed, reference order.  Nodes are the
 * handle's records: 88-byte tsb_pfsp_node, or 208-byte tsb_pfsp_node50 on a MAX_JOBS = 50 handle; there
 * children_d must be 16-byte aligned as well (TSB_EALIGN otherwise). */
int tsb_pfsp_expand(tsb_pfsp* h, int lb_kind, const void* parents, int count, int64_t* best, void* children,
                    uint64_t capacity_nodes, uint64_t* n_children, uint64_t* n_solutions);
int tsb_pfsp_expand_device(tsb_pfsp* h, int lb_kind, const void* parents_d /*16-B aligned*/, int count,
                           int64_t* best, void* children_d /*8-B aligned*/, uint64_t* n_children,
                           uint64_t* n_solutions, void* stream);
/* ---- device-resident pool (SURVEY §8f row 3), the PFSP twin of tsb_nq_pool_*: one offload round of
 * pfsp_gpu_chpl.chpl:376-392 (popBackBulk, evaluate, generate_children) per tsb_pfsp_pool_step, the pool kept
 * in HBM and read in place.  Both builds (88- or 208-byte records, as the handle was created).  The arena starts
 * at 4 * M_max * jobs nodes (at least 2^20; env TSB200_POOL_CAP overrides) and a second arena of the same size is
 * allocated on the first compaction: on a MAX_JOBS = 50 handle with M_max = 50 000 that is 10 M x 208 B = 2.1 GB
 * per arena.  tsb_pfsp_pool_steal moves nodes between two handles of the same build only (TSB_EINVAL otherwise). */
int tsb_pfsp_pool_push(tsb_pfsp* h, const void* nodes, int64_t n);
int64_t tsb_pfsp_pool_size(const tsb_pfsp* h);
int tsb_pfsp_pool_step(tsb_pfsp* h, int lb_kind, int m, int M, int64_t* best, int64_t* n_parents,
                       uint64_t* n_children, uint64_t* n_solutions);
int tsb_pfsp_pool_drain(tsb_pfsp* h, void* nodes, int64_t capacity_nodes, int64_t* n);
int tsb_pfsp_pool_steal(tsb_pfsp* victim, tsb_pfsp* thief, int m, int64_t* n_stolen);
int tsb_pfsp_register_host(tsb_pfsp* h, void* ptr, size_t bytes);
int tsb_pfsp_unregister_host(tsb_pfsp* h, void* ptr);
int tsb_pfsp_set_xfer(tsb_pfsp* h, int mode);
uint64_t tsb_pfsp_kernel_launches(const tsb_pfsp* h);
void* tsb_pfsp_stream(const tsb_pfsp* h);
uint64_t tsb_pfsp_slow_rounds(const tsb_pfsp* h); /* expand rounds redone on the host because a leaf improved best */

/* ------------------------------------------------------------------ host-side problem data
 * (CPU code the Chapel drivers already own — lib/pfsp/Taillard.chpl, fill_* in Bound_*.chpl —
 * restated here only so that the C++ emulation drivers and the Python binding can run without
 * Chapel; a Chapel build passes its own arrays to tsb_pfsp_create instead.) */
typedef struct {
  int32_t jobs, machines, pairs;
  int32_t p_times[TSB_MAX_MACHINES * TSB_MAX_JOBS];
  int32_t min_heads[TSB_MAX_MACHINES];
  int32_t min_tails[TSB_MAX_MACHINES];
  int32_t johnson[TSB_MAX_PAIRS * TSB_MAX_JOBS];
  int32_t lags[TSB_MAX_PAIRS * TSB_MAX_JOBS];
  int32_t mp0[TSB_MAX_PAIRS], mp1[TSB_MAX_PAIRS], mp_order[TSB_MAX_PAIRS];
} tsb_pfsp_tables;

int tsb_taillard_nb_jobs(int inst);      /* lib/pfsp/Taillard.chpl:29-36 */
int tsb_taillard_nb_machines(int inst);  /* :38-52 */
int64_t tsb_taillard_best_ub(int inst);  /* :54-70 */
int tsb_pfsp_tables_build(tsb_pfsp_tables* t, int inst); /* pfsp_gpu_chpl.chpl:325-332, Chapel semantics */
/* the same with one of the reference's lb2 variants (lib/pfsp/Bound_johnson.chpl:6,36-43,50-87; the reference
 * hard-codes LB2_FULL / LB2_LEARN = all machine pairs): the pair tables are an INPUT of tsb_pfsp_create, so the
 * kernels evaluate whichever variant they are given */
enum { TSB_LB2_FULL = 0, TSB_LB2_NABESHIMA = 1, TSB_LB2_LAGEWEG = 2, TSB_LB2_LEARN = 3 };
int tsb_pfsp_tables_build_variant(tsb_pfsp_tables* t, int inst, int variant);
int tsb_pfsp_create_from_tables(tsb_pfsp** h, int device, int M_max, const tsb_pfsp_tables* t);
/* the same for a MAX_JOBS = 50 build (ta031..ta060) */
typedef struct {
  int32_t jobs, machines, pairs;
  int32_t p_times[TSB_MAX_MACHINES * TSB_MAX_JOBS_WIDE];
  int32_t min_heads[TSB_MAX_MACHINES];
  int32_t min_tails[TSB_MAX_MACHINES];
  int32_t johnson[TSB_MAX_PAIRS * TSB_MAX_JOBS_WIDE];
  int32_t lags[TSB_MAX_PAIRS * TSB_MAX_JOBS_WIDE];
  int32_t mp0[TSB_MAX_PAIRS], mp1[TSB_MAX_PAIRS], mp_order[TSB_MAX_PAIRS];
} tsb_pfsp_tables50;
int tsb_pfsp_tables50_build(tsb_pfsp_tables50* t, int inst, int variant);
int tsb_pfsp_create50_from_tables(tsb_pfsp** h, int device, int M_max, const tsb_pfsp_tables50* t);

/* ------------------------------------------------------------------ emulation of the Chapel drivers
 * (same 3-step search, same Pool contract, same --m/--M/--D meaning; used for measurement
 * because no Chapel compiler exists on the build/bench hosts).  D > 1 = static strided split
 * of the warm-up pool over D GPUs, one host thread + handle + stream per GPU, no stealing. */
typedef struct {
  uint64_t explored_tree, explored_sol;
  int64_t best;                   /* PFSP optimum (N-Queens: 0) */
  double t_step1, t_step2, t_step3; /* seconds */
  uint64_t offloads, offloaded_parents, kernel_launches;
  uint64_t per_gpu_tree[8];
  uint64_t steals;                /* successful steals between TASKS (D > 1, one process); moves between the pools of one task are not counted */
} tsb_search_stats;

/* step 1 of the drivers alone (nqueens_gpu_chpl.chpl:169-175): breadth-first from the root until the pool holds
 * min_size nodes; returns that pool (in order) and the nodes / solutions counted on the way */
int tsb_nq_warmup(int N, int min_size, void* nodes, int64_t capacity_nodes, int64_t* n, uint64_t* tree, uint64_t* sol);
/* nqueens_gpu_chpl.chpl:152-248 / nqueens_multigpu_chpl.chpl:158-352 */
int tsb_nq_search(int N, int g, int m, int M, int D, tsb_search_stats* out);
/* tsb_nq_search_device[_part] keep their handles (device pools, arenas) per (device, N, g, M) between calls; this
 * frees them.  TSB200_NO_HANDLE_CACHE=1: create and destroy per search. */
void tsb_release_cached_handles(void);
/* the same 3-step search with the pool(s) of step 2 resident on the device(s) (tsb_nq_pool_*): identical counts; the
 * host only reads three counters per call.  For chunks that fit the persistent kernel (M <= 56 832 on a B200) every
 * task splits its pool once more (the same strided split) into 4 device pools that share every launch
 * (tsb_nq_pool_run_multi): the chunk sequence is then the reference's for 4 D tasks; env TSB200_POOLS=1 = one pool
 * per task = the reference's chunk sequence for D tasks.  D > 1 = the same static strided split over the GPUs; a
 * task whose pools run dry steals the oldest half of the fullest device
 * pool over NVLink (the reference's intra-node work stealing, nqueens_multigpu_chpl.chpl:255-312, moved to the
 * device pools; env TSB200_NO_STEAL=1 = the static split alone). */
int tsb_nq_search_device(int N, int g, int m, int M, int D, tsb_search_stats* out);
/* the D = 1 search on a handle the caller created (N and M_max >= M must match): set-up stays outside the
 * search's timers, as the `on device var` declarations of the Chapel drivers do */
int tsb_nq_search_on(tsb_nq* h, int N, int m, int M, tsb_search_stats* out);
/* one task of that D-way split, on `device` — for process-per-GPU launches (one rank = one part): step 1 is
 * credited to part 0 and each part drains its own leftovers, so the parts' counts add up to the whole search */
int tsb_nq_search_device_part(int N, int g, int m, int M, int D, int part, int device, tsb_search_stats* out);
/* pfsp_gpu_chpl.chpl:306-431 / pfsp_multigpu_chpl.chpl:316-560, as the MAX_JOBS = 20 build runs them (jobs <= 20:
 * ta001..ta030; TSB_EUNSUPPORTED for larger instances) */
int tsb_pfsp_search(int inst, int lb_kind, int ub, int m, int M, int D, tsb_search_stats* out);
/* the same with the pool(s) of step 2 resident on the device(s) (tsb_pfsp_pool_*) */
int tsb_pfsp_search_device(int inst, int lb_kind, int ub, int m, int M, int D, tsb_search_stats* out);
/* the two searches as the reference built with MAX_JOBS = max_jobs runs them (`chpl -sMAX_JOBS=50`,
 * lib/pfsp/PFSP_node.chpl:7): max_jobs == 20 is tsb_pfsp_search / tsb_pfsp_search_device; max_jobs == 50 takes
 * ta031..ta060 with 208-byte nodes (TSB_EUNSUPPORTED for any other instance); any other max_jobs is
 * TSB_EUNSUPPORTED.  Arguments are checked before any device is touched.  D > 1 as for 20 jobs: static split,
 * device pools that steal from each other under ub = 1. */
int tsb_pfsp_search_wide(int max_jobs, int inst, int lb_kind, int ub, int m, int M, int D, tsb_search_stats* out);
int tsb_pfsp_search_device_wide(int max_jobs, int inst, int lb_kind, int ub, int m, int M, int D,
                                tsb_search_stats* out);
/* one task of the split (see tsb_nq_search_device_part).  The parts do not exchange their incumbent: with ub = 1 (the
 * optimum is known up front) the parts' counts add up to the whole search's; with ub = 0 every part prunes with the
 * best it finds itself, so the sum of the parts can exceed the single-process count (the optimum is still found). */
int tsb_pfsp_search_device_part(int inst, int lb_kind, int ub, int m, int M, int D, int part, int device,
                                tsb_search_stats* out);
/* the D = 1 device-pool search on a handle the caller created; a MAX_JOBS = 50 handle runs ta031..ta060 */
int tsb_pfsp_search_on(tsb_pfsp* h, int inst, int lb_kind, int ub, int m, int M, tsb_search_stats* out);

#ifdef __cplusplus
}
#endif
#endif /* TSB200_H */
