// pfsp_b200 — C++ stand-in for pfsp_gpu_chpl / pfsp_multigpu_chpl.  Same CLI (--inst --lb --ub --m --M
// --D; README.md:47-87), same defaults (pfsp_multigpu_chpl.chpl:24-30: inst 14, lb "lb1", ub 1), same
// result lines (pfsp_gpu_chpl.chpl:66-77).  --lb takes the Chapel spelling lb1 | lb1_d | lb2.  --inst 31..60 (50 jobs)
// runs as the reference built with `-sMAX_JOBS=50` (lib/pfsp/PFSP_node.chpl:7) does: 208-byte nodes.
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "tsb200.h"

int main(int argc, char** argv) {
  int inst = 14, ub = 1, m = 25, M = 50000, D = 1, lb = TSB_LB1, devpool = 0;
  const char* lbs = "lb1";
  for (int i = 1; i < argc; i++) {
    if (!std::strcmp(argv[i], "-h") || !std::strcmp(argv[i], "--help")) {
      std::printf("\n  PFSP Benchmark Parameters:\n\n   --inst   int   Taillard's instance to solve (between 001 and 120)\n"
                  "   --lb     str   lower bound function (lb1, lb1_d, lb2)\n"
                  "   --ub     int   initial upper bound (0, 1)\n   --m --M --D as for N-Queens\n\n");
      return 1;
    }
    if (i + 1 >= argc) break;
    if (!std::strcmp(argv[i], "--lb")) {
      lbs = argv[++i];
      lb = !std::strcmp(lbs, "lb1") ? TSB_LB1 : !std::strcmp(lbs, "lb1_d") ? TSB_LB1_D
           : !std::strcmp(lbs, "lb2") ? TSB_LB2 : -1;
      continue;
    }
    int* dst = !std::strcmp(argv[i], "--inst") ? &inst : !std::strcmp(argv[i], "--ub") ? &ub
             : !std::strcmp(argv[i], "--m") ? &m : !std::strcmp(argv[i], "--M") ? &M
             : !std::strcmp(argv[i], "--D") ? &D
             : !std::strcmp(argv[i], "--devpool") ? &devpool : nullptr;  // 1: pool(s) of step 2 resident on the GPU
    if (dst) *dst = std::atoi(argv[++i]);
  }
  if (m <= 0 || M <= 0) { std::fprintf(stderr, "Error: m and M must be positive integers.\n"); return 2; }
  if (inst < 1 || inst > 120) { std::fprintf(stderr, "Error: unsupported Taillard's instance\n"); return 2; }
  if (lb < 0) { std::fprintf(stderr, "Error - Unsupported lower bound\n"); return 2; }
  if (ub != 0 && ub != 1) { std::fprintf(stderr, "Error: unsupported upper bound initialization\n"); return 2; }
  std::printf("\n=================================================\n%s B200 (tsb200)\n\n"
              "Resolution of PFSP Taillard's instance: ta%d (m = %d, n = %d)\nInitial upper bound: %s\n"
              "Lower bound function: %s\nBranching rule: fwd\n=================================================\n",
              D > 1 ? "Multi-GPU" : "Single-GPU", inst, tsb_taillard_nb_machines(inst), tsb_taillard_nb_jobs(inst),
              ub ? "opt" : "inf", lbs);
  if (tsb_taillard_nb_jobs(inst) > TSB_MAX_JOBS_WIDE) {
    std::fprintf(stderr, "Error: ta%03d has %d jobs; this build takes up to %d (ta001..ta060)\n", inst,
                 tsb_taillard_nb_jobs(inst), TSB_MAX_JOBS_WIDE);
    return 2;
  }
  const int max_jobs = tsb_taillard_nb_jobs(inst) > TSB_MAX_JOBS ? TSB_MAX_JOBS_WIDE : TSB_MAX_JOBS;
  tsb_search_stats st;
  const int rc = devpool ? tsb_pfsp_search_device_wide(max_jobs, inst, lb, ub, m, M, D, &st)
                         : tsb_pfsp_search_wide(max_jobs, inst, lb, ub, m, M, D, &st);
  if (rc != TSB_OK) {
    std::fprintf(stderr, "tsb_pfsp_search: %s (%s)\n", tsb_strerror(rc), tsb_last_cuda_error());
    return 3;
  }
  const double t = st.t_step1 + st.t_step2 + st.t_step3;
  std::printf("\nInitial search on CPU completed\nElapsed time: %f [s]\n\nSearch on GPU completed\n"
              "Elapsed time: %f [s]\n\nSearch on CPU completed\nElapsed time: %f [s]\n\nExploration terminated.\n",
              st.t_step1, st.t_step2, st.t_step3);
  const long long initUB = ub ? tsb_taillard_best_ub(inst) : 0x7fffffffffffffffLL;
  std::printf("\n=================================================\n"
              "Size of the explored tree: %llu\nNumber of explored solutions: %llu\n"
              "Optimal makespan: %lld%s\nElapsed time: %f [s]\n"
              "=================================================\n\n",
              (unsigned long long)st.explored_tree, (unsigned long long)st.explored_sol, (long long)st.best,
              st.best < initUB ? " (improved)" : " (not improved)", t);
  std::printf("GPU diagnostics:\n   kernel_launch: %llu\n   offloads: %llu\n   Mnodes/s: %.3f\n",
              (unsigned long long)st.kernel_launches, (unsigned long long)st.offloads, st.explored_tree / t / 1e6);
  return 0;
}
