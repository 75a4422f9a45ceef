// Library-wide runtime shared by every operator: error state, version, the launch counter, the live kernel timing
// behind bench.py's roofline, and the sweep launch every search step goes through.
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <vector>

#include "../../include/ptq4vit_b200.h"
#include "common.cuh"

// ---------------------------------------------------------------- error / misc
static thread_local char g_err[512] = "";
static long long g_launches = 0;
extern "C" __attribute__((visibility("default"))) void p4v_set_error(const char* fmt, ...) {
  va_list ap; va_start(ap, fmt); vsnprintf(g_err, sizeof(g_err), fmt, ap); va_end(ap);
}
extern "C" const char* p4v_last_error(void) { return g_err; }
extern "C" int p4v_version(void) { return 100; }
extern "C" long long p4v_launch_count(void) { return g_launches; }
void p4v_count_launch() { ++g_launches; }

// ---- live kernel timing (bench.py's roofline) ---------------------------------
// While enabled every tensor-core launch (slab sweep, Gram GEMM) is bracketed by CUDA events on its own stream and
// recorded with its kind and the tensor-core operations (2*MAC) it executes.
static bool g_prof = false;
struct ProfRec { cudaEvent_t e0, e1; int kind; double ops; int n_cand, nfg, ncg, nfj, ncj, out; long long tiles; };
static std::vector<ProfRec> g_prof_recs;
static std::vector<cudaEvent_t> g_prof_pool;
static cudaEvent_t prof_event() {
  if (!g_prof_pool.empty()) { cudaEvent_t e = g_prof_pool.back(); g_prof_pool.pop_back(); return e; }
  cudaEvent_t e; cudaEventCreate(&e); return e;
}
bool p4v_prof_on() { return g_prof; }
void p4v_prof_begin(cudaStream_t st, cudaEvent_t* e0) { *e0 = prof_event(); cudaEventRecord(*e0, st); }
void p4v_prof_end(cudaStream_t st, cudaEvent_t e0, int kind, double ops) {
  cudaEvent_t e1 = prof_event(); cudaEventRecord(e1, st);
  g_prof_recs.push_back(ProfRec{e0, e1, kind, ops, 0, 0, 0, 0, 0, 0, 0});
}
extern "C" int p4v_profile_enable(int on) { g_prof = on != 0; return 0; }
// out[0..2] ms per kind (bf16 sweep, int8 sweep, Gram GEMM), out[3..5] executed ops, out[6..8] launches,
// out[9..11] the longest single launch: ms, ops, kind.  Synchronises the recorded events and clears the record.
extern "C" int p4v_profile_collect_kinds(double* out, int n) {
  P4V_REQUIRE(out && n >= 12, "profile_collect_kinds: need 12 doubles");
  for (int i = 0; i < 12; ++i) out[i] = 0.0;
  static const bool log_each = getenv("P4V_PROFILE_LOG") != nullptr;   // debug: one stderr line per launch
  for (auto& r : g_prof_recs) {
    P4V_CUDA_OK(cudaEventSynchronize(r.e1));
    float t = 0.f;
    P4V_CUDA_OK(cudaEventElapsedTime(&t, r.e0, r.e1));
    out[r.kind] += t; out[3 + r.kind] += r.ops; out[6 + r.kind] += 1.0;
    if (t > out[9]) { out[9] = t; out[10] = r.ops; out[11] = r.kind; }
    if (log_each)
      fprintf(stderr, "[p4v launch] %8.1f us kind=%d cand=%d fixed_groups=%d cand_groups=%d fixed_jobs=%d cand_jobs=%d out=%d tiles=%lld  %.1f TOP/s\n",
              t * 1e3, r.kind, r.n_cand, r.nfg, r.ncg, r.nfj, r.ncj, r.out, r.tiles, r.ops / (t * 1e-3) / 1e12);
    g_prof_pool.push_back(r.e0); g_prof_pool.push_back(r.e1);
  }
  g_prof_recs.clear();
  return 0;
}
extern "C" int p4v_profile_collect(double* sweep_ms, long long* sweep_launches, double* executed_ops) {
  double o[12];
  int rc = p4v_profile_collect_kinds(o, 12);
  if (rc) return rc;
  if (sweep_ms) *sweep_ms = o[0] + o[1];
  if (sweep_launches) *sweep_launches = (long long)(o[6] + o[7]);
  if (executed_ops) *executed_ops = o[3] + o[4];
  return 0;
}
// tensor-core work of one sweep launch: every job multiplies a 128x128 tile over kb bytes of K
static double sweep_ops(const SweepParams& sp, const P4VJob* host_jobs) {
  double kf = 0.0, kc = 0.0;
  const double ew = sp.is_int8 ? 1.0 : 2.0;
  for (int j = 0; j < sp.n_fixed_jobs; ++j) kf += host_jobs[j].kb * p4v_job_nsub(host_jobs[j]) / ew;
  for (int j = 0; j < sp.n_cand_jobs; ++j) kc += host_jobs[sp.n_fixed_jobs + j].kb * p4v_job_nsub(host_jobs[sp.n_fixed_jobs + j]) / ew;
  const double tiles = (double)sp.P * sp.tiles_m * sp.tiles_n;
  return 2.0 * P4V_TILE * P4V_TILE * tiles * (kf + kc * sp.n_cand);
}
static long long* g_trace = nullptr;
extern "C" __attribute__((visibility("default"))) int p4v_debug_trace(void* dev_ptr) { g_trace = (long long*)dev_ptr; return 0; }
int p4v_run_sweep(const SweepParams& sp_in, const P4VJob* host_jobs, int kernel, cudaStream_t st) {
  SweepParams sp = sp_in; sp.trace = g_trace;
  ++g_launches;
  cudaEvent_t e0 = nullptr;
  if (g_prof) p4v_prof_begin(st, &e0);
  int rc = kernel == P4V_KERNEL_SIMT ? p4v_launch_sweep_simt(sp, st) : p4v_launch_sweep_tc(sp, host_jobs, p4v_num_sms(), st);
  if (g_prof) {
    p4v_prof_end(st, e0, sp.is_int8 ? P4V_PROF_SWEEP_INT8 : P4V_PROF_SWEEP_BF16, sweep_ops(sp, host_jobs));
    ProfRec& r = g_prof_recs.back();
    r.n_cand = sp.n_cand; r.nfg = sp.n_fixed_groups; r.ncg = sp.n_cand_groups; r.nfj = sp.n_fixed_jobs; r.ncj = sp.n_cand_jobs;
    r.out = sp.out != nullptr; r.tiles = (long long)sp.P * sp.tiles_m * sp.tiles_n;
  }
  return rc;
}

int p4v_num_sms() {
  static int sms = 0;
  if (sms == 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 148;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0) sms = 148;
  }
  return sms;
}
