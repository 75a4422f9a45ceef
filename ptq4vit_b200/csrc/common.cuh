// Shared device/host declarations for the PTQ4ViT scale-factor search on sm_100a.
//
// Data model (see DESIGN.md):
//   * "operand image": a quantised matrix [rows][K] stored tile-wise in the tcgen05
//     no-swizzle K-major canonical layout so that one contiguous bulk copy (TMA 1-D,
//     cp.async.bulk) lands a ready-to-multiply tile in shared memory:
//         image[tile][chunk][128 rows][16 bytes]      (chunk = 16 bytes of K)
//     K is cut into "segments" (intersection of the weight column blocks and the
//     activation chunks, each padded to a multiple of 32 bytes) -- inside one
//     segment both step sizes are constant, so the integer accumulation is exact.
//   * "job": one <=128-byte-per-row slice of a segment = one shared-memory stage =
//     up to 4 tcgen05.mma K-steps.  Consecutive jobs of a segment accumulate into
//     one TMEM accumulator ("group"); the epilogue consumes one accumulator at a time.
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>

#define P4V_TILE 128           // rows per operand tile == UMMA M == UMMA N
#define P4V_JOB_KB 128         // max bytes of K per row and job
#define P4V_MAX_JOBS 320
#define P4V_MAX_GROUPS 96
#define P4V_MAX_CAND 128
#define P4V_CG 16              // columns per scale / score group
#define P4V_TILE_CG (P4V_TILE / P4V_CG)   // 8

enum : uint8_t {
  P4V_JOB_FIRST  = 1,   // first job of an accumulator group
  P4V_JOB_LAST   = 2,   // last job of an accumulator group
  P4V_JOB_RCAND  = 4,   // row operand comes from the candidate plane
  P4V_JOB_CCAND  = 8,   // column operand comes from the candidate plane
  P4V_JOB_RRES   = 16,  // row operand is candidate independent: loaded once per tile fragment (resident), not per job
  P4V_JOB_CRES   = 32,  // column operand comes from the tile's resident copy of the current column image
};

struct __align__(16) P4VJob {
  uint32_t r_off;      // byte offset inside the row-operand tile image
  uint32_t c_off;      // byte offset inside the column-operand tile image
  uint8_t  kb;         // bytes of K per row and per sub-accumulator (multiple of 32; kb * nsub <= P4V_JOB_KB)
  uint8_t  nsub;       // 0/1: one accumulator (FIRST/LAST chain rules apply); n > 1: the stage holds n consecutive K slabs,
                       //      each its own accumulator (groups group .. group+n-1), operand offsets advance by kb*128 bytes
  uint8_t  flags;
  uint8_t  group;      // accumulator group index (row of the scale table) of the first sub-accumulator
  uint32_t res_off;    // byte offset inside the resident row-operand buffer (P4V_JOB_RRES)
};

// score-group mapping of the 16-column groups (used by the sweep for scales and by
// the reduction for the argmax groups)
enum { P4V_SG_COLUMN = 0,   // scale group = global 16-column group index (Linear)
       P4V_SG_PROBLEM = 1   // scale group = problem % nsg (head-wise MatMul)
};

struct SweepParams {
  const uint8_t* R_cur;  const uint8_t* R_cand;
  const uint8_t* C_cur;  const uint8_t* C_cand;
  unsigned long long R_tile_bytes, C_tile_bytes;            // 128 * padded K bytes (current planes)
  unsigned long long R_cand_tile_bytes, C_cand_tile_bytes;  // same for the candidate planes
  unsigned long long R_cand_stride, C_cand_stride;          // bytes between candidate planes
  int P, M, N, tiles_m, tiles_n;
  const float* Y; const float* Gr; const float* bias;   // bias may be null
  const float* gscale;                                  // device scalar: power-of-two gradient scale
  long long ld, prob_stride;
  const P4VJob* jobs;       // [n_fixed_jobs] then [n_cand_jobs]
  int n_fixed_jobs, n_cand_jobs, n_fixed_groups, n_cand_groups;
  const float* fix_scale;   // [n_fixed_groups][nsg]
  const float* candA;       // [n_cand][nsg]
  const float* candB;       // [n_cand_groups][nsg]
  int nsg, sg_mode;
  unsigned long long cand_noA_mask;   // bit g set: candidate group g ignores candA (scale = candB only)
  int n_cand;
  float* partial;           // [tiles_total][n_cand][4][8]
  float* out;               // if non-null: no candidates; write bias + sum(scale*acc) of the fixed groups (quant_forward)
  int out_residual;         // with out: write y - bias - sum(scale*acc) instead (the current residual e)
  int order;                // 0: tile_m fastest, 1: tile_n fastest
  int is_int8;
  int R_shared;             // the row operand does not depend on the problem index (conv: kernel planes shared by all images)
  int row_keys;             // single-segment steps: one score per ROW, partial = [tile][candidate][column half][128 rows]
  // shared-memory plan, filled by the launcher
  unsigned int stage_r_bytes, stage_c_bytes, n_stages, resident_bytes, resident_bufs, cres_bytes;
  long long* trace;         // debug: clock64 timeline of CTA 0 ([3 roles][512 events][4]) or null
  int debug_mode;           // debug (env P4V_SWEEP_DEBUG): 1 = no operand traffic / no MMA (epilogue + handshakes only), 2 = epilogue does no math
};

static inline __host__ __device__ int p4v_cdiv(int a, int b) { return (a + b - 1) / b; }
static inline __host__ __device__ unsigned p4v_job_nsub(const P4VJob& j) { return j.nsub ? j.nsub : 1u; }
static inline __host__ __device__ unsigned p4v_job_bytes(const P4VJob& j) { return (unsigned)j.kb * p4v_job_nsub(j) * P4V_TILE; }   // per operand

#ifdef __CUDACC__
// ---- exact rounding division shared by the operand-image and the Gram kernels ----
// rintf(__fdiv_rn(v, delta)) without the general-purpose division: rcp must be __frcp_rn(delta).
// q1 = q0 + (v - delta*q0)*rcp differs from the correctly rounded quotient by at most one ulp, so rint(q1) equals
// rint(v/delta) unless q1 lies within a few ulps of a half-integer; those (one in ~10^4) and non-finite values
// take the exact division.  Only valid for 2^-100 < |delta| < 2^100 (p4v_rint_div_ok, checked once per step size).
__device__ __forceinline__ float p4v_rint_div(float v, float delta, float rcp) {
  const float q0 = v * rcp;
  const float q1 = fmaf(fmaf(-delta, q0, v), rcp, q0);
  const float n = rintf(q1);
  const float aq = fabsf(q1);
  const float dist = fabsf(fabsf(q1 - n) - 0.5f);
  if (!(aq <= 3.0e38f) || dist <= aq * 4.8e-7f) return rintf(__fdiv_rn(v, delta));
  return n;
}

__device__ __forceinline__ bool p4v_rint_div_ok(float delta) { const float ad = fabsf(delta); return ad > 7.9e-31f && ad < 1.2e30f; }

#endif

// ---- error plumbing (host) --------------------------------------------------
#ifdef __cplusplus
extern "C" void p4v_set_error(const char* fmt, ...);
#endif
#define P4V_CUDA_OK(expr)                                                            \
  do { cudaError_t _e = (expr);                                                      \
       if (_e != cudaSuccess) { p4v_set_error("%s:%d %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
                                return 2; } } while (0)
#define P4V_REQUIRE(cond, ...)                                                       \
  do { if (!(cond)) { p4v_set_error(__VA_ARGS__); return 1; } } while (0)

// ---- kernel launchers shared between translation units ----------------------
int p4v_launch_sweep_tc(const SweepParams& p, const P4VJob* host_jobs, int num_sms, cudaStream_t st);
int p4v_launch_sweep_simt(const SweepParams& p, cudaStream_t st);

// ---- library runtime (runtime.cu) -------------------------------------------
void p4v_count_launch();     // every kernel launch of the library counts itself (p4v_launch_count)
int p4v_num_sms();
// one sweep launch on the kernel desc.kernel selects (P4V_KERNEL_*), counted and, while profiling is on, timed
int p4v_run_sweep(const SweepParams& sp, const P4VJob* host_jobs, int kernel, cudaStream_t st);
// live kernel timing: kinds of the record p4v_profile_collect_kinds reports
enum { P4V_PROF_SWEEP_BF16 = 0, P4V_PROF_SWEEP_INT8 = 1, P4V_PROF_GRAM_GEMM = 2, P4V_PROF_KINDS = 3 };
bool p4v_prof_on();
void p4v_prof_begin(cudaStream_t st, cudaEvent_t* e0);
void p4v_prof_end(cudaStream_t st, cudaEvent_t e0, int kind, double ops);
