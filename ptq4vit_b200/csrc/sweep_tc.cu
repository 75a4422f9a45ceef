// The hot kernel: candidate sweep on tcgen05 tensor cores (sm_100a).
//
// Replaces, for one search step, the reference's loop
//   for c in candidates: out = F.linear(x_sim, w_sim_c) ; sim = -(g*(y-out))**2 ; mean/sum
// (quant_layers/linear.py:466-488, :507-526; quant_layers/matmul.py:500-514, :541-555)
// without ever writing a candidate output to HBM.
//
// One persistent CTA per SM.  Work = (output tile 128x128) x (candidates).  Whole tiles are dealt
// round-robin in waves of gridDim.x (CTAs that run together share operand tiles in L2); the last partial
// wave is split at candidate granularity so that every SM finishes together.  Per tile fragment:
//   1. the 256 epilogue threads load r = y - bias and g = grad * 2^k for their (row, 64 columns): r into
//      registers; g into registers (single-segment steps) or into this thread's shared-memory row
//      (multi-segment steps, where it is needed once per candidate);
//   2. "fixed" segments (everything the candidate does not change) are multiplied on the tensor cores and
//      subtracted: r -= scale * acc;
//   3. per candidate only the segment(s) touched by the candidate step size are multiplied (bulk copy
//      -> smem ring -> tcgen05.mma -> TMEM); the epilogue forms (g * (r - scale_c * acc))^2 straight from
//      TMEM and writes one partial per (row quarter, 16 columns): single-segment steps sum the rows through
//      shared memory in batches of candidates, multi-segment steps with a shuffle butterfly per candidate.
// A job = one ring stage = up to 128 bytes of K of both operands, possibly several adjacent K slabs with an
// accumulator each (P4VJob::nsub); operands that do not change between candidates stay resident in shared memory.
// Roles: warp 0 = bulk-copy producer, warp 1 = MMA issuer (+TMEM alloc), warps 4..11 = epilogue
// (setmaxnreg moves the register budget of warpgroup 0 to the epilogue warpgroups; it only REDISTRIBUTES the
// registers the CTA was launched with, 384 x 168 = 128 x 56 + 256 x 224 -- asking for more blocks the .inc forever).
// Round-2 measurements of two epilogue alternatives, both parity-green and both rejected (profiles/README.md):
//   * one tcgen05.ld.x64 per accumulator, double buffered over whole accumulators (192 live registers, spills):
//     fc2 weight step 547 vs 467 us, qkv activation step 6.3 vs 4.6 ms;
//   * 16 epilogue warps x 32 columns (104 registers each): fc2 weight step 436 us, QK step 1.18 vs 1.38 ms, but the
//     qkv activation step 5.5 vs 4.6 ms -- that step streams 393 KB of operands per candidate tile from L2 (6.8 TB/s in
//     ncu = the L2->SM limit), so more epilogue parallelism cannot help it and the extra TMEM traffic hurts.
#include "common.cuh"
#include <algorithm>
#include <cstdio>
#include <cstdlib>

namespace {

#ifdef P4V_DEBUG_MODES   // debug build only (-DP4V_DEBUG_MODES): runtime-selectable partial execution, see SweepParams::debug_mode
#define DBG_MODE(P) ((P).debug_mode)
#else
#define DBG_MODE(P) 0
#endif
#ifdef P4V_TRACE   // debug build only: clock64 timeline of CTA 0 (tools/trace_sweep.py)
#define TRACE(role, ev, col) do { if (P.trace && blockIdx.x == 0 && (ev) < 512 && (threadIdx.x & 31) == 0) P.trace[((role) * 512 + (ev)) * 4 + (col)] = clock64(); } while (0)
#else
#define TRACE(role, ev, col) do { } while (0)
#endif

constexpr int kMaxStages = 16;
constexpr int kAccCols = 128;
constexpr int kTmemCols = 512;
constexpr int kEpiThreads = 256;
constexpr int kEpiWarps = 8;
constexpr int kThreads = 128 + kEpiThreads;   // warpgroup 0: producer, MMA, 2 idle warps; warpgroups 1-2: epilogue
constexpr int kSmemBudget = 200 * 1024;       // ring + resident operand (+ score reduction buffers of the single-segment steps)
// Score reduction of the single-segment steps: every epilogue thread drops its 4 per-group sums of one candidate into
// shared memory (one conflict-free 16-byte store, no shuffle chain); every kRedBatch candidates the 256 threads sum
// the 128 rows of each (candidate, group) in 4 row quarters.  Layout [buffer][candidate][column half][row][4].
constexpr int kRedBatch = 8;
constexpr int kRedHalf = P4V_TILE * 4 + 4;    // floats; +4 shifts the second column half by four banks
constexpr int kRedCand = 2 * kRedHalf;
constexpr int kRedBytes = 2 * kRedBatch * kRedCand * 4;

struct SmemCtl {
  alignas(16) P4VJob jobs[P4V_MAX_JOBS];
  float fixs[P4V_MAX_GROUPS][P4V_TILE_CG];
  float candA[P4V_MAX_CAND][P4V_TILE_CG];
  float candB[P4V_MAX_GROUPS][P4V_TILE_CG];
  alignas(8) unsigned long long full[kMaxStages];
  unsigned long long empty[kMaxStages];
  unsigned long long acc_full[4];
  unsigned long long acc_empty[4];
  unsigned long long res_full[2];
  unsigned long long res_empty[2];
  unsigned long long cres_full, cres_empty;
  uint32_t tmem_base;
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(void* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(void* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(void* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try(uint32_t addr, uint32_t parity) {
  uint32_t ok;
  asm volatile("{\n\t.reg .pred p;\n\t"
               "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
               "selp.u32 %0, 1, 0, p;\n\t}" : "=r"(ok) : "r"(addr), "r"(parity) : "memory");
  return ok != 0;
}
// Bounded wait: a protocol bug must surface as a trapped launch (cudaErrorLaunchFailure), never as a hung GPU.  The bound
// is ~10 s of SM clocks: clock64 keeps counting while a context is time-sliced (MPS, profilers), a legitimate wait of a
// sub-millisecond kernel must never reach it.
[[noreturn]] __device__ __noinline__ void mbar_timeout(uint32_t addr, uint32_t parity) {
  printf("ptq4vit_b200 sweep: mbarrier wait timed out (block %d thread %d smem 0x%x parity %u)\n",
         (int)blockIdx.x, (int)threadIdx.x, addr, parity);
  __trap();
  while (true) {}
}
__device__ __noinline__ void mbar_wait_slow(uint32_t addr, uint32_t parity) {
  const long long t0 = clock64();
  while (!mbar_try(addr, parity))
    if (clock64() - t0 > 20000000000ll) mbar_timeout(addr, parity);
}
__device__ __forceinline__ void mbar_wait(void* bar, uint32_t parity) {     // fully inline: safe with many live registers
  const uint32_t addr = smem_u32(bar);
  if (mbar_try(addr, parity)) return;
  const long long t0 = clock64();
  while (!mbar_try(addr, parity))
    if (clock64() - t0 > 20000000000ll) mbar_timeout(addr, parity);
}
__device__ __forceinline__ void mbar_wait_addr(uint32_t addr, uint32_t parity) {
  if (!mbar_try(addr, parity)) mbar_wait_slow(addr, parity);
}
__device__ __forceinline__ void mbar_expect_tx_addr(uint32_t addr, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(addr), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s_addr(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ void tc_commit_addr(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, void* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(dst), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
// Warp-uniform single-lane election: code guarded by this predicate lets ptxas keep the operands of the
// async-proxy instructions (UTCHMMA / UTCBAR / UBLKCP) in uniform registers without a per-lane waterfall loop.
__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(void* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// K-major, no swizzle: core matrix = 8 rows x 16 B; LBO = stride between the 16-byte chunks of one K-step (2048 B),
// SBO = stride between 8-row groups (128 B).  Descriptor with the constant fields only; the 14-bit start-address field (bits 0..13, units of 16 B) is added per use
__device__ __forceinline__ uint64_t desc_hi_const() {
  constexpr uint64_t lbo = (P4V_TILE * 16) >> 4, sbo = 128 >> 4;
  return (lbo << 16) | (sbo << 32) | (1ull << 46);
}
template <bool kInt8>
__device__ __forceinline__ void umma(uint32_t d_tmem, uint64_t da, uint64_t db, uint32_t accumulate) {
  // instruction descriptor: c_format (S32=2 | F32=1) @4, a/b format (S8=1 | BF16=1) @7/@10,
  // K-major both, N>>3 @17, M>>4 @24
  constexpr uint32_t idesc = ((kInt8 ? 2u : 1u) << 4) | (1u << 7) | (1u << 10) |
                             ((uint32_t)(P4V_TILE >> 3) << 17) | ((uint32_t)(P4V_TILE >> 4) << 24);
  if constexpr (kInt8) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}"
                 ::"r"(d_tmem), "l"(da), "l"(db), "r"(idesc), "r"(accumulate) : "memory");
  } else {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
                 ::"r"(d_tmem), "l"(da), "l"(db), "r"(idesc), "r"(accumulate) : "memory");
  }
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld32f(uint32_t taddr, float* v) {   // same, straight into a float register array
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
      "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7]),
        "=f"(v[8]), "=f"(v[9]), "=f"(v[10]), "=f"(v[11]), "=f"(v[12]), "=f"(v[13]), "=f"(v[14]), "=f"(v[15]),
        "=f"(v[16]), "=f"(v[17]), "=f"(v[18]), "=f"(v[19]), "=f"(v[20]), "=f"(v[21]), "=f"(v[22]), "=f"(v[23]),
        "=f"(v[24]), "=f"(v[25]), "=f"(v[26]), "=f"(v[27]), "=f"(v[28]), "=f"(v[29]), "=f"(v[30]), "=f"(v[31])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const float* v) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,"
      "%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31,%32};"
      ::"r"(taddr),
        "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]), "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7]),
        "f"(v[8]), "f"(v[9]), "f"(v[10]), "f"(v[11]), "f"(v[12]), "f"(v[13]), "f"(v[14]), "f"(v[15]),
        "f"(v[16]), "f"(v[17]), "f"(v[18]), "f"(v[19]), "f"(v[20]), "f"(v[21]), "f"(v[22]), "f"(v[23]),
        "f"(v[24]), "f"(v[25]), "f"(v[26]), "f"(v[27]), "f"(v[28]), "f"(v[29]), "f"(v[30]), "f"(v[31])
      : "memory");
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// ---- work distribution -------------------------------------------------------------------------
struct Frag { int tile, p, tm, tn, c0, c1; };
struct Sched {
  int waves, k;                 // whole-tile waves, next wave index
  long long u, u_end;           // candidate-granular units of the tail wave
  int tail_tile0;
};
__device__ __forceinline__ void sched_init(const SweepParams& P, Sched& s) {
  const int tiles = P.P * P.tiles_m * P.tiles_n;
  const int G = gridDim.x;
  s.waves = tiles / G; s.k = 0;
  const long long tail_units = (long long)(tiles % G) * P.n_cand;
  s.u = tail_units * blockIdx.x / G; s.u_end = tail_units * (blockIdx.x + 1) / G;
  s.tail_tile0 = s.waves * G;
}
__device__ __forceinline__ bool next_frag(const SweepParams& P, Sched& s, Frag& f) {
  if (s.k < s.waves) {
    f.tile = s.k * gridDim.x + blockIdx.x; f.c0 = 0; f.c1 = P.n_cand; ++s.k;
  } else {
    if (s.u >= s.u_end) return false;
    f.tile = s.tail_tile0 + (int)(s.u / P.n_cand);
    f.c0 = (int)(s.u % P.n_cand);
    const long long rem = s.u_end - s.u;
    f.c1 = (int)((rem < (long long)(P.n_cand - f.c0)) ? f.c0 + rem : P.n_cand);
    s.u += f.c1 - f.c0;
  }
  const int per_p = P.tiles_m * P.tiles_n;
  f.p = f.tile / per_p;
  const int t = f.tile % per_p;
  if (P.order == 0) { f.tm = t % P.tiles_m; f.tn = t / P.tiles_m; }
  else              { f.tn = t % P.tiles_n; f.tm = t / P.tiles_n; }
  return true;
}

template <bool kInt8>
__device__ __forceinline__ float acc_to_float(uint32_t a) {
  if constexpr (kInt8) return __int2float_rn((int)a);
  else return __uint_as_float(a);
}

// ---- packed fp32x2 math (sm_100: FFMA2/FMUL2 halve the issue slots of the epilogue) ----
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 pack2(float a, float b) { f32x2 r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a), "f"(b)); return r; }
__device__ __forceinline__ void unpack2(f32x2 v, float& a, float& b) { asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v)); }
__device__ __forceinline__ f32x2 fma2(f32x2 a, f32x2 b, f32x2 c) { f32x2 d; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c)); return d; }
__device__ __forceinline__ f32x2 mul2(f32x2 a, f32x2 b) { f32x2 d; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }

// A quarter of this thread's 64 accumulator columns (16 columns = one scale / score group, already in registers)
// against the running residual.
//   kScore == false:  r -= s * acc                        (fixed segments / non-final candidate segments)
//   kScore == true :  p = sum (g * (r - s*acc))^2          (final candidate segment; r is not modified)
template <bool kInt8, bool kScore, int OFF>
__device__ __forceinline__ void consume16(const uint32_t (&a)[16], float (&r)[64], const float (&g)[64], const float s, float& p) {
  f32x2 q0 = 0ull, q1 = 0ull;
  const f32x2 ns = pack2(-s, -s);
#pragma unroll
  for (int j = 0; j < 16; j += 2) {
    const f32x2 f = pack2(acc_to_float<kInt8>(a[j]), acc_to_float<kInt8>(a[j + 1]));
    const f32x2 d = fma2(ns, f, pack2(r[OFF + j], r[OFF + j + 1]));
    if constexpr (kScore) {
      const f32x2 w = mul2(pack2(g[OFF + j], g[OFF + j + 1]), d);
      if (j & 2) q1 = fma2(w, w, q1); else q0 = fma2(w, w, q0);
    } else {
      unpack2(d, r[OFF + j], r[OFF + j + 1]);
    }
  }
  if constexpr (kScore) { float x0, y0, x1, y1; unpack2(q0, x0, y0); unpack2(q1, x1, y1); p = (x0 + y0) + (x1 + y1); }
}

// Reduce 4 per-lane values over the 32 lanes (= rows) of the warp, fixed order: lane 8*k ends up with the total of value k.
__device__ __forceinline__ float reduce4_over_rows(float v0, float v1, float v2, float v3, int lane) {
  const unsigned full = 0xffffffffu;
  const bool hi16 = lane & 16;
  float s0 = hi16 ? v0 : v2, s1 = hi16 ? v1 : v3;
  float k0 = hi16 ? v2 : v0, k1 = hi16 ? v3 : v1;
  k0 += __shfl_xor_sync(full, s0, 16);
  k1 += __shfl_xor_sync(full, s1, 16);
  const bool hi8 = lane & 8;
  float s = hi8 ? k0 : k1, k = hi8 ? k1 : k0;
  k += __shfl_xor_sync(full, s, 8);
  k += __shfl_xor_sync(full, k, 4);
  k += __shfl_xor_sync(full, k, 2);
  k += __shfl_xor_sync(full, k, 1);
  return k;
}

// ---- epilogue accumulator pipeline ----------------------------------------------------------------
// The epilogue walks the accumulators of the TMEM ring in order.  `a0` always holds the first 32 columns
// of the accumulator about to be consumed (already complete); while the CUDA cores work on one half the
// TMEM load of the next half is in flight, and the slot goes back to the MMA warp as soon as its second
// half has landed in registers.
struct AccRing { uint32_t slot, phase, nslots; };

__device__ __forceinline__ void acc_begin(SmemCtl& S, AccRing& ring, uint32_t tbase, uint32_t (&a0)[16]) {
  mbar_wait(&S.acc_full[ring.slot], ring.phase);
  tc_fence_after();
  tmem_ld16(tbase + ring.slot * kAccCols, a0);
  tmem_wait_ld();
}

// One accumulator = four 16-column quarters, double buffered in a0/a1: the TMEM load of the next quarter is in flight
// while the CUDA cores work on the current one; the slot returns to the MMA warp once its last quarter is in registers.
template <bool kInt8, bool kScore>
__device__ __forceinline__ void acc_step(SmemCtl& S, AccRing& ring, uint32_t tbase, int lane, uint32_t (&a0)[16],
                                         uint32_t (&a1)[16], float (&r)[64], const float (&g)[64], const float4 sc,
                                         float (&p)[4], const bool has_next, const bool skip_math = false) {
  const uint32_t t0 = tbase + ring.slot * kAccCols;
  uint32_t nslot = ring.slot + 1, nphase = ring.phase;
  if (nslot == ring.nslots) { nslot = 0; nphase ^= 1; }
  if (skip_math) {                 // debug mode 2: handshakes only
    p[0] = p[1] = p[2] = p[3] = 0.f;
    tc_fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive(&S.acc_empty[ring.slot]);
    ring.slot = nslot; ring.phase = nphase;
    if (has_next) { mbar_wait(&S.acc_full[ring.slot], ring.phase); tc_fence_after(); }
    return;
  }
  // non-blocking probe of the NEXT accumulator's barrier: its latency hides behind this accumulator's math
  const uint32_t next_bar = smem_u32(&S.acc_full[nslot]);
  bool next_ready = true;
  if (has_next) next_ready = mbar_try(next_bar, nphase);
  tmem_ld16(t0 + 16, a1);
  consume16<kInt8, kScore, 0>(a0, r, g, sc.x, p[0]);
  tmem_wait_ld();
  tmem_ld16(t0 + 32, a0);
  consume16<kInt8, kScore, 16>(a1, r, g, sc.y, p[1]);
  tmem_wait_ld();
  tmem_ld16(t0 + 48, a1);
  consume16<kInt8, kScore, 32>(a0, r, g, sc.z, p[2]);
  tmem_wait_ld();
  tc_fence_before();
  __syncwarp();
  if (lane == 0) mbar_arrive(&S.acc_empty[ring.slot]);      // one arrival per epilogue warp
  ring.slot = nslot; ring.phase = nphase;
  if (has_next) {
    if (!next_ready) mbar_wait(&S.acc_full[nslot], nphase);
    tc_fence_after();
    tmem_ld16(tbase + nslot * kAccCols, a0);
  }
  consume16<kInt8, kScore, 48>(a1, r, g, sc.w, p[3]);
  if (has_next) tmem_wait_ld();
}


// ---- multi-segment steps: 32-column halves, gradient tile parked in shared memory ----------------------------
// Steps with many accumulators per candidate (activation steps) spend one FMA per element on all but the last
// accumulator, so a 16-column quarter does not cover the latency of the next TMEM load.  Here the gradient tile is
// NOT kept in registers (it is needed once per candidate); the registers hold two 32-column halves instead.
__device__ __forceinline__ void tmem_ld32u(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
      "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
        "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
        "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr));
}
// gp: this thread's row of the parked gradient tile, [column quad][128 rows] float4 (quad stride = 128 float4)
template <bool kInt8, bool kScore, int OFF>
__device__ __forceinline__ void consume32(const uint32_t (&a)[32], float (&r)[64], const float4* gp, const float s0,
                                          const float s1, float& p0, float& p1) {
  if constexpr (!kScore) {
#pragma unroll
    for (int j = 0; j < 32; j += 2) {
      const float s = j < 16 ? s0 : s1;
      const f32x2 d = fma2(pack2(-s, -s), pack2(acc_to_float<kInt8>(a[j]), acc_to_float<kInt8>(a[j + 1])), pack2(r[OFF + j], r[OFF + j + 1]));
      unpack2(d, r[OFF + j], r[OFF + j + 1]);
    }
  } else {
    float q[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const float4 gv = gp[(OFF / 4 + k) * P4V_TILE];
      const float s = k < 4 ? s0 : s1;
      const int j = 4 * k;
      const float d0 = fmaf(-s, acc_to_float<kInt8>(a[j]), r[OFF + j]), d1 = fmaf(-s, acc_to_float<kInt8>(a[j + 1]), r[OFF + j + 1]);
      const float d2 = fmaf(-s, acc_to_float<kInt8>(a[j + 2]), r[OFF + j + 2]), d3 = fmaf(-s, acc_to_float<kInt8>(a[j + 3]), r[OFF + j + 3]);
      const float w0 = gv.x * d0, w1 = gv.y * d1, w2 = gv.z * d2, w3 = gv.w * d3;
      float& qa = q[(k < 4 ? 0 : 2)]; float& qb = q[(k < 4 ? 1 : 3)];
      qa = fmaf(w0, w0, qa); qb = fmaf(w1, w1, qb); qa = fmaf(w2, w2, qa); qb = fmaf(w3, w3, qb);
    }
    p0 = q[0] + q[1]; p1 = q[2] + q[3];
  }
}
__device__ __forceinline__ void accm_begin(SmemCtl& S, AccRing& ring, uint32_t tbase, uint32_t (&a0)[32]) {
  mbar_wait(&S.acc_full[ring.slot], ring.phase);
  tc_fence_after();
  tmem_ld32u(tbase + ring.slot * kAccCols, a0);
  tmem_wait_ld();
}
template <bool kInt8, bool kScore>
__device__ __forceinline__ void accm_step(SmemCtl& S, AccRing& ring, uint32_t tbase, int lane, uint32_t (&a0)[32],
                                          uint32_t (&a1)[32], float (&r)[64], const float4* gp, const float4 sc,
                                          float (&p)[4], const bool has_next, const bool skip_math) {
  const uint32_t t0 = tbase + ring.slot * kAccCols;
  uint32_t nslot = ring.slot + 1, nphase = ring.phase;
  if (nslot == ring.nslots) { nslot = 0; nphase ^= 1; }
  if (skip_math) {                 // debug mode 2: handshakes only
    p[0] = p[1] = p[2] = p[3] = 0.f;
    tc_fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive(&S.acc_empty[ring.slot]);
    ring.slot = nslot; ring.phase = nphase;
    if (has_next) { mbar_wait(&S.acc_full[ring.slot], ring.phase); tc_fence_after(); }
    return;
  }
  bool next_ready = true;
  if (has_next) next_ready = mbar_try(smem_u32(&S.acc_full[nslot]), nphase);
  tmem_ld32u(t0 + 32, a1);
  consume32<kInt8, kScore, 0>(a0, r, gp, sc.x, sc.y, p[0], p[1]);
  tmem_wait_ld();
  tc_fence_before();
  __syncwarp();
  if (lane == 0) mbar_arrive(&S.acc_empty[ring.slot]);      // one arrival per epilogue warp
  ring.slot = nslot; ring.phase = nphase;
  if (has_next) {
    if (!next_ready) mbar_wait(&S.acc_full[nslot], nphase);
    tc_fence_after();
    tmem_ld32u(tbase + nslot * kAccCols, a0);
  }
  consume32<kInt8, kScore, 32>(a1, r, gp, sc.z, sc.w, p[2], p[3]);
  if (has_next) tmem_wait_ld();
}

template <bool kInt8, bool kSingle>
__global__ void __launch_bounds__(kThreads, 1) sweep_tc_kernel(const __grid_constant__ SweepParams P) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 127) & ~uintptr_t(127));
  // carve: [ring R stages][ring C stages][resident R x2][control]
  const uint32_t sR = P.stage_r_bytes, sC = P.stage_c_bytes, nst = P.n_stages, resB = P.resident_bytes, cresB = P.cres_bytes;
  const uint32_t ringR = smem_u32(smem), ringC = ringR + nst * sR, resR = ringC + nst * sC, resC = resR + P.resident_bufs * resB;
  const size_t ctl_off = (size_t)nst * (sR + sC) + (size_t)P.resident_bufs * resB + cresB;
  SmemCtl& S = *reinterpret_cast<SmemCtl*>(smem + ctl_off);
  [[maybe_unused]] float* const red = reinterpret_cast<float*>(smem + ctl_off + ((sizeof(SmemCtl) + 127) & ~size_t(127)));
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  constexpr uint32_t kSlots = kSingle ? 4 : 3;            // single-segment steps do not park the target in TMEM
  constexpr uint32_t kAccBase = kSingle ? 0 : kAccCols;

  // ---- one-time setup ----
  const int n_jobs = P.n_fixed_jobs + P.n_cand_jobs;
  for (int i = threadIdx.x; i < n_jobs; i += kThreads) S.jobs[i] = P.jobs[i];
  if (threadIdx.x == 0) {
    for (uint32_t i = 0; i < nst; ++i) { mbar_init(&S.full[i], 1); mbar_init(&S.empty[i], 1); }
    for (int i = 0; i < 4; ++i) { mbar_init(&S.acc_full[i], 1); mbar_init(&S.acc_empty[i], kEpiWarps); }
    for (int i = 0; i < 2; ++i) { mbar_init(&S.res_full[i], 1); mbar_init(&S.res_empty[i], 1); }
    mbar_init(&S.cres_full, 1); mbar_init(&S.cres_empty, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&S.tmem_base)), "n"(kTmemCols));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = S.tmem_base;

  Sched sched; sched_init(P, sched);
  Frag f;

  if (warp < 4) {
  asm volatile("setmaxnreg.dec.sync.aligned.u32 56;");
  if (warp == 0) {
    // ======================= TMA producer (whole warp runs the loop, one elected lane issues) =======================
    // Single-warp loop: every instruction is on the critical path of a ~100-instruction-per-job budget, so addresses
    // are advanced incrementally and barrier / stage addresses are plain 32-bit shared-memory offsets.
    {
      uint32_t stage = 0, phase = 0, rbuf = 0, rphase = 0, cphase = 0;
      [[maybe_unused]] int tev = 0;
      const uint32_t full0 = smem_u32(&S.full[0]), empty0 = smem_u32(&S.empty[0]);
      while (!(DBG_MODE(P) & 1) && next_frag(P, sched, f)) {
        const size_t rt = P.R_shared ? (size_t)f.tm : (size_t)(f.p * P.tiles_m + f.tm), ct = (size_t)(f.p * P.tiles_n + f.tn);
        const uint8_t* r_cur = P.R_cur + rt * P.R_tile_bytes;
        const uint8_t* c_cur = P.C_cur + ct * P.C_tile_bytes;
        if (cresB) {     // the tile's whole current column image: once per fragment (single buffer: wait for the previous tile's MMAs)
          mbar_wait(&S.cres_empty, cphase ^ 1);
          if (elect_one()) {
            mbar_expect_tx(&S.cres_full, cresB);
            for (uint32_t o = 0; o < cresB; o += 32768u)
              bulk_g2s(resC + o, c_cur + o, (cresB - o < 32768u) ? cresB - o : 32768u, &S.cres_full);
          }
          cphase ^= 1;
        }
        if (resB) {      // row operand of the candidate jobs: once per fragment, reused by every candidate
          mbar_wait(&S.res_empty[rbuf], rphase ^ 1);
          uint32_t total = 0;
          for (int j = 0; j < P.n_cand_jobs; ++j) total += p4v_job_bytes(S.jobs[P.n_fixed_jobs + j]);
          if (elect_one()) {
            mbar_expect_tx(&S.res_full[rbuf], total);
            for (int j = 0; j < P.n_cand_jobs; ++j) {
              const P4VJob jb = S.jobs[P.n_fixed_jobs + j];
              bulk_g2s(resR + rbuf * resB + jb.res_off, r_cur + jb.r_off, p4v_job_bytes(jb), &S.res_full[rbuf]);
            }
          }
          if (++rbuf == P.resident_bufs) { rbuf = 0; rphase ^= 1; }
        }
        auto issue = [&](const P4VJob j, const uint8_t* rr, const uint8_t* cc) {
          TRACE(0, tev, 0);
          mbar_wait_addr(empty0 + stage * 8, phase ^ 1);
          TRACE(0, tev, 1);
          const uint32_t bytes = p4v_job_bytes(j);
          if (elect_one()) {
            const uint32_t fb = full0 + stage * 8;
            const uint32_t nload = ((j.flags & P4V_JOB_RRES) ? 0u : 1u) + ((j.flags & P4V_JOB_CRES) ? 0u : 1u);
            mbar_expect_tx_addr(fb, nload * bytes);
            if (!(j.flags & P4V_JOB_RRES)) bulk_g2s_addr(ringR + stage * sR, rr + j.r_off, bytes, fb);
            if (!(j.flags & P4V_JOB_CRES)) bulk_g2s_addr(ringC + stage * sC, cc + j.c_off, bytes, fb);
          }
          TRACE(0, tev, 2); ++tev;
          if (++stage == nst) { stage = 0; phase ^= 1; }
        };
        for (int j = 0; j < P.n_fixed_jobs; ++j) issue(S.jobs[j], r_cur, c_cur);
        const uint8_t* r_cand = P.R_cand + rt * P.R_cand_tile_bytes + (size_t)f.c0 * P.R_cand_stride;
        const uint8_t* c_cand = P.C_cand + ct * P.C_cand_tile_bytes + (size_t)f.c0 * P.C_cand_stride;
        if (P.n_cand_jobs == 1) {              // the common single-slab step: the job is loop invariant
          const P4VJob j = S.jobs[P.n_fixed_jobs];
          const uint8_t* rr = (j.flags & P4V_JOB_RCAND) ? r_cand : r_cur;
          const uint8_t* cc = (j.flags & P4V_JOB_CCAND) ? c_cand : c_cur;
          const size_t rstep = (j.flags & P4V_JOB_RCAND) ? P.R_cand_stride : 0, cstep = (j.flags & P4V_JOB_CCAND) ? P.C_cand_stride : 0;
          for (int c = f.c0; c < f.c1; ++c) { issue(j, rr, cc); rr += rstep; cc += cstep; }
        } else {
          for (int c = f.c0; c < f.c1; ++c) {
            for (int jj = 0; jj < P.n_cand_jobs; ++jj) {
              const P4VJob j = S.jobs[P.n_fixed_jobs + jj];
              issue(j, (j.flags & P4V_JOB_RCAND) ? r_cand : r_cur, (j.flags & P4V_JOB_CCAND) ? c_cand : c_cur);
            }
            r_cand += P.R_cand_stride; c_cand += P.C_cand_stride;
          }
        }
      }
    }
  } else if (warp == 1) {
    // ======================= MMA issuer (whole warp runs the loop, one elected lane issues) =======================
    {
      uint32_t stage = 0, phase = 0, slot = 0, slot_phase = 0, rbuf = 0, rphase = 0;
      const uint32_t full0 = smem_u32(&S.full[0]), empty0 = smem_u32(&S.empty[0]);
      const uint32_t accf0 = smem_u32(&S.acc_full[0]), acce0 = smem_u32(&S.acc_empty[0]);
      const uint64_t dconst = desc_hi_const();
      const uint32_t sR16 = sR >> 4, sC16 = sC >> 4, ringR16 = (ringR & 0x3FFFF) >> 4, ringC16 = (ringC & 0x3FFFF) >> 4;
      // one job: wait (slot if FIRST, stage), K-steps into TMEM slot, hand the stage back, publish the accumulator if LAST
      [[maybe_unused]] int tev = 0;
      uint32_t cphase = 0;
      const uint32_t resC16 = (resC & 0x3FFFF) >> 4;
      // one job = one stage: wait for its bytes, then per sub-accumulator (slot if FIRST, K-steps, publish if LAST);
      // the stage goes back to the producer with the last sub-accumulator
      auto run = [&](const P4VJob jb, const uint32_t ra16) {
        const uint32_t flags = jb.flags, kb = jb.kb, nsub = p4v_job_nsub(jb);
        TRACE(1, tev, 0);
        if (!(DBG_MODE(P) & 1)) mbar_wait_addr(full0 + stage * 8, phase);
        TRACE(1, tev, 1);
        tc_fence_after();
        uint32_t a16 = (flags & P4V_JOB_RRES) ? ra16 : ringR16 + stage * sR16;
        uint32_t b16 = (flags & P4V_JOB_CRES) ? resC16 + (jb.c_off >> 4) : ringC16 + stage * sC16;
        for (uint32_t sub = 0; sub < nsub; ++sub) {
          if (flags & P4V_JOB_FIRST) mbar_wait_addr(acce0 + slot * 8, slot_phase ^ 1);
          TRACE(1, tev, 2);
          if (DBG_MODE(P) & 1) {
            if ((flags & P4V_JOB_LAST) && elect_one()) tc_commit_addr(accf0 + slot * 8);
          } else if (elect_one()) {
            const uint64_t da = dconst | (uint64_t)a16, db = dconst | (uint64_t)b16;
            const uint32_t d = tmem + kAccBase + slot * kAccCols;
            umma<kInt8>(d, da, db, (flags & P4V_JOB_FIRST) ? 0u : 1u);
            if (kb > 32) umma<kInt8>(d, da + 256, db + 256, 1u);
            if (kb > 64) umma<kInt8>(d, da + 512, db + 512, 1u);
            if (kb > 96) umma<kInt8>(d, da + 768, db + 768, 1u);
            if (sub + 1 == nsub) tc_commit_addr(empty0 + stage * 8);
            if (flags & P4V_JOB_LAST) tc_commit_addr(accf0 + slot * 8);
          }
          a16 += kb * 8; b16 += kb * 8;        // kb * 128 bytes, in 16-byte units
          if (flags & P4V_JOB_LAST) { if (++slot == kSlots) { slot = 0; slot_phase ^= 1; } }
        }
        TRACE(1, tev, 3); ++tev;
        if (++stage == nst) { stage = 0; phase ^= 1; }
      };
      while (next_frag(P, sched, f)) {
        if (cresB) { if (!(DBG_MODE(P) & 1)) mbar_wait(&S.cres_full, cphase); cphase ^= 1; }
        for (int j = 0; j < P.n_fixed_jobs; ++j) run(S.jobs[j], 0u);
        uint32_t res16 = 0;
        if (resB) {
          if (!(DBG_MODE(P) & 1)) mbar_wait(&S.res_full[rbuf], rphase);
          res16 = ((resR + rbuf * resB) & 0x3FFFF) >> 4;
        }
        if (P.n_cand_jobs == 1) {              // loop-invariant job: keep its fields in registers
          const P4VJob jb = S.jobs[P.n_fixed_jobs];
          const uint32_t ra16 = res16 + (jb.res_off >> 4);
          for (int c = f.c0; c < f.c1; ++c) run(jb, ra16);
        } else {
          for (int c = f.c0; c < f.c1; ++c)
            for (int jj = 0; jj < P.n_cand_jobs; ++jj) {
              const P4VJob jb = S.jobs[P.n_fixed_jobs + jj];
              run(jb, res16 + (jb.res_off >> 4));
            }
        }
        if (resB) {
          if (!(DBG_MODE(P) & 1) && elect_one()) tc_commit(&S.res_empty[rbuf]);   // resident buffer free once every MMA reading it has retired
          if (++rbuf == P.resident_bufs) { rbuf = 0; rphase ^= 1; }
        }
        if (cresB && !(DBG_MODE(P) & 1) && elect_one()) tc_commit(&S.cres_empty);
      }
    }
  }
  } else {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 224;");
    // ======================= epilogue (8 warps) =======================
    const int ew = warp - 4;                 // 0..7
    const int quarter = warp & 3;            // TMEM lane quarter this warp may access
    const int hf = ew >> 2;                  // column half
    const int et = threadIdx.x - 128;        // 0..255
    const uint32_t lane_addr = (uint32_t)(quarter * 32) << 16;
    const uint32_t tbase = tmem + lane_addr + kAccBase + hf * 64;       // this thread's columns of slot 0
    const uint32_t tstore = tmem + lane_addr + hf * 64;                 // parked residual target (!kSingle)
    const float gs = (P.out && !P.out_residual) ? 1.f : *P.gscale;
    AccRing ring{0u, 0u, kSlots};
    const bool dbg2 = DBG_MODE(P) & 2;
    [[maybe_unused]] int tev = 0;
    if constexpr (!kSingle) {
    // ---------------- several accumulators per candidate (or output mode) ----------------
    float r[64];
    uint32_t a0[32], a1[32];
    float4* const gp = reinterpret_cast<float4*>(red) + (size_t)(hf * 16) * P4V_TILE + quarter * 32 + lane;
    while (next_frag(P, sched, f)) {
      asm volatile("bar.sync 1, %0;" ::"n"(kEpiThreads));   // previous fragment done with the tables
      {
        const int sg0 = (P.sg_mode == P4V_SG_COLUMN) ? f.tn * P4V_TILE_CG : (f.p % P.nsg);
        const int sgs = (P.sg_mode == P4V_SG_COLUMN) ? 1 : 0;
        for (int i = et; i < P.n_fixed_groups * P4V_TILE_CG; i += kEpiThreads)
          S.fixs[i >> 3][i & 7] = P.fix_scale[(size_t)(i >> 3) * P.nsg + sg0 + (i & 7) * sgs];
        for (int i = et; i < P.n_cand_groups * P4V_TILE_CG; i += kEpiThreads)
          S.candB[i >> 3][i & 7] = P.candB[(size_t)(i >> 3) * P.nsg + sg0 + (i & 7) * sgs];
        for (int i = et + f.c0 * P4V_TILE_CG; i < f.c1 * P4V_TILE_CG; i += kEpiThreads)
          S.candA[i >> 3][i & 7] = P.candA[(size_t)(i >> 3) * P.nsg + sg0 + (i & 7) * sgs];
      }
      {   // residual target into registers, gradient tile (scaled) into this thread's shared-memory row
        const int gm = f.tm * P4V_TILE + quarter * 32 + lane;
        const int col0 = f.tn * P4V_TILE + hf * 64;
        const float* yrow = P.Y + (size_t)f.p * P.prob_stride + (size_t)gm * P.ld;
        const float* grow = P.Gr + (size_t)f.p * P.prob_stride + (size_t)gm * P.ld;
        const bool row_ok = gm < P.M;
        if (P.out != nullptr && !P.out_residual) {           // quant_forward: r starts at -bias, output = -r
#pragma unroll
          for (int j = 0; j < 64; ++j) r[j] = (P.bias && col0 + j < P.N) ? -P.bias[col0 + j] : 0.f;
        } else if (row_ok && (P.ld & 3) == 0 && (P.prob_stride & 3) == 0 && col0 + 64 <= P.N) {
#pragma unroll
          for (int j = 0; j < 64; j += 4) {
            const float4 yv = *reinterpret_cast<const float4*>(yrow + col0 + j);
            const float4 bv = P.bias ? *reinterpret_cast<const float4*>(P.bias + col0 + j) : make_float4(0.f, 0.f, 0.f, 0.f);
            r[j] = yv.x - bv.x; r[j + 1] = yv.y - bv.y; r[j + 2] = yv.z - bv.z; r[j + 3] = yv.w - bv.w;
            if (P.out == nullptr) {
              const float4 gv = *reinterpret_cast<const float4*>(grow + col0 + j);
              gp[(j >> 2) * P4V_TILE] = make_float4(gv.x * gs, gv.y * gs, gv.z * gs, gv.w * gs);
            }
          }
        } else {
#pragma unroll
          for (int j = 0; j < 64; j += 4) {
            float gq[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const int col = col0 + j + k;
              const bool ok = row_ok && col < P.N;
              r[j + k] = ok ? (yrow[col] - (P.bias ? P.bias[col] : 0.f)) : 0.f;
              gq[k] = (ok && P.out == nullptr) ? grow[col] * gs : 0.f;
            }
            if (P.out == nullptr) gp[(j >> 2) * P4V_TILE] = make_float4(gq[0], gq[1], gq[2], gq[3]);
          }
        }
      }
      asm volatile("bar.sync 1, %0;" ::"n"(kEpiThreads));   // tables visible
      float p[4] = {0.f, 0.f, 0.f, 0.f};
      if (P.n_fixed_groups > 0) {
        accm_begin(S, ring, tbase, a0);
        for (int gi = 0; gi < P.n_fixed_groups; ++gi) {
          const float4 sc = *reinterpret_cast<const float4*>(&S.fixs[gi][hf * 4]);
          accm_step<kInt8, false>(S, ring, tbase, lane, a0, a1, r, gp, sc, p, gi + 1 < P.n_fixed_groups, dbg2);
        }
      }
      if (P.out != nullptr) {
        const int gm = f.tm * P4V_TILE + quarter * 32 + lane;
        const int col0 = f.tn * P4V_TILE + hf * 64;
        if (gm < P.M) {
          float* orow = P.out + (size_t)f.p * P.prob_stride + (size_t)gm * P.ld;
#pragma unroll
          for (int j = 0; j < 64; ++j) if (col0 + j < P.N) orow[col0 + j] = P.out_residual ? r[j] : -r[j];
        }
        continue;
      }
      float* part_base = P.partial + ((size_t)f.tile * P.n_cand) * 32 + quarter * 8 + hf * 4;
      // park the residual target in TMEM columns [0,128); every candidate starts from it
      tmem_st32(tstore, r);
      tmem_st32(tstore + 32, r + 32);
      tmem_wait_st();
      if (f.c1 > f.c0) accm_begin(S, ring, tbase, a0);       // later candidates: prefetched by the previous candidate's last step
      for (int c = f.c0; c < f.c1; ++c) {
        const float4 ca = *reinterpret_cast<const float4*>(&S.candA[c][hf * 4]);
        tmem_ld32f(tstore, r);
        tmem_ld32f(tstore + 32, r + 32);
        tmem_wait_ld();
        for (int gi = 0; gi < P.n_cand_groups; ++gi) {
          const float4 cb = *reinterpret_cast<const float4*>(&S.candB[gi][hf * 4]);
          const bool noA = (P.cand_noA_mask >> gi) & 1ull;
          const float4 sc = noA ? cb : make_float4(ca.x * cb.x, ca.y * cb.y, ca.z * cb.z, ca.w * cb.w);
          if (ew == 0) TRACE(2, tev, 0);
          if (gi == P.n_cand_groups - 1) accm_step<kInt8, true>(S, ring, tbase, lane, a0, a1, r, gp, sc, p, c + 1 < f.c1, dbg2);
          else accm_step<kInt8, false>(S, ring, tbase, lane, a0, a1, r, gp, sc, p, true, dbg2);
          if (ew == 0) { TRACE(2, tev, 1); ++tev; }
        }
        const float tot = reduce4_over_rows(p[0], p[1], p[2], p[3], lane);
        if ((lane & 7) == 0) part_base[(size_t)c * 32 + (lane >> 3)] = tot;
      }
    }
    } else {
    // ---------------- one accumulator per candidate ----------------
    float r[64], g[64];
    uint32_t a0[16], a1[16];

    while (next_frag(P, sched, f)) {
      // -- scale tables for this tile's 8 column groups --
      asm volatile("bar.sync 1, %0;" ::"n"(kEpiThreads));   // previous fragment done with the tables
      {
        const int sg0 = (P.sg_mode == P4V_SG_COLUMN) ? f.tn * P4V_TILE_CG : (f.p % P.nsg);
        const int sgs = (P.sg_mode == P4V_SG_COLUMN) ? 1 : 0;
        for (int i = et; i < P.n_fixed_groups * P4V_TILE_CG; i += kEpiThreads)
          S.fixs[i >> 3][i & 7] = P.fix_scale[(size_t)(i >> 3) * P.nsg + sg0 + (i & 7) * sgs];
        for (int i = et; i < P.n_cand_groups * P4V_TILE_CG; i += kEpiThreads)
          S.candB[i >> 3][i & 7] = P.candB[(size_t)(i >> 3) * P.nsg + sg0 + (i & 7) * sgs];
        for (int i = et + f.c0 * P4V_TILE_CG; i < f.c1 * P4V_TILE_CG; i += kEpiThreads)
          S.candA[i >> 3][i & 7] = P.candA[(size_t)(i >> 3) * P.nsg + sg0 + (i & 7) * sgs];
      }
      // -- residual target and gradient tile into registers --
      {
        const int gm = f.tm * P4V_TILE + quarter * 32 + lane;
        const int col0 = f.tn * P4V_TILE + hf * 64;
        const float* yrow = P.Y + (size_t)f.p * P.prob_stride + (size_t)gm * P.ld;
        const float* grow = P.Gr + (size_t)f.p * P.prob_stride + (size_t)gm * P.ld;
        const bool row_ok = gm < P.M;
        if (P.out != nullptr && !P.out_residual) {           // quant_forward: r starts at -bias, output = -r
#pragma unroll
          for (int j = 0; j < 64; ++j) {
            const int col = col0 + j;
            r[j] = (P.bias && col < P.N) ? -P.bias[col] : 0.f;
            g[j] = 0.f;
          }
        } else if (row_ok && (P.ld & 3) == 0 && (P.prob_stride & 3) == 0 && col0 + 64 <= P.N) {
#pragma unroll
          for (int j = 0; j < 64; j += 4) {
            float4 yv = *reinterpret_cast<const float4*>(yrow + col0 + j);
            float4 gv = *reinterpret_cast<const float4*>(grow + col0 + j);
            float4 bv = P.bias ? *reinterpret_cast<const float4*>(P.bias + col0 + j) : make_float4(0.f, 0.f, 0.f, 0.f);
            r[j] = yv.x - bv.x; r[j + 1] = yv.y - bv.y; r[j + 2] = yv.z - bv.z; r[j + 3] = yv.w - bv.w;
            g[j] = gv.x * gs; g[j + 1] = gv.y * gs; g[j + 2] = gv.z * gs; g[j + 3] = gv.w * gs;
          }
        } else {
#pragma unroll
          for (int j = 0; j < 64; ++j) {
            const int col = col0 + j;
            const bool ok = row_ok && col < P.N;
            r[j] = ok ? (yrow[col] - (P.bias ? P.bias[col] : 0.f)) : 0.f;
            g[j] = ok ? grow[col] * gs : 0.f;
          }
        }
      }
      asm volatile("bar.sync 1, %0;" ::"n"(kEpiThreads));   // tables visible

      // -- fixed segments: r -= scale * acc --
      float pdummy[4];
      if (P.n_fixed_groups > 0) {
        acc_begin(S, ring, tbase, a0);
        for (int gi = 0; gi < P.n_fixed_groups; ++gi) {
          const float4 sc = *reinterpret_cast<const float4*>(&S.fixs[gi][hf * 4]);
          acc_step<kInt8, false>(S, ring, tbase, lane, a0, a1, r, g, sc, pdummy, gi + 1 < P.n_fixed_groups, dbg2);
        }
      }
      if (P.out != nullptr) {
        const int gm = f.tm * P4V_TILE + quarter * 32 + lane;
        const int col0 = f.tn * P4V_TILE + hf * 64;
        if (gm < P.M) {
          float* orow = P.out + (size_t)f.p * P.prob_stride + (size_t)gm * P.ld;
#pragma unroll
          for (int j = 0; j < 64; ++j) if (col0 + j < P.N) orow[col0 + j] = P.out_residual ? r[j] : -r[j];
        }
        continue;
      }
      float* const part_base_tile = P.partial + ((size_t)f.tile * P.n_cand) * 32;

      {
        // -- one accumulator per candidate --
        if (f.c1 > f.c0) acc_begin(S, ring, tbase, a0);
        const float4 cb = *reinterpret_cast<const float4*>(&S.candB[0][hf * 4]);
        const bool noA = P.cand_noA_mask & 1ull;
        // my slot in the reduction buffers (writer) and my (candidate, row quarter, group) task (reader)
        float* const red_w = red + hf * kRedHalf + (quarter * 32 + lane) * 4;
        const int rd_j = et >> 5, rd_q = (et >> 3) & 3, rd_g = et & 7;
        const float* const red_r = red + rd_j * kRedCand + (rd_g >> 2) * kRedHalf + (rd_q * 32) * 4 + (rd_g & 3);
        int nb = 0, buf = 0;
        for (int c = f.c0; c < f.c1; ++c) {
          float p[4];
          if (ew == 0) TRACE(2, tev, 0);
          const float4 ca = *reinterpret_cast<const float4*>(&S.candA[c][hf * 4]);
          const float4 sc = noA ? cb : make_float4(ca.x * cb.x, ca.y * cb.y, ca.z * cb.z, ca.w * cb.w);
          acc_step<kInt8, true>(S, ring, tbase, lane, a0, a1, r, g, sc, p, c + 1 < f.c1, dbg2);
          if (ew == 0) TRACE(2, tev, 1);
          if (P.row_keys) {        // one score per ROW (channel-wise conv search): [tile][candidate][column half][128 rows]
            P.partial[((size_t)f.tile * P.n_cand + c) * 256 + hf * P4V_TILE + quarter * 32 + lane] = (p[0] + p[1]) + (p[2] + p[3]);
            continue;
          }
          *reinterpret_cast<float4*>(red_w + (buf * kRedBatch + nb) * kRedCand) = make_float4(p[0], p[1], p[2], p[3]);
          if (ew == 0) TRACE(2, tev, 2);
          if (++nb == kRedBatch || c + 1 == f.c1) {
            asm volatile("bar.sync 1, %0;" ::"n"(kEpiThreads));
            if (rd_j < nb) {                       // sum 32 rows; the start row is rotated per quarter (bank spread)
              const float* src = red_r + buf * kRedBatch * kRedCand;
              float t0 = 0.f, t1 = 0.f;
#pragma unroll
              for (int i = 0; i < 32; i += 2) {
                t0 += src[((i + 2 * rd_q) & 31) * 4];
                t1 += src[((i + 1 + 2 * rd_q) & 31) * 4];
              }
              part_base_tile[(size_t)(c + 1 - nb + rd_j) * 32 + (et & 31)] = t0 + t1;
            }
            buf ^= 1; nb = 0;
          }
          if (ew == 0) { TRACE(2, tev, 3); ++tev; }
        }
      }
    }
  }

    }
  // ---- teardown ----
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "n"(kTmemCols));
  }
}

}  // namespace

// debug hook (not part of the public header): 1 = no operand traffic / MMA, 2 = no epilogue math; initialised from P4V_SWEEP_DEBUG
static int g_sweep_debug = [] { const char* e = getenv("P4V_SWEEP_DEBUG"); return e ? atoi(e) : 0; }();
extern "C" __attribute__((visibility("default"))) int p4v_debug_sweep_mode(int mode) { g_sweep_debug = mode; return 0; }

int p4v_launch_sweep_tc(const SweepParams& p_in, const P4VJob* host_jobs, int num_sms, cudaStream_t st) {
  SweepParams p = p_in;
  const int n_jobs = p.n_fixed_jobs + p.n_cand_jobs;
  P4V_REQUIRE(n_jobs <= P4V_MAX_JOBS, "sweep: too many jobs (%d)", n_jobs);
  P4V_REQUIRE(p.n_fixed_groups <= P4V_MAX_GROUPS && p.n_cand_groups <= P4V_MAX_GROUPS, "sweep: too many segment groups");
  P4V_REQUIRE(p.n_cand <= P4V_MAX_CAND && p.n_cand >= 1, "sweep: bad candidate count");
  P4V_REQUIRE(p.out != nullptr ? (p.n_cand == 1 && p.n_cand_jobs == 0) : p.n_cand_groups >= 1, "sweep: bad mode");
  P4V_REQUIRE(!p.row_keys || (p.n_cand_groups == 1 && p.out == nullptr), "sweep: per-row scores need a single-segment step");
  const long long tiles = (long long)p.P * p.tiles_m * p.tiles_n;
  const long long units = tiles * p.n_cand;
  int grid = (int)(units < num_sms ? units : num_sms);
  if (grid < 1) return 0;
  // smem plan: stage size = largest job; resident row operand when the host marked the candidate jobs P4V_JOB_RRES
  uint32_t max_kb = 32, res_bytes = 0;
  bool any_r_stream = false, any_c_stream = false, any_cres = false;
  for (int j = 0; j < n_jobs; ++j) {
    const uint32_t kb_total = host_jobs[j].kb * p4v_job_nsub(host_jobs[j]);
    P4V_REQUIRE(host_jobs[j].kb % 32 == 0 && kb_total >= 32 && kb_total <= P4V_JOB_KB, "sweep: bad job size");
    if (kb_total > max_kb) max_kb = kb_total;
    if (host_jobs[j].flags & P4V_JOB_RRES) res_bytes = std::max(res_bytes, host_jobs[j].res_off + kb_total * P4V_TILE);
    else any_r_stream = true;
    if (host_jobs[j].flags & P4V_JOB_CRES) any_cres = true; else any_c_stream = true;
  }
  p.stage_r_bytes = any_r_stream ? max_kb * P4V_TILE : 0;
  p.stage_c_bytes = any_c_stream ? max_kb * P4V_TILE : 0;
  p.resident_bytes = res_bytes;
  p.cres_bytes = any_cres ? (unsigned int)p.C_tile_bytes : 0;
  P4V_REQUIRE(p.cres_bytes % 16 == 0 && p.cres_bytes <= 128 * 1024, "sweep: resident column image too large");
  const uint32_t per_stage = p.stage_r_bytes + p.stage_c_bytes;
  P4V_REQUIRE(per_stage > 0, "sweep: no streamed operand");
  const bool single = p.n_cand_groups == 1 && p.out == nullptr;
  const long long red_bytes = single ? kRedBytes : (p.out == nullptr ? (long long)P4V_TILE * P4V_TILE * 4 : 0);   // score reduction buffers / parked gradient tile
  p.resident_bufs = 2;                      // double buffered when that leaves a useful ring, else one buffer (a bubble per tile)
  if ((kSmemBudget - 2 * (long long)res_bytes - red_bytes - (long long)p.cres_bytes) / per_stage < 3) p.resident_bufs = 1;
  int nst = (int)((kSmemBudget - (long long)p.resident_bufs * res_bytes - red_bytes - (long long)p.cres_bytes) / per_stage);
  if (nst > kMaxStages) nst = kMaxStages;
  P4V_REQUIRE(nst >= 2, "sweep: operand tiles do not fit the shared-memory ring");
  p.n_stages = nst;
  const size_t smem = (size_t)nst * per_stage + (size_t)p.resident_bufs * res_bytes + p.cres_bytes + ((sizeof(SmemCtl) + 127) & ~size_t(127)) + (size_t)red_bytes + 256;
#define P4V_LAUNCH(I8, SG)                                                                             \
  do {                                                                                                 \
    P4V_CUDA_OK(cudaFuncSetAttribute(sweep_tc_kernel<I8, SG>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
    sweep_tc_kernel<I8, SG><<<grid, kThreads, smem, st>>>(p);                                          \
  } while (0)
  p.debug_mode = g_sweep_debug;
  if (p.is_int8) { if (single) P4V_LAUNCH(true, true); else P4V_LAUNCH(true, false); }
  else           { if (single) P4V_LAUNCH(false, true); else P4V_LAUNCH(false, false); }
#undef P4V_LAUNCH
  P4V_CUDA_OK(cudaGetLastError());
  return 0;
}
