// Gram GEMM of the normal-equation weight search (gram.cu):   H[o][pair] = sum_m (gs*g[m,o])^2 * Xq[m,k] * Xq[m,k']
// for ALL column blocks of a search round in one launch.  Both operands are exact two-term bf16 splits
//   A = (gs*g)^2 = A_hi + A_lo   (rows = output channels, K = tokens; image of 128-row tiles)
//   Z = Xq_k*Xq_k' = Z_hi + Z_lo (rows = (block, pair),   K = tokens; image of 256-row tiles)
// and the product keeps the three significant combinations hi*hi + hi*lo + lo*hi, accumulated in ONE fp32 TMEM
// accumulator.  A stage of the shared-memory ring carries 64 bytes of K of all four term tiles, so every byte pulled
// from L2 feeds three tensor-core passes, and the 128x256 output tile halves the operand bytes per flop once more:
// 48 KB per 768 MMA cycles = 62 B/clk/SM (the per-step 128x128 three-pass version needed 125 B/clk/SM and ran at the
// L2->SM limit with 90 of 148 SMs).
// The tensor core adds into the fp32 accumulator with truncation, so a long contraction of same-signed terms (the
// diagonal of H: 6304 tokens x 3 products) drifts by ~1e-5 relative (measured against an fp64 evaluation; it was the
// whole 2e-5..2e-4 score error of the normal-equation steps).  The contraction is therefore cut into splits of
// `kSplitChunks` stages (256 tokens): each split accumulates in its own TMEM slot and the epilogue adds the splits in
// registers with round-to-nearest fp32 adds.  The epilogue pass of a split (128 columns per thread) takes ~300 cycles
// against ~6000 cycles of MMAs per split.
// Roles: warp 0 = bulk-copy producer, warp 1 = MMA issuer (+TMEM alloc), warps 2..9 = epilogue (TMEM -> registers -> H).
#include "gram.cuh"
#include <cstdio>

namespace {

constexpr int kThreads = 64 + 256;
constexpr int kSplitChunks = 8;                                     // stages (64 B of K = 32 tokens each) per accumulation split
constexpr int kStages = 4;
constexpr uint32_t kStageKB = 64;                                   // bytes of K per row and stage
constexpr uint32_t kRTerm = kStageKB * 128, kCTerm = kStageKB * 256;  // bytes of one term tile in a stage
constexpr uint32_t kStageBytes = 2 * kRTerm + 2 * kCTerm;            // 48 KB
constexpr uint32_t kAccCols = 256, kTmemCols = 512;

struct Ctl {
  alignas(8) unsigned long long full[kStages], empty[kStages], acc_full[2], acc_empty[2];
  uint32_t tmem_base;
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ void mbar_init(void* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ bool mbar_try(uint32_t addr, uint32_t parity) {
  uint32_t ok;
  asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
               : "=r"(ok) : "r"(addr), "r"(parity) : "memory");
  return ok != 0;
}
__device__ __noinline__ void mbar_wait_slow(uint32_t addr, uint32_t parity) {     // bounded: a protocol bug traps, never hangs
  const long long t0 = clock64();
  while (!mbar_try(addr, parity))
    if (clock64() - t0 > 20000000000ll) {
      printf("ptq4vit_b200 gram gemm: mbarrier wait timed out (block %d thread %d smem 0x%x parity %u)\n", (int)blockIdx.x,
             (int)threadIdx.x, addr, parity);
      __trap();
    }
}
__device__ __forceinline__ void mbar_wait(void* bar, uint32_t parity) {
  const uint32_t addr = smem_u32(bar);
  if (!mbar_try(addr, parity)) mbar_wait_slow(addr, parity);
}
__device__ __forceinline__ void mbar_arrive(void* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(void* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, void* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(dst), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
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
// K-major, no swizzle (same canonical layout as the sweep kernel): core matrix = 8 rows x 16 B, SBO = 128 B between
// 8-row groups, LBO = rows*16 B between the 16-byte K chunks of one tile.
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t rows) {
  const uint64_t lbo = (rows * 16) >> 4, sbo = 128 >> 4;
  return (uint64_t)((saddr & 0x3FFFF) >> 4) | (lbo << 16) | (sbo << 32) | (1ull << 46);
}
__device__ __forceinline__ void umma_bf16_n256(uint32_t d_tmem, uint64_t da, uint64_t db, uint32_t accumulate) {
  // c_format F32 @4, a/b BF16 @7/@10, K-major both, N>>3 @17, M>>4 @24
  constexpr uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((256u >> 3) << 17) | ((128u >> 4) << 24);
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
               "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
               ::"r"(d_tmem), "l"(da), "l"(db), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float* v) {
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
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

__global__ void __launch_bounds__(kThreads, 1) gram_gemm_kernel(const __grid_constant__ GramGemmArgs a) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 127) & ~uintptr_t(127));
  Ctl& S = *reinterpret_cast<Ctl*>(smem + (size_t)kStages * kStageBytes);
  const uint32_t ring = smem_u32(smem);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int i = 0; i < kStages; ++i) { mbar_init(&S.full[i], 1); mbar_init(&S.empty[i], 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(&S.acc_full[i], 1); mbar_init(&S.acc_empty[i], 8); }
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
  const int tiles = a.tiles_o * a.tiles_p;
  const uint32_t term = a.term_bytes;
  const int n_chunks = (int)((term + kStageKB - 1) / kStageKB);

  if (warp == 0) {
    // ---------------- producer ----------------
    uint32_t stage = 0, phase = 0;
    for (int t = blockIdx.x; t < tiles; t += gridDim.x) {
      const uint8_t* rt = a.R + (size_t)(t % a.tiles_o) * a.R_tile_bytes;
      const uint8_t* ct = a.C + (size_t)(t / a.tiles_o) * a.C_tile_bytes;
      for (int ch = 0; ch < n_chunks; ++ch) {
        const uint32_t k0 = ch * kStageKB, kb = (term - k0 < kStageKB) ? term - k0 : kStageKB;
        mbar_wait(&S.empty[stage], phase ^ 1);
        if (elect_one()) {
          const uint32_t s0 = ring + stage * kStageBytes;
          mbar_expect_tx(&S.full[stage], kb * (2 * 128 + 2 * 256));
          bulk_g2s(s0, rt + (size_t)k0 * 128, kb * 128, &S.full[stage]);
          bulk_g2s(s0 + kRTerm, rt + ((size_t)term + k0) * 128, kb * 128, &S.full[stage]);
          bulk_g2s(s0 + 2 * kRTerm, ct + (size_t)k0 * 256, kb * 256, &S.full[stage]);
          bulk_g2s(s0 + 2 * kRTerm + kCTerm, ct + ((size_t)term + k0) * 256, kb * 256, &S.full[stage]);
        }
        if (++stage == kStages) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    // ---------------- MMA issuer ----------------
    uint32_t stage = 0, phase = 0, slot = 0, sphase = 0;
    for (int t = blockIdx.x; t < tiles; t += gridDim.x) {
      for (int ch = 0; ch < n_chunks; ++ch) {
        const bool first = ch % kSplitChunks == 0, last = (ch % kSplitChunks == kSplitChunks - 1) || ch == n_chunks - 1;
        if (first) mbar_wait(&S.acc_empty[slot], sphase ^ 1);
        const uint32_t d = tmem + slot * kAccCols;
        const uint32_t k0 = ch * kStageKB, kb = (term - k0 < kStageKB) ? term - k0 : kStageKB;
        mbar_wait(&S.full[stage], phase);
        tc_fence_after();
        if (elect_one()) {
          const uint32_t s0 = ring + stage * kStageBytes;
          const uint64_t rhi = make_desc(s0, 128), rlo = make_desc(s0 + kRTerm, 128);
          const uint64_t chi = make_desc(s0 + 2 * kRTerm, 256), clo = make_desc(s0 + 2 * kRTerm + kCTerm, 256);
          for (uint32_t ks = 0; ks * 32 < kb; ++ks) {          // one K step = 16 bf16 = two 16-byte chunks
            const uint64_t ra = ks * ((2u * 128 * 16) >> 4), ca = ks * ((2u * 256 * 16) >> 4);
            umma_bf16_n256(d, rhi + ra, chi + ca, (!first || ks) ? 1u : 0u);
            umma_bf16_n256(d, rhi + ra, clo + ca, 1u);
            umma_bf16_n256(d, rlo + ra, chi + ca, 1u);
          }
          tc_commit(&S.empty[stage]);
          if (last) tc_commit(&S.acc_full[slot]);
        }
        if (++stage == kStages) { stage = 0; phase ^= 1; }
        if (last) { if (++slot == 2) { slot = 0; sphase ^= 1; } }
      }
    }
  } else {
    // ---------------- epilogue: TMEM -> registers (sum of the splits) -> H ----------------
    const int quarter = warp & 3;                 // TMEM lane quarter this warp may access
    const int half = (warp - 2) >> 2;             // column half: 128 of the tile's 256 columns
    const int n_splits = (n_chunks + kSplitChunks - 1) / kSplitChunks;
    uint32_t slot = 0, sphase = 0;
    for (int t = blockIdx.x; t < tiles; t += gridDim.x) {
      const int o = (t % a.tiles_o) * 128 + quarter * 32 + lane;
      float* hrow = a.H + (size_t)o * a.ldH + (size_t)(t / a.tiles_o) * 256 + half * 128;
      float acc[128];
#pragma unroll
      for (int j = 0; j < 128; ++j) acc[j] = 0.f;
      for (int sp = 0; sp < n_splits; ++sp) {
        mbar_wait(&S.acc_full[slot], sphase);
        tc_fence_after();
        const uint32_t tb = tmem + ((uint32_t)(quarter * 32) << 16) + slot * kAccCols + half * 128;
#pragma unroll
        for (int c = 0; c < 128; c += 32) {
          float v[32];
          tmem_ld32(tb + c, v);
          tmem_wait_ld();
#pragma unroll
          for (int j = 0; j < 32; ++j) acc[c + j] += v[j];
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&S.acc_empty[slot]);
        if (++slot == 2) { slot = 0; sphase ^= 1; }
      }
      if (o < a.O) {
#pragma unroll
        for (int j = 0; j < 128; j += 4) *reinterpret_cast<float4*>(hrow + j) = make_float4(acc[j], acc[j + 1], acc[j + 2], acc[j + 3]);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "n"(kTmemCols));
  }
}

}  // namespace

int p4v_gram_gemm(const GramGemmArgs& a, cudaStream_t st) {
  P4V_REQUIRE(a.term_bytes % 32 == 0 && a.ldH % 4 == 0, "gram gemm: bad operand geometry");
  const int tiles = a.tiles_o * a.tiles_p;
  if (tiles < 1) return 0;
  const int grid = tiles < p4v_num_sms() ? tiles : p4v_num_sms();
  const size_t smem = (size_t)kStages * kStageBytes + sizeof(Ctl) + 256;
  P4V_CUDA_OK(cudaFuncSetAttribute(gram_gemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  cudaEvent_t e0 = nullptr;
  if (p4v_prof_on()) p4v_prof_begin(st, &e0);
  gram_gemm_kernel<<<grid, kThreads, smem, st>>>(a); p4v_count_launch();
  // three bf16 term products per (output channel, pair, token): 128x256 tiles over term_bytes/2 tokens
  if (p4v_prof_on()) p4v_prof_end(st, e0, P4V_PROF_GRAM_GEMM, 3.0 * 2.0 * 128.0 * 256.0 * (double)tiles * (double)(a.term_bytes / 2));
  P4V_CUDA_OK(cudaGetLastError());
  return 0;
}
