// Normal-equation ("Gram") form of the weight-step search for narrow column blocks.
//
// For column block h, row block v and candidate c the reference evaluates
//     score_c[v] = - sum_{m, o in v} ( g[m,o] * ( y[m,o] - yhat_c[m,o] ) )^2          (linear.py:417-423, :466-488)
// and yhat_c differs from the current quantised output only through the ks = K/n_H weights of block h:
//     y - yhat_c = e - xhat_h * (w_c - w_cur)^T ,   e = y - yhat_cur ,  xhat_h = fake-quantised x[:, block h].
// Expanding the square per output channel o with d = w_c[o,:] - w_cur[o,:] (ks numbers):
//     sum_m (g e)^2  -  2 d . U[o]  +  d^T H[o] d ,   U[o] = sum_m g^2 e xhat ,  H[o] = sum_m g^2 xhat xhat^T .
// All three terms are of the size of the quantisation error (no cancellation; fp32 reproduces the reference's
// score tables to 2e-7 on the CPU and <= 2.3e-5 on the GPU, see tests).  H is a contraction over the TOKENS, so it
// runs as ONE tensor-core GEMM per round, (g^2)^T[O x M] . Z[M x n_H*ks(ks+1)/2] (gram_gemm.cu; the activations do not
// change during the weight steps) -- the candidates never touch TMEM or HBM again: evaluating all eq_n candidates
// costs eq_n * O * ks^2/2 FMAs.  This removes the per-candidate accumulator hand-over (TMEM -> registers, three
// fp32 operations per output element) that bounds the slab sweep of narrow column blocks.
// This file: token-major activations, the pair image Z, the per-step update pass (e, U, sum (g e)^2), the candidate
// evaluation and the small reductions.
#include "gram.cuh"

namespace {

__device__ __forceinline__ float fq_dev(float w, float delta, float lo, float hi) {
  return fminf(fmaxf(rintf(__fdiv_rn(w, delta)), lo), hi) * delta;
}

// x [M][K] fp32 -> XqT [K][Mp] int8 (quantised with the current activation step sizes)
__global__ void xq_transpose_kernel(const float* __restrict__ x, int M, int K, int Mp, const float* __restrict__ dX,
                                    int crb_acts, float qlo, float qhi, int8_t* __restrict__ out) {
  __shared__ float tile[32][33];
  const int m0 = blockIdx.x * 32, k0 = blockIdx.y * 32;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int m = m0 + i, k = k0 + threadIdx.x;
    tile[i][threadIdx.x] = (m < M && k < K) ? x[(size_t)m * K + k] : 0.f;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int k = k0 + i, m = m0 + threadIdx.x;
    if (k < K && m < Mp) {
      float q = 0.f;
      if (m < M) {
        q = fminf(fmaxf(rintf(__fdiv_rn(tile[threadIdx.x][i], dX[k / crb_acts])), qlo), qhi);
        if (!(q == q)) q = 0.f;
      }
      out[(size_t)k * Mp + m] = (int8_t)(int)q;
    }
  }
}

// Z image: rows = (column block, pair k <= k' of the block), K = tokens; value = Xq[m,k] * Xq[m,k'] split exactly into two
// bf16 terms.  Layout [tile of 256 rows][chunk][256][16 B]; hi term at byte offset 0 of the padded row, lo term at term_bytes.
__global__ void pair_image_kernel(const int8_t* __restrict__ XqT, int Mp, int M, int k_first, int ks, int npairs, int n_blocks,
                                  int tiles_p, unsigned long long tile_bytes, unsigned int term_bytes, uint8_t* __restrict__ dst) {
  const int rows_pad = tiles_p * GRAM_PT;
  const int row = blockIdx.x * blockDim.x + threadIdx.x;        // (block, pair) index (padded)
  const int chunk = blockIdx.y;                                  // 8 tokens
  if (row >= rows_pad) return;
  uint32_t hi[4] = {0, 0, 0, 0}, lo[4] = {0, 0, 0, 0};
  if (row < npairs * n_blocks) {
    const int blk = row / npairs, pr = row % npairs;
    // invert p = k*ks - k(k-1)/2 + (k' - k)
    int k = 0, base = 0;
    while (base + (ks - k) <= pr) { base += ks - k; ++k; }
    const int k2 = k + (pr - base);
    const int8_t* a = XqT + (size_t)(k_first + blk * ks + k) * Mp + chunk * 8;
    const int8_t* b = XqT + (size_t)(k_first + blk * ks + k2) * Mp + chunk * 8;
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const int m = chunk * 8 + e;
      const float z = m < M ? (float)((int)a[e] * (int)b[e]) : 0.f;
      const __nv_bfloat16 h = __float2bfloat16_rn(z);
      const __nv_bfloat16 l = __float2bfloat16_rn(z - __bfloat162float(h));     // |z| < 2^15: two terms are exact
      hi[e >> 1] |= (uint32_t)__bfloat16_as_ushort(h) << ((e & 1) * 16);
      lo[e >> 1] |= (uint32_t)__bfloat16_as_ushort(l) << ((e & 1) * 16);
    }
  }
  const int tile = row / GRAM_PT, r = row % GRAM_PT;
  uint8_t* base_p = dst + (size_t)tile * tile_bytes + ((size_t)chunk * GRAM_PT + r) * 16;
  *reinterpret_cast<uint4*>(base_p) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
  *reinterpret_cast<uint4*>(base_p + (size_t)term_bytes * GRAM_PT) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
}

// packed fp32x2 math (sm_100): one issue slot per two FMAs
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 pack2(float a, float b) { f32x2 r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a), "f"(b)); return r; }
__device__ __forceinline__ void unpack2(f32x2 v, float& a, float& b) { asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v)); }
__device__ __forceinline__ f32x2 fma2(f32x2 a, f32x2 b, f32x2 c) { f32x2 d; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c)); return d; }

// D[o][k] = what the previous step's pick changed in the quantised weights of its column block (ks numbers per channel)
__global__ void gram_delta_kernel(const float* __restrict__ W, int O, int K, int k_prev, int ks, int ldD,
                                  const float* __restrict__ dW, const float* __restrict__ dW_prev, int n_V, int n_H, int crb_rows,
                                  int h_prev, float w_lo, float w_hi, float* __restrict__ D) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= O * ldD) return;
  const int o = i / ldD, k = i % ldD;
  float v = 0.f;
  if (k < ks) {
    const int vb = min(o / crb_rows, n_V - 1);
    const float w = W[(size_t)o * K + k_prev + k];
    v = fq_dev(w, dW[vb * n_H + h_prev], w_lo, w_hi) - fq_dev(w, dW_prev[vb], w_lo, w_hi);
  }
  D[i] = v;
}

// One pass over e and g: apply the rank-ks update of the previous step, accumulate U and sum (g e)^2 for the next slab.
// grid = (256-channel blocks) x (token splits, sized so that the grid is ONE balanced wave); a block walks its token
// range in chunks of GRAM_BM tokens and keeps the U accumulators of its channels in registers the whole time, so there
// is one partial per block.  thread = one output channel (16 warps per SM hide the e/g load latency better than
// two channels per thread at 8 warps); xhat values come from shared memory as broadcast 16-byte loads.
template <int KS>
__global__ void __launch_bounds__(256, 2) gram_update_kernel(const GramUpdateArgs a) {
  __shared__ __align__(16) float xp[GRAM_BM * KS];       // previous slab (xhat), only if a.h_prev >= 0
  __shared__ __align__(16) float xn[GRAM_BM * KS];       // next slab
  const int o = blockIdx.x * 256 + threadIdx.x;
  const bool ok_o = o < a.O;
  const float gs = a.gscale[0];
  const bool has_prev = a.h_prev >= 0;
  const int nb16 = (a.M + 15) / 16;                     // split on 16-token boundaries: the slab loads stay 16-byte aligned
  const int m_begin = (int)((long long)nb16 * blockIdx.y / gridDim.y) * 16;
  const int m_end = min(a.M, (int)((long long)nb16 * (blockIdx.y + 1) / gridDim.y) * 16);
  f32x2 dd[KS / 2], acc[KS / 2];
#pragma unroll
  for (int k = 0; k < KS / 2; ++k) { dd[k] = 0ull; acc[k] = 0ull; }
  if (has_prev && ok_o) {
#pragma unroll
    for (int k = 0; k < KS; k += 4) {
      const float4 v = *reinterpret_cast<const float4*>(a.D + (size_t)o * KS + k);
      dd[k / 2] = pack2(v.x, v.y); dd[k / 2 + 1] = pack2(v.z, v.w);
    }
  }
  float e2 = 0.f;
  for (int m0 = m_begin; m0 < m_end; m0 += GRAM_BM) {
    const int rows = min(GRAM_BM, m_end - m0);
    __syncthreads();                                      // previous chunk consumed
    // slab chunks of the token-major int8 activations -> fp32 xhat in shared memory ([token][k], k contiguous);
    // thread = (k, 16-token piece): one 16-byte load per slab row piece, conflict-free stores (lanes = consecutive k)
    for (int it = threadIdx.x; it < KS * (GRAM_BM / 16); it += 256) {
      const int k = it % KS, mm0 = (it / KS) * 16;
      float vn[16], vp[16];
#pragma unroll
      for (int e = 0; e < 16; ++e) { vn[e] = 0.f; vp[e] = 0.f; }
      if (k < a.ks && mm0 < rows) {
        const float dn = a.dX[(a.k_next + k) / a.crb_acts];
        const int4 qn = *reinterpret_cast<const int4*>(a.XqT + (size_t)(a.k_next + k) * a.Mp + m0 + mm0);
        const int8_t* bn = reinterpret_cast<const int8_t*>(&qn);
#pragma unroll
        for (int e = 0; e < 16; ++e) vn[e] = (mm0 + e < rows) ? dn * (float)bn[e] : 0.f;
        if (has_prev) {
          const float dp = a.dX[(a.k_prev + k) / a.crb_acts];
          const int4 qp = *reinterpret_cast<const int4*>(a.XqT + (size_t)(a.k_prev + k) * a.Mp + m0 + mm0);
          const int8_t* bp = reinterpret_cast<const int8_t*>(&qp);
#pragma unroll
          for (int e = 0; e < 16; ++e) vp[e] = (mm0 + e < rows) ? dp * (float)bp[e] : 0.f;
        }
      }
#pragma unroll
      for (int e = 0; e < 16; ++e) { xn[(mm0 + e) * KS + k] = vn[e]; xp[(mm0 + e) * KS + k] = vp[e]; }
    }
    __syncthreads();
    constexpr int UN = GRAM_UN;                             // tokens per group; the NEXT group's e and g are in flight
    float en[UN], gn[UN];                                   // while the current group is multiplied
    auto fetch = [&](int mm0) {
#pragma unroll
      for (int u = 0; u < UN; ++u) {
        const bool ok = ok_o && mm0 + u < rows;
        const size_t off = (size_t)(m0 + mm0 + u) * a.O + o;
        en[u] = ok ? a.E[off] : 0.f; gn[u] = ok ? a.G[off] : 0.f;
      }
    };
    fetch(0);
    for (int mm0 = 0; mm0 < rows; mm0 += UN) {
      float ec[UN], gc[UN];
#pragma unroll
      for (int u = 0; u < UN; ++u) { ec[u] = en[u]; gc[u] = gn[u] * gs; }
      if (mm0 + UN < rows) fetch(mm0 + UN);
#pragma unroll
      for (int u = 0; u < UN; ++u) {
        const int mm = mm0 + u;
        if (mm < rows) {
          float ev = ec[u];
          if (has_prev) {
            f32x2 s0 = 0ull, s1 = 0ull;
#pragma unroll
            for (int k = 0; k < KS; k += 4) {
              const float4 xv = *reinterpret_cast<const float4*>(&xp[mm * KS + k]);
              s0 = fma2(pack2(xv.x, xv.y), dd[k / 2], s0); s1 = fma2(pack2(xv.z, xv.w), dd[k / 2 + 1], s1);
            }
            float t0, t1, t2, t3; unpack2(s0, t0, t1); unpack2(s1, t2, t3);
            ev -= (t0 + t1) + (t2 + t3);
            if (ok_o) a.E[(size_t)(m0 + mm) * a.O + o] = ev;
          }
          const float ge = gc[u] * ev;
          e2 = fmaf(ge, ge, e2);
          const float w = gc[u] * ge;
          const f32x2 w2 = pack2(w, w);
#pragma unroll
          for (int k = 0; k < KS; k += 4) {
            const float4 xv = *reinterpret_cast<const float4*>(&xn[mm * KS + k]);
            acc[k / 2] = fma2(w2, pack2(xv.x, xv.y), acc[k / 2]); acc[k / 2 + 1] = fma2(w2, pack2(xv.z, xv.w), acc[k / 2 + 1]);
          }
        }
      }
    }
  }
  if (ok_o) {
    float* up = a.Upart + ((size_t)blockIdx.y * a.O + o) * a.ks;
#pragma unroll
    for (int k = 0; k < KS; k += 2) {
      float u0, u1; unpack2(acc[k / 2], u0, u1);
      if (k < a.ks) up[k] = u0;
      if (k + 1 < a.ks) up[k + 1] = u1;
    }
    a.E2part[(size_t)blockIdx.y * a.O + o] = e2;
  }
}

// U[o][k] = sum over token blocks (fixed order), E2[o] likewise.  thread = (o, k) ; k == ks handles E2.
__global__ void gram_reduce_kernel(const float* __restrict__ Upart, const float* __restrict__ E2part, int n_mblk, int O, int ks,
                                   float* __restrict__ U, float* __restrict__ E2) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long nU = (long long)O * ks;
  if (i < nU) {
    float s = 0.f;
    for (int b = 0; b < n_mblk; ++b) s += Upart[(size_t)b * nU + i];
    U[i] = s;
  } else if (i < nU + O) {
    const int o = (int)(i - nU);
    float s = 0.f;
    for (int b = 0; b < n_mblk; ++b) s += E2part[(size_t)b * O + o];
    E2[o] = s;
  }
}

// sums2[c][v] = sum over the osplit thread-block partials of row block v (fixed order).
__global__ void gram_keysum_kernel(const double* __restrict__ sums, int n_cand, int n_groups, int osplit, double* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_cand * n_groups) return;
  const int c = i / n_groups, v = i % n_groups;
  const double* p = sums + ((size_t)c * n_groups + v) * osplit;
  double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
  int k = 0;
  for (; k + 4 <= osplit; k += 4) { s0 += p[k]; s1 += p[k + 1]; s2 += p[k + 2]; s3 += p[k + 3]; }
  for (; k < osplit; ++k) s0 += p[k];
  out[i] = (s0 + s1) + (s2 + s3);
}

// block = a slice of one row block v (a.rows_per_block channels), thread = candidate.
// sums[c][block] = sum_o ( E2 - 2 d.U + d^T H d ).
template <int KS>
__global__ void __launch_bounds__(128) gram_eval_kernel(const GramEvalArgs a) {
  extern __shared__ float sm[];
  float* Hs = sm;                        // [npairs]
  float* Us = Hs + a.npairs;             // [KS]
  float* Ws = Us + KS;                   // [KS] fp32 weights of this channel
  float* Wc = Ws + KS;                   // [KS] currently quantised weights
  __shared__ float e2s;
  const int v = blockIdx.x / a.osplit, part = blockIdx.x % a.osplit;
  const int c = threadIdx.x;
  const int o_begin = v * a.rows_per_group + part * a.rows_per_block;
  const int o_end = min(min(a.O, (v + 1) * a.rows_per_group), o_begin + a.rows_per_block);
  const float d_cur = a.dW[v * a.n_H + a.h];
  const float d_c = c < a.n_cand ? a.factors[c] * a.dW0[v * a.n_H + a.h] : 1.f;
  const float dx = a.dX[a.k_first / a.crb_acts];
  const float dx2 = dx * dx;
  double total = 0.0;
  for (int o = o_begin; o < o_end; ++o) {
    __syncthreads();
    for (int i = threadIdx.x; i < a.npairs; i += blockDim.x) Hs[i] = a.H[(size_t)o * a.ldH + i] * dx2;
    for (int k = threadIdx.x; k < a.ks; k += blockDim.x) {
      Us[k] = a.U[(size_t)o * a.ks + k];
      const float w = a.W[(size_t)o * a.K + a.k_first + k];
      Ws[k] = w; Wc[k] = fq_dev(w, d_cur, a.w_lo, a.w_hi);
    }
    if (threadIdx.x == 0) e2s = a.E2[o];
    __syncthreads();
    if (c < a.n_cand) {
      float d[KS];
#pragma unroll
      for (int k = 0; k < KS; ++k) d[k] = k < a.ks ? fq_dev(Ws[k], d_c, a.w_lo, a.w_hi) - Wc[k] : 0.f;
      float lin = 0.f, quad = 0.f;
      int p = 0;
#pragma unroll
      for (int k = 0; k < KS; ++k) {
        if (k < a.ks) {
          lin = fmaf(d[k], Us[k], lin);
          float row = 0.5f * d[k] * Hs[p];                       // diagonal counted once
#pragma unroll
          for (int k2 = k + 1; k2 < KS; ++k2)
            if (k2 < a.ks) row = fmaf(d[k2], Hs[p + (k2 - k)], row);
          quad = fmaf(2.f * d[k], row, quad);
          p += a.ks - k;
        }
      }
      total += (double)(e2s - 2.f * lin + quad);
    }
  }
  if (c < a.n_cand) a.sums[(size_t)c * a.n_keys + blockIdx.x] = total;
}

}  // namespace

int p4v_xq_transpose(const float* x, int M, int K, int Mp, const float* dX, int crb_acts, float qlo, float qhi, int8_t* out,
                     cudaStream_t st) {
  dim3 grid(p4v_cdiv(Mp, 32), p4v_cdiv(K, 32)), block(32, 8);
  xq_transpose_kernel<<<grid, block, 0, st>>>(x, M, K, Mp, dX, crb_acts, qlo, qhi, out); p4v_count_launch();
  P4V_CUDA_OK(cudaGetLastError());
  return 0;
}

int p4v_pair_image(const int8_t* XqT, int Mp, int M, int k_first, int ks, int npairs, int n_blocks, int tiles_p,
                   unsigned long long tile_bytes, unsigned int term_bytes, uint8_t* dst, cudaStream_t st) {
  dim3 grid(tiles_p * (GRAM_PT / 128), term_bytes / 16);
  pair_image_kernel<<<grid, 128, 0, st>>>(XqT, Mp, M, k_first, ks, npairs, n_blocks, tiles_p, tile_bytes, term_bytes, dst); p4v_count_launch();
  P4V_CUDA_OK(cudaGetLastError());
  return 0;
}

template <int KS> static int launch_update(const GramUpdateArgs& a, cudaStream_t st) {
  if (a.h_prev >= 0) {
    const int n = a.O * KS;
    gram_delta_kernel<<<p4v_cdiv(n, 256), 256, 0, st>>>(a.W, a.O, a.K, a.k_prev, a.ks, KS, a.dW, a.dW_prev, a.n_V, a.n_H, a.crb_rows,
                                                        a.h_prev, a.w_lo, a.w_hi, a.D); p4v_count_launch();
    P4V_CUDA_OK(cudaGetLastError());
  }
  dim3 grid(p4v_cdiv(a.O, 256), a.n_split);
  gram_update_kernel<KS><<<grid, 256, 0, st>>>(a); p4v_count_launch();
  P4V_CUDA_OK(cudaGetLastError());
  return 0;
}
int p4v_gram_update(const GramUpdateArgs& a, cudaStream_t st) {
  P4V_REQUIRE(a.ks <= 64 && a.ks % 4 == 0, "gram: column block must be a multiple of 4 and <= 64 (got %d)", a.ks);
  P4V_REQUIRE(a.n_split >= 1 && a.D != nullptr, "gram: bad update plan");
  if (a.ks <= 32) return launch_update<32>(a, st);
  return launch_update<64>(a, st);
}
int p4v_gram_update_splits(int O, int M) {      // token splits: one wave of two blocks per SM
  const int cb = p4v_cdiv(O, 256);
  int s = (2 * p4v_num_sms()) / cb;
  const int max_s = p4v_cdiv(M, GRAM_BM);
  if (s > max_s) s = max_s;
  return s < 1 ? 1 : s;
}

int p4v_gram_reduce(const float* Upart, const float* E2part, int n_mblk, int O, int ks, float* U, float* E2, cudaStream_t st) {
  const long long n = (long long)O * ks + O;
  gram_reduce_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(Upart, E2part, n_mblk, O, ks, U, E2); p4v_count_launch();
  P4V_CUDA_OK(cudaGetLastError());
  return 0;
}

template <int KS> static int launch_eval(const GramEvalArgs& a, cudaStream_t st) {
  const size_t smem = ((size_t)a.npairs + 3 * KS) * sizeof(float);
  P4V_CUDA_OK(cudaFuncSetAttribute(gram_eval_kernel<KS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  gram_eval_kernel<KS><<<a.n_groups * a.osplit, 128, smem, st>>>(a); p4v_count_launch();
  P4V_CUDA_OK(cudaGetLastError());
  return 0;
}
int p4v_gram_eval(const GramEvalArgs& a, cudaStream_t st) {
  P4V_REQUIRE(a.n_cand <= 128, "gram: at most 128 candidates");
  int rc = a.ks <= 32 ? launch_eval<32>(a, st) : launch_eval<64>(a, st);
  if (rc) return rc;
  gram_keysum_kernel<<<p4v_cdiv(a.n_cand * a.n_groups, 256), 256, 0, st>>>(a.sums, a.n_cand, a.n_groups, a.osplit, a.sums2); p4v_count_launch();
  P4V_CUDA_OK(cudaGetLastError());
  return 0;
}
