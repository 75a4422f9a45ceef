#include "prep.cuh"
#include "../../include/ptq4vit_b200.h"
#include <math.h>
#include <stdlib.h>

namespace {

// order-preserving float <-> int key (so that atomicMax on ints is max on floats)
__device__ __forceinline__ int f2key(float f) {
  int b = __float_as_int(f);
  return b >= 0 ? b : b ^ 0x7fffffff;
}
__device__ __forceinline__ float key2f(int k) {
  return __int_as_float(k >= 0 ? k : k ^ 0x7fffffff);
}
constexpr int kKeyMin = (int)0x80000000;

__global__ void keys_reset_kernel(int* keys, int n) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) keys[i] = kKeyMin;
}

// grid (row_split, n_col_blocks, n_row_blocks)
__global__ void block_max_kernel(const float* __restrict__ src, long long ld, int rows, int row_block,
                                 int col_block, int use_abs, int* keys) {
  const int rb = blockIdx.z, cb = blockIdx.y;
  const int r_begin = rb * row_block, r_end = min(rows, r_begin + row_block);
  const int rows_here = max(0, r_end - r_begin);
  const int per = (rows_here + gridDim.x - 1) / gridDim.x;
  const int r0 = r_begin + blockIdx.x * per, r1 = min(r_end, r0 + per);
  float m = -INFINITY;
  for (int r = r0 + threadIdx.y; r < r1; r += blockDim.y) {
    const float* row = src + (size_t)r * ld + (size_t)cb * col_block;
    for (int c = threadIdx.x; c < col_block; c += blockDim.x) {
      float v = row[c];
      m = fmaxf(m, use_abs ? fabsf(v) : v);
    }
  }
  __shared__ float red[32];
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  const int tid = threadIdx.y * blockDim.x + threadIdx.x;
  if ((tid & 31) == 0) red[tid >> 5] = m;
  __syncthreads();
  if (tid == 0) {
    const int nw = (blockDim.x * blockDim.y + 31) / 32;
    for (int i = 1; i < nw; ++i) m = fmaxf(m, red[i]);
    if (m > -INFINITY) atomicMax(&keys[rb * gridDim.y + cb], f2key(m));
  }
}

// absmax over all problems p with p % n_groups == g ; grid (split, n_groups)
__global__ void group_absmax_kernel(const float* __restrict__ src, long long prob_elems, int P, int n_groups, int* keys) {
  const int g = blockIdx.y;
  float m = 0.f;
  for (int p = g; p < P; p += n_groups) {
    const float* base = src + (size_t)p * prob_elems;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < prob_elems; i += (long long)gridDim.x * blockDim.x)
      m = fmaxf(m, fabsf(base[i]));
  }
  __shared__ float red[32];
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int i = 1; i < (int)(blockDim.x + 31) / 32; ++i) m = fmaxf(m, red[i]);
    atomicMax(&keys[g], f2key(m));
  }
}

// The reference divides the block maxima by the Python scalar (qmax - 0.5) (linear.py:385, :395; matmul.py:424-436).
// On the GPU -- where the reference's Batching classes always run -- torch's true-divide by a CPU scalar is a
// multiplication by the fp32 reciprocal (ATen BinaryDivTrueKernel.cu), which differs from the IEEE quotient by one ulp
// for about a third of the inputs; a one-ulp step size moves the rounding of ~1e-5 of the quantised elements and with
// 32x32 weight blocks that is visible in the scores (measured: up to 2.6e-3 of an entry).  ieee_div = 1 selects the IEEE
// quotient instead (what torch computes on the CPU; the CPU-made golden vectors).
__global__ void keys_to_delta_kernel(const int* keys, int n, float denom, int ieee_div, float* d0, float* d1) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) {
    float v = ieee_div ? __fdiv_rn(key2f(keys[i]), denom) : __fmul_rn(key2f(keys[i]), __fdiv_rn(1.f, denom));
    d0[i] = v;
    if (d1) d1[i] = v;
  }
}

// init_layerwise: every key of the range becomes the maximum of the range (one block)
__global__ void keys_broadcast_max_kernel(int* keys, int n) {
  __shared__ int m;
  if (threadIdx.x == 0) m = kKeyMin;
  __syncthreads();
  int v = kKeyMin;
  for (int i = threadIdx.x; i < n; i += blockDim.x) v = max(v, keys[i]);
  atomicMax(&m, v);
  __syncthreads();
  for (int i = threadIdx.x; i < n; i += blockDim.x) keys[i] = m;
}

__global__ void make_gscale_kernel(const int* key, float* gscale) {
  float m = key2f(key[0]);
  float s = 1.f;
  if (m > 0.f && isfinite(m)) {
    int e;
    frexpf(m, &e);             // m = f * 2^e, f in [0.5,1)
    e = max(-100, min(100, 1 - e));
    s = ldexpf(1.f, e);        // m * s in [1,2)
  }
  gscale[0] = s;
}

// One thread = one (problem, 16-byte chunk, padded row) for a strided subset of the planes.  grid = (row blocks,
// P * chunks, plane groups): rows are the fastest index so that the 16-byte stores of a warp are contiguous in the
// image; the source values are loaded once and quantised for every plane (candidate step size) of the subset.
template <bool kInt8>
__global__ void quant_image_kernel(const QuantImageArgs a, int chunks_total, int row_blocks) {
  const int rows_pad = a.tiles * P4V_TILE;
  const int row_p = (int)(blockIdx.x % row_blocks) * blockDim.x + threadIdx.x;      // rows fastest, then (problem, chunk)
  if (row_p >= rows_pad) return;
  const unsigned pc = blockIdx.x / row_blocks;
  const int p = (int)(pc / chunks_total);
  int chunk = (int)(pc % chunks_total);
  constexpr int epc = kInt8 ? 16 : 8;          // elements per 16-byte chunk
  int s = 0;
  while (true) {
    const int nch = ((a.segs[s].klen + (kInt8 ? 31 : 15)) / (kInt8 ? 32 : 16)) * 2;   // chunks of this segment (padded to 32 B)
    if (chunk < nch) break;
    chunk -= nch; ++s;
  }
  const P4VSeg sg = a.segs[s];
  const int tile = row_p / P4V_TILE, r = row_p % P4V_TILE;
  uint8_t* dst0 = a.dst + ((size_t)p * a.tiles + tile) * a.tile_bytes + sg.dst_off + ((size_t)chunk * P4V_TILE + r) * 16;
  float vals[epc];
  float delta0 = 1.f;
  const bool plain = !(sg.sos_part || sg.split3);
  if (row_p < a.rows) {
    if (plain) {
      if (sg.fixed_delta > 0.f) delta0 = sg.fixed_delta;
      else {
        const int rb = a.rows_per_block > 0 ? row_p / a.rows_per_block : (p % a.d_mod);
        delta0 = a.delta[(size_t)rb * a.d_stride + sg.didx];
      }
    }
    const float* base = a.src + (size_t)p * a.prob_stride;
    if (!a.src_transposed && chunk * epc + epc <= sg.klen && ((a.ld | sg.k0) & 3) == 0) {
      const float4* src4 = reinterpret_cast<const float4*>(base + (size_t)row_p * a.ld + sg.k0 + chunk * epc);
#pragma unroll
      for (int e = 0; e < epc / 4; ++e) { const float4 t4 = src4[e]; vals[4 * e] = t4.x; vals[4 * e + 1] = t4.y; vals[4 * e + 2] = t4.z; vals[4 * e + 3] = t4.w; }
    } else {
#pragma unroll
      for (int e = 0; e < epc; ++e) {
        const int kk = chunk * epc + e;
        const int k = sg.k0 + kk;
        vals[e] = kk < sg.klen ? (a.src_transposed ? base[(size_t)k * a.ld + row_p] : base[(size_t)row_p * a.ld + k]) : 0.f;
      }
    }
    if (sg.square) {
      const float ps = a.presc ? a.presc[0] : 1.f;
#pragma unroll
      for (int e = 0; e < epc; ++e) { const float v = vals[e] * ps; vals[e] = v * v; }
    }
  }
  for (int plane = blockIdx.z; plane < a.n_planes; plane += gridDim.z) {
    uint32_t w[4] = {0u, 0u, 0u, 0u};
    if (row_p < a.rows) {
      const float split = sg.sos_part ? (a.factors ? a.factors[plane] : a.split[0]) : 0.f;
      float delta = delta0;
      if (plain && sg.fixed_delta <= 0.f && a.factors) delta = a.factors[plane] * delta0;   // fl(f_c * delta0), as the reference's candidate table
      const bool fast = plain && p4v_rint_div_ok(delta);
      const float rcp = fast ? __frcp_rn(delta) : 0.f;
      const float rcp_fixed = sg.fixed_delta > 0.f ? __fdiv_rn(1.f, sg.fixed_delta) : 0.f;
#pragma unroll
      for (int e = 0; e < epc; ++e) {
        const int kk = chunk * epc + e;
        float q = 0.f;
        if (kk < sg.klen) {
          const float v = vals[e];
          if (sg.split3) {
            const float b1 = __bfloat162float(__float2bfloat16_rn(v));
            const float b2 = __bfloat162float(__float2bfloat16_rn(v - b1));
            q = sg.split3 == 1 ? b1 : (sg.split3 == 2 ? b2 : __bfloat162float(__float2bfloat16_rn((v - b1) - b2)));
          } else if (sg.sos_part == 1) {
            q = fminf(fmaxf(rintf(fminf(fmaxf(v, split), 1.f) * sg.qm1), 0.f), sg.qm1);
          } else if (sg.sos_part == 2) {
            q = fminf(fmaxf(rintf(__fdiv_rn(fminf(fmaxf(v, 0.f), split), __fdiv_rn(split, sg.qm1))), 0.f), sg.qm1);
          } else {
            // A step size that the reference holds as a Python scalar (the constant negative-part step of the post-GELU
            // twin quantizer, linear.py:574, :605) is divided by as `x * (1/delta)` on the GPU: torch's CUDA true-divide
            // multiplies by the fp32 reciprocal when the divisor is a CPU scalar (ATen BinaryDivTrueKernel.cu).  Tensors
            // (every searched step size) take the IEEE division.
            if (sg.fixed_delta > 0.f && !a.ieee_div) q = fminf(fmaxf(rintf(v * rcp_fixed), sg.lo), sg.hi);
            else q = fminf(fmaxf(fast ? p4v_rint_div(v, delta, rcp) : rintf(__fdiv_rn(v, delta)), sg.lo), sg.hi);
          }
          if (!(q == q)) q = 0.f;   // NaN (0/0) cannot be represented in the integer operand
        }
        if constexpr (kInt8) {
          const int qi = (int)q;
          w[e >> 2] |= (uint32_t)(qi & 0xff) << ((e & 3) * 8);
        } else {
          const uint32_t hb = (uint32_t)__bfloat16_as_ushort(__float2bfloat16_rn(q));
          w[e >> 1] |= hb << ((e & 1) * 16);
        }
      }
    }
    *reinterpret_cast<uint4*>(dst0 + (size_t)plane * a.plane_stride) = make_uint4(w[0], w[1], w[2], w[3]);
  }
}

__device__ __forceinline__ void step_tables_body(const StepTablesArgs& a, int tid, int nthreads) {
  const int total_fix = a.n_fixed_groups * a.nsg;
  const int total_cb = a.n_cand_groups * a.nsg;
  const int total_ca = a.n_cand * a.nsg;
  for (int i = tid; i < total_fix + total_cb + total_ca; i += nthreads) {
    if (i < total_fix) {
      const int g = i / a.nsg, sg = i % a.nsg;
      const GroupMeta m = a.fixed_meta[g];
      if (a.kind >= 2) {
        a.fix_scale[i] = a.dW[sg] * (a.kind == 2 ? a.dX[sg] : a.dX[m.a]);
      } else {
        const int v = min((sg * P4V_CG) / a.crb_rows, a.n_V - 1);
        a.fix_scale[i] = a.dW[v * a.n_H + m.h] * (m.neg ? a.d_neg : a.dX[m.a]);
      }
    } else if (i < total_fix + total_cb) {
      const int j = i - total_fix;
      const int g = j / a.nsg, sg = j % a.nsg;
      const GroupMeta m = a.cand_meta[g];
      float val;
      if (a.kind == 0)      val = m.neg ? a.d_neg : a.dX[m.a];
      else if (a.kind == 1) val = a.dW[min((sg * P4V_CG) / a.crb_rows, a.n_V - 1) * a.n_H + m.h];
      else if (a.kind == 2) val = a.dX[sg];                         // head-wise other operand
      else                  val = m.neg ? a.d_neg : a.dX[m.a];      // uniform other-operand scale per group
      a.candB[j] = val;
    } else {
      const int j = i - total_fix - total_cb;
      const int c = j / a.nsg, sg = j % a.nsg;
      float base;
      if (a.kind == 0)      base = a.dW0[min((sg * P4V_CG) / a.crb_rows, a.n_V - 1) * a.n_H + a.target];
      else if (a.kind == 1) base = a.dX0[a.target];
      else                  base = a.dW0[sg];
      a.candA[j] = a.factors[c] * base;
    }
  }
}
__global__ void step_tables_kernel(const StepTablesArgs a) {
  step_tables_body(a, blockIdx.x * blockDim.x + threadIdx.x, gridDim.x * blockDim.x);
}

// One warp per (candidate, key): coalesced 128-byte rows of the partial buffer, fixed order, fp64.
__global__ void reduce_scores_kernel(const ReduceArgs a) {
  const int warps_per_block = blockDim.x >> 5;
  const int task = blockIdx.x * warps_per_block + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  const int n_task_keys = a.mode == P4V_SG_COLUMN ? a.tiles_n : a.n_keys;
  if (task >= a.n_cand * n_task_keys) return;
  const int c = task / n_task_keys, key = task % n_task_keys;
  const int per_p = a.tiles_m * a.tiles_n;
  double acc = 0.0;
  if (a.mode == P4V_SG_COLUMN) {          // key = tn ; lane = quarter * 8 + i8
    for (int p = 0; p < a.P; ++p)
      for (int tm = 0; tm < a.tiles_m; ++tm) {
        const int t = a.order == 0 ? key * a.tiles_m + tm : tm * a.tiles_n + key;
        acc += (double)a.partial[(((size_t)p * per_p + t) * a.n_cand + c) * 32 + lane];
      }
    acc += __shfl_xor_sync(0xffffffffu, acc, 8);
    acc += __shfl_xor_sync(0xffffffffu, acc, 16);
    if (lane < 8) a.sums[(size_t)c * a.n_keys + key * P4V_TILE_CG + lane] = acc;
  } else {                                // key = p % n_keys ; all 32 entries belong to the key
    for (int p = key; p < a.P; p += a.n_keys)
      for (int t = 0; t < per_p; ++t)
        acc += (double)a.partial[(((size_t)p * per_p + t) * a.n_cand + c) * 32 + lane];
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) a.sums[(size_t)c * a.n_keys + key] = acc;
  }
}

__global__ void __launch_bounds__(1024) select_step_kernel(const SelectArgs a) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
  const double gs = (double)a.gscale[0];
  const double norm = a.inv_count / (gs * gs);
  for (int g = warp; g < a.n_groups; g += nwarps) {
    // The comparison runs on the fp32-rounded score, like the reference's argmax over its fp32 similarity tensor
    // (linear.py:493, :531): candidates whose scores round to the same float tie, and the first one wins.  (Comparing
    // the fp64 sums would pick the later candidate of such a pair and send that row block down another greedy path;
    // it would also disagree with the argmax of the logged fp32 table.)
    float bv = 0.f; int bi = -1;
    for (int c = lane; c < a.n_cand; c += 32) {      // ascending c: strict '>' keeps the first maximum
      double sacc = 0.0;
      for (int k = 0; k < a.keys_per_group; ++k) sacc += a.sums[(size_t)c * a.n_keys + g * a.keys_per_group + k];
      const float v = (float)(-sacc * norm);
      if (a.score_log) a.score_log[(size_t)c * a.n_groups + g] = v;
      bool take;
      if (bi < 0) take = true;
      else if (bv != bv) take = false;               // an earlier NaN already won
      else take = (v != v) || (v > bv);
      if (take) { bv = v; bi = c; }
    }
    for (int o = 16; o > 0; o >>= 1) {
      const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
      const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
      bool take;
      if (oi < 0) take = false;
      else if (bi < 0) take = true;
      else if ((ov != ov) != (bv != bv)) take = (ov != ov);                // NaN beats a number
      else if (ov != ov) take = oi < bi;                                   // both NaN: lower index
      else take = ov > bv || (ov == bv && oi < bi);
      if (take) { bv = ov; bi = oi; }
    }
    if (lane == 0) {
      const size_t di = (size_t)g * a.d_stride + a.d_col;
      if (a.d_prev) a.d_prev[g] = a.d[di];
      a.d[di] = a.factors[bi] * a.d0[di];
      a.best[g] = bi;
    }
  }
  if (a.has_next) {
    __threadfence_block();
    __syncthreads();
    step_tables_body(a.next, threadIdx.x, blockDim.x);
  }
}

__global__ void commit_step_kernel(const CommitArgs a, int chunks_total) {
  const long long rows_pad = (long long)a.tiles * P4V_TILE;
  const long long total = (long long)a.P * rows_pad * chunks_total;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
    const int row_p = (int)(idx % rows_pad); long long rem = idx / rows_pad;
    int chunk = (int)(rem % chunks_total); const int p = (int)(rem / chunks_total);
    int s = 0;
    while (chunk >= (a.segs[s].kb >> 4)) { chunk -= a.segs[s].kb >> 4; ++s; }
    int g = 0;
    if (a.problem_groups) g = p % a.n_groups;
    else if (a.rows_per_group > 0) g = min(row_p / a.rows_per_group, a.n_groups - 1);
    const int tile = row_p / P4V_TILE, r = row_p % P4V_TILE;
    const size_t in_tile = ((size_t)chunk * P4V_TILE + r) * 16;
    const uint4 v = *reinterpret_cast<const uint4*>(a.cand + (size_t)a.best[g] * a.cand_plane_stride +
                                                   ((size_t)p * a.tiles + tile) * a.cand_tile_bytes + a.segs[s].src_off + in_tile);
    *reinterpret_cast<uint4*>(a.cur + ((size_t)p * a.tiles + tile) * a.cur_tile_bytes + a.segs[s].dst_off + in_tile) = v;
  }
}

int grid_for(long long total, int block, int cap = 148 * 16) {
  long long g = (total + block - 1) / block;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return (int)g;
}

}  // namespace

int p4v_keys_reset(int* keys, int n, cudaStream_t st) {
  keys_reset_kernel<<<p4v_cdiv(n, 128), 128, 0, st>>>(keys, n); p4v_count_launch();
  P4V_CUDA_OK(cudaGetLastError());
  return 0;
}

int p4v_block_max(const float* src, long long ld, int rows, int row_block, int n_row_blocks, int col_block,
                  int n_col_blocks, int use_abs, int* keys, cudaStream_t st) {
  long long elems = (long long)row_block * col_block;
  int split = (int)((elems + (1 << 16) - 1) >> 16);
  if (split < 1) split = 1;
  if (split > 256) split = 256;
  if (split > row_block) split = row_block;
  dim3 grid(split, n_col_blocks, n_row_blocks), block(32, 8);
  block_max_kernel<<<grid, block, 0, st>>>(src, ld, rows, row_block, col_block, use_abs, keys); p4v_count_launch();
  P4V_CUDA_OK(cudaGetLastError());
  return 0;
}

int p4v_group_absmax(const float* src, long long prob_elems, int P, int n_groups, int* keys, cudaStream_t st) {
  long long per_group = prob_elems * ((P + n_groups - 1) / n_groups);
  int split = (int)((per_group + (1 << 16) - 1) >> 16);
  if (split < 1) split = 1;
  if (split > 128) split = 128;
  dim3 grid(split, n_groups);
  group_absmax_kernel<<<grid, 256, 0, st>>>(src, prob_elems, P, n_groups, keys); p4v_count_launch();
  P4V_CUDA_OK(cudaGetLastError());
  return 0;
}

int p4v_keys_broadcast_max(int* keys, int n, cudaStream_t st) {
  keys_broadcast_max_kernel<<<1, 256, 0, st>>>(keys, n); p4v_count_launch();
  P4V_CUDA_OK(cudaGetLastError());
  return 0;
}
int p4v_scalar_div_ieee() {
  const char* e = getenv("P4V_SCALAR_DIV");      // "ieee": reference executed on the CPU; default: reference executed on the GPU
  return (e && e[0] == 'i') ? 1 : 0;
}
int p4v_keys_to_delta(const int* keys, int n, float denom, float* d0, float* d1, cudaStream_t st) {
  keys_to_delta_kernel<<<p4v_cdiv(n, 128), 128, 0, st>>>(keys, n, denom, p4v_scalar_div_ieee(), d0, d1); p4v_count_launch();
  P4V_CUDA_OK(cudaGetLastError());
  return 0;
}

int p4v_make_gscale(const int* key, float* gscale, cudaStream_t st) {
  make_gscale_kernel<<<1, 1, 0, st>>>(key, gscale); p4v_count_launch();
  P4V_CUDA_OK(cudaGetLastError());
  return 0;
}

namespace {
__device__ __forceinline__ unsigned long long mix64(unsigned long long z) {       // splitmix64
  z += 0x9E3779B97F4A7C15ull; z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull; z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}
__global__ void rint_div_selftest_kernel(unsigned long long n, unsigned long long seed, unsigned long long* mismatches) {
  unsigned long long bad = 0;
  for (unsigned long long i = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; i < n; i += (unsigned long long)gridDim.x * blockDim.x) {
    const unsigned long long h = mix64(seed + i), h2 = mix64(h);
    // delta: random mantissa, exponent 2^-24 .. 2^4; quotient target |q| < 300
    const float delta = __uint_as_float(((unsigned)(103 + (h & 31)) << 23) | (unsigned)((h >> 8) & 0x7fffff));
    float v;
    const unsigned mode = (unsigned)(h2 & 3);
    if (mode == 0) {            // free mantissa
      v = __uint_as_float((unsigned)(h2 >> 32));
      if (!(fabsf(v) < 3e38f)) v = 1.f;
      v = fmodf(v, 300.f * delta);
    } else {                    // on / next to a rounding tie: (k + 0.5) * delta, moved by -2..+2 ulps
      const float k = (float)((int)((h2 >> 8) % 600) - 300) + 0.5f;
      v = k * delta;
      const int steps = (int)((h2 >> 40) % 5) - 2;
      v = __uint_as_float(__float_as_uint(v) + steps);
    }
    const float want = rintf(__fdiv_rn(v, delta));
    const float got = p4v_rint_div_ok(delta) ? p4v_rint_div(v, delta, __frcp_rn(delta)) : want;
    if (!(want == got) && !(want != want && got != got)) ++bad;
  }
  if (bad) atomicAdd(mismatches, bad);
}
}  // namespace

extern "C" int p4v_selftest_rint_div(unsigned long long n, unsigned long long seed, unsigned long long* mismatches, void* stream) {
  P4V_REQUIRE(mismatches != nullptr, "selftest: null output");
  cudaStream_t st = (cudaStream_t)stream;
  unsigned long long* d = nullptr;
  P4V_CUDA_OK(cudaMalloc(&d, 8));
  P4V_CUDA_OK(cudaMemsetAsync(d, 0, 8, st));
  rint_div_selftest_kernel<<<148 * 8, 256, 0, st>>>(n, seed, d); p4v_count_launch();
  P4V_CUDA_OK(cudaGetLastError());
  P4V_CUDA_OK(cudaMemcpyAsync(mismatches, d, 8, cudaMemcpyDeviceToHost, st));
  P4V_CUDA_OK(cudaStreamSynchronize(st));
  P4V_CUDA_OK(cudaFree(d));
  return 0;
}

int p4v_quant_image(const QuantImageArgs& a_in, cudaStream_t st) {
  QuantImageArgs a = a_in;
  a.ieee_div = p4v_scalar_div_ieee();
  const int chunks_total = (int)(a.tile_bytes / P4V_TILE / 16);     // every segment is padded to 32 B
  const int rows_pad = a.tiles * P4V_TILE;
  if (rows_pad == 0 || chunks_total == 0 || a.n_planes == 0 || a.P == 0) return 0;
  const int row_blocks = p4v_cdiv(rows_pad, 128);
  const long long blocks_xy = (long long)row_blocks * a.P * chunks_total;
  P4V_REQUIRE(blocks_xy <= 0x7fffffffll && a.n_planes <= 65535, "quant_image: grid too large");
  long long zg = (4096 + blocks_xy - 1) / blocks_xy;        // enough blocks to fill the GPU, otherwise all planes per thread
  if (zg > a.n_planes) zg = a.n_planes;
  if (zg < 1) zg = 1;
  dim3 grid((unsigned)blocks_xy, 1, (unsigned)zg);
  if (a.is_int8) quant_image_kernel<true><<<grid, 128, 0, st>>>(a, chunks_total, row_blocks);
  else quant_image_kernel<false><<<grid, 128, 0, st>>>(a, chunks_total, row_blocks);
  p4v_count_launch();
  P4V_CUDA_OK(cudaGetLastError());
  return 0;
}

int p4v_step_tables(const StepTablesArgs& a, cudaStream_t st) {
  const int total = (a.n_fixed_groups + a.n_cand_groups + a.n_cand) * a.nsg;
  if (total == 0) return 0;
  step_tables_kernel<<<grid_for(total, 256, 64), 256, 0, st>>>(a); p4v_count_launch();
  P4V_CUDA_OK(cudaGetLastError());
  return 0;
}

int p4v_reduce_scores(const ReduceArgs& a, cudaStream_t st) {
  const int tasks = a.n_cand * (a.mode == P4V_SG_COLUMN ? a.tiles_n : a.n_keys);
  reduce_scores_kernel<<<p4v_cdiv(tasks, 8), 256, 0, st>>>(a); p4v_count_launch();
  P4V_CUDA_OK(cudaGetLastError());
  return 0;
}

int p4v_select_step(const SelectArgs& a, cudaStream_t st) {
  int threads = 32 * a.n_groups;
  if (a.has_next || threads > 1024) threads = 1024;
  if (threads < 32) threads = 32;
  select_step_kernel<<<1, threads, 0, st>>>(a); p4v_count_launch();
  P4V_CUDA_OK(cudaGetLastError());
  return 0;
}

int p4v_commit_step(const CommitArgs& a, cudaStream_t st) {
  if (a.nseg <= 0) return 0;
  const long long total = (long long)a.P * a.tiles * P4V_TILE * a.commit_chunks;
  commit_step_kernel<<<grid_for(total, 256, 148 * 8), 256, 0, st>>>(a, a.commit_chunks); p4v_count_launch();
  P4V_CUDA_OK(cudaGetLastError());
  return 0;
}
