// C-ABI for the channel-wise weight search of the patch-embedding convolution
// (ChannelwiseBatchingQuantConv2d with a_bit >= 32, reference quant_layers/conv.py:444-614, as wired by
// configs/PTQ4ViT.py:52-54): per output channel o the step size f_c * delta0[o] minimising
//     sum_images mean_positions ( g * (y - b - conv(x, fq(w, f_c * delta0))) )^2          (conv.py:526-557)
// The convolution is a product over the im2col matrix: for image p
//     D_p[o, l] = sum_k q_c[o, k] * cols_p[l, k] ,   yhat = b[o] + f_c * delta0[o] * D_p[o, l]
// rows = output channels (row operand: candidate planes of the integer kernel, shared by all images), columns = output
// positions (column operand: the FP32 im2col matrix split exactly into three bf16 terms -- the activations are not
// quantised), one accumulator per candidate, three term products chained into it.  The per-channel step size would be a
// per-ROW scale; the sweep's scales are per column group, so delta0[o] is folded into the targets once:
//     (g * (y - b - f*d0*D))^2 = (g*d0 * ((y - b)/d0 - f*D))^2
// and the candidate scale is the plain factor f_c.  Scores are kept per row (SweepParams::row_keys).
#include <algorithm>
#include <vector>

#include "../../include/ptq4vit_b200.h"
#include "plan.cuh"
#include "prep.cuh"

namespace {

struct ConvPlan {
  p4v_conv_desc d;
  int P, O, K, L, tiles_o, tiles_l, kb, w_qmax;
  std::vector<P4VJob> jobs; std::vector<P4VSeg> segW, segC; std::vector<float> factors;
  size_t o_factors, o_keys, o_d0, o_d, o_gscale, o_ones, o_scores, o_best, o_candA, o_candB, o_fix, o_jobs, o_segW, o_segC,
      o_partial, o_Wcand, o_Cimg, o_Y, o_G, total;
};

int build_plan(const p4v_conv_desc* d, ConvPlan& p) {
  P4V_REQUIRE(d != nullptr, "null desc");
  p.d = *d;
  p.P = d->images; p.O = d->out_channels; p.K = d->K; p.L = d->positions;
  P4V_REQUIRE(p.P > 0 && p.O > 0 && p.K > 0 && p.L > 0, "conv: empty shape");
  P4V_REQUIRE(d->w_bit >= 2 && d->w_bit <= 8, "conv: w_bit must be in [2,8]");
  P4V_REQUIRE(d->eq_n >= 1 && d->eq_n <= P4V_MAX_CAND, "conv: eq_n must be in [1,%d]", P4V_MAX_CAND);
  P4V_REQUIRE(d->kernel == P4V_KERNEL_TCGEN05, "conv: the channel-wise search runs on the tcgen05 kernel only");
  p.w_qmax = 1 << (d->w_bit - 1);
  p.tiles_o = p4v_cdiv(p.O, P4V_TILE); p.tiles_l = p4v_cdiv(p.L, P4V_TILE);
  p.kb = (int)align_up((size_t)p.K * 2, 32);                    // bf16 row bytes of one term
  P4V_REQUIRE(3 * (p.kb / 32) <= P4V_MAX_JOBS * 4 && 3 * p4v_cdiv(p.kb, P4V_JOB_KB) <= P4V_MAX_JOBS, "conv: kernel volume too large");
  p.segW = {P4VSeg{0, p.K, 0, 0, 0.f, (float)-p.w_qmax, (float)(p.w_qmax - 1), 0, 0.f, 0, 0}};
  p.segC.clear();
  for (int t = 0; t < 3; ++t) p.segC.push_back(P4VSeg{0, p.K, t * p.kb * P4V_TILE, 0, 0.f, 0.f, 0.f, 0, 0.f, t + 1, 0});
  p.factors = candidate_factors(d->eq_alpha, d->eq_beta, d->eq_n);
  p.jobs.clear();
  int n_jobs = 0;
  for (int t = 0; t < 3; ++t)        // the three term products chain into one accumulator
    push_jobs(p.jobs, 0, t * p.kb, p.kb, P4V_JOB_RCAND, 0, t == 0, t == 2, n_jobs);
  Carver w;
  const int n_c = d->eq_n;
  p.o_factors = w.take((n_c + 1) * 4); p.o_keys = w.take((p.O + 1) * 4);
  p.o_d0 = w.take(p.O * 4); p.o_d = w.take(p.O * 4); p.o_gscale = w.take(4); p.o_ones = w.take(4);
  p.o_scores = w.take((size_t)n_c * p.O * 8); p.o_best = w.take(p.O * 4);
  p.o_candA = w.take((size_t)n_c * 4); p.o_candB = w.take(4); p.o_fix = w.take(4);
  p.o_jobs = w.take(p.jobs.size() * sizeof(P4VJob)); p.o_segW = w.take(sizeof(P4VSeg)); p.o_segC = w.take(3 * sizeof(P4VSeg));
  p.o_partial = w.take((size_t)p.P * p.tiles_o * p.tiles_l * n_c * 256 * 4);
  p.o_Wcand = w.take((size_t)n_c * p.tiles_o * P4V_TILE * p.kb);
  p.o_Cimg = w.take((size_t)p.P * p.tiles_l * P4V_TILE * 3 * p.kb);
  p.o_Y = w.take((size_t)p.P * p.O * p.L * 4); p.o_G = w.take((size_t)p.P * p.O * p.L * 4);
  p.total = w.total;
  return 0;
}

// y' = (y - b[o]) / d0[o] ,  g' = g * d0[o]      ([P][O][L], one thread per element)
__global__ void conv_prescale_kernel(const float* __restrict__ y, const float* __restrict__ g, const float* __restrict__ bias,
                                     const float* __restrict__ d0, int O, int L, long long n, float* __restrict__ yo, float* __restrict__ go) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int o = (int)((i / L) % O);
    const float d = d0[o];
    yo[i] = __fdiv_rn(y[i] - (bias ? bias[o] : 0.f), d);
    go[i] = g[i] * d;
  }
}

// sums[c][o] = sum over images, position tiles and column halves of the per-row partials (fixed order, fp64)
__global__ void conv_reduce_kernel(const float* __restrict__ partial, int P, int tiles_o, int tiles_l, int n_cand, int O, double* sums) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n_cand * O) return;
  const int c = idx / O, o = idx % O;
  const int to = o / P4V_TILE, r = o % P4V_TILE;
  double acc = 0.0;
  for (int p = 0; p < P; ++p)
    for (int tl = 0; tl < tiles_l; ++tl) {
      // tile index of the sweep: order 0 -> t = tn * tiles_m + tm inside a problem
      const size_t tile = (size_t)p * tiles_o * tiles_l + (size_t)tl * tiles_o + to;
      const float* base = partial + (tile * n_cand + c) * 256;          // [column half][128 rows]
      acc += (double)base[r] + (double)base[128 + r];
    }
  sums[(size_t)c * O + o] = acc;
}

__global__ void conv_fill_kernel(float* candA, const float* factors, int n, float* ones) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) candA[i] = factors[i];
  if (i == 0) ones[0] = 1.f;
}

}  // namespace

extern "C" int p4v_conv_workspace_bytes(const p4v_conv_desc* d, size_t* bytes) {
  return plan_workspace_bytes(build_plan, d, bytes);
}

extern "C" int p4v_conv_calibrate(const p4v_conv_desc* d, const float* cols, const float* weight, const float* bias,
                                  const float* raw_out, const float* raw_grad, void* ws, size_t workspace_bytes,
                                  float* w_interval, float* score_log, void* stream) {
  ConvPlan p; int rc = build_plan(d, p);
  if (rc) return rc;
  P4V_REQUIRE(cols && weight && raw_out && raw_grad && ws && w_interval, "conv_calibrate: null pointer");
  P4V_REQUIRE(!d->has_bias || bias, "conv_calibrate: has_bias set but bias is null");
  P4V_REQUIRE(workspace_bytes >= p.total, "conv_calibrate: workspace too small (%zu < %zu)", workspace_bytes, p.total);
  cudaStream_t st = (cudaStream_t)stream;
  if ((rc = upload(ws, p.o_factors, p.factors, st)) || (rc = upload(ws, p.o_jobs, p.jobs, st)) ||
      (rc = upload(ws, p.o_segW, p.segW, st)) || (rc = upload(ws, p.o_segC, p.segC, st))) return rc;
  // min-max step size per output channel (conv.py:487) and the gradient scale
  int* keys = at<int>(ws, p.o_keys);
  if ((rc = p4v_keys_reset(keys, p.O + 1, st))) return rc;
  if ((rc = p4v_block_max(weight, p.K, p.O, 1, p.O, p.K, 1, 1, keys, st))) return rc;
  if ((rc = p4v_group_absmax(raw_grad, (long long)p.P * p.O * p.L, 1, 1, keys + p.O, st))) return rc;
  if ((rc = p4v_keys_to_delta(keys, p.O, (float)p.w_qmax - 0.5f, at<float>(ws, p.o_d0), at<float>(ws, p.o_d), st))) return rc;
  if ((rc = p4v_make_gscale(keys + p.O, at<float>(ws, p.o_gscale), st))) return rc;
  conv_fill_kernel<<<p4v_cdiv(d->eq_n, 128), 128, 0, st>>>(at<float>(ws, p.o_candA), at<float>(ws, p.o_factors), d->eq_n, at<float>(ws, p.o_candB));
  p4v_count_launch();
  const long long n = (long long)p.P * p.O * p.L;
  conv_prescale_kernel<<<148 * 8, 256, 0, st>>>(raw_out, raw_grad, d->has_bias ? bias : nullptr, at<float>(ws, p.o_d0), p.O, p.L, n,
                                                 at<float>(ws, p.o_Y), at<float>(ws, p.o_G));
  p4v_count_launch();
  P4V_CUDA_OK(cudaGetLastError());
  {   // candidate planes of the integer kernel: rows = channels, one step size per row
    QuantImageArgs q{};
    q.src = weight; q.ld = p.K; q.prob_stride = 0; q.src_transposed = 0; q.P = 1; q.rows = p.O; q.tiles = p.tiles_o;
    q.dst = at<uint8_t>(ws, p.o_Wcand); q.tile_bytes = (unsigned long long)P4V_TILE * p.kb; q.plane_stride = q.tile_bytes * p.tiles_o;
    q.n_planes = d->eq_n; q.factors = at<float>(ws, p.o_factors); q.delta = at<float>(ws, p.o_d0);
    q.rows_per_block = 1; q.d_stride = 1; q.d_mod = 1; q.segs = at<P4VSeg>(ws, p.o_segW); q.nseg = 1; q.is_int8 = 0;
    if ((rc = p4v_quant_image(q, st))) return rc;
  }
  {   // exact three-term bf16 split of the FP32 im2col matrix: rows = output positions
    QuantImageArgs q{};
    q.src = cols; q.ld = p.K; q.prob_stride = (long long)p.L * p.K; q.src_transposed = 0; q.P = p.P; q.rows = p.L; q.tiles = p.tiles_l;
    q.dst = at<uint8_t>(ws, p.o_Cimg); q.tile_bytes = (unsigned long long)P4V_TILE * 3 * p.kb; q.plane_stride = 0;
    q.n_planes = 1; q.factors = nullptr; q.delta = at<float>(ws, p.o_d0); q.rows_per_block = 0; q.d_stride = 0; q.d_mod = 1;
    q.segs = at<P4VSeg>(ws, p.o_segC); q.nseg = 3; q.is_int8 = 0;
    if ((rc = p4v_quant_image(q, st))) return rc;
  }
  SweepParams sp{};
  sp.R_cur = sp.R_cand = at<uint8_t>(ws, p.o_Wcand); sp.C_cur = sp.C_cand = at<uint8_t>(ws, p.o_Cimg);
  sp.R_tile_bytes = sp.R_cand_tile_bytes = (unsigned long long)P4V_TILE * p.kb;
  sp.C_tile_bytes = sp.C_cand_tile_bytes = (unsigned long long)P4V_TILE * 3 * p.kb;
  sp.R_cand_stride = sp.R_cand_tile_bytes * p.tiles_o; sp.C_cand_stride = 0;
  sp.R_shared = 1;                                          // the kernel planes do not depend on the image
  sp.P = p.P; sp.M = p.O; sp.N = p.L; sp.tiles_m = p.tiles_o; sp.tiles_n = p.tiles_l;
  sp.Y = at<float>(ws, p.o_Y); sp.Gr = at<float>(ws, p.o_G); sp.bias = nullptr;
  sp.ld = p.L; sp.prob_stride = (long long)p.O * p.L;
  sp.gscale = at<float>(ws, p.o_gscale);
  sp.jobs = at<P4VJob>(ws, p.o_jobs);
  sp.n_fixed_jobs = 0; sp.n_cand_jobs = (int)p.jobs.size(); sp.n_fixed_groups = 0; sp.n_cand_groups = 1;
  sp.fix_scale = at<float>(ws, p.o_fix); sp.candA = at<float>(ws, p.o_candA); sp.candB = at<float>(ws, p.o_candB);
  sp.nsg = 1; sp.sg_mode = P4V_SG_PROBLEM;                  // one scale group: the candidate factor
  sp.n_cand = d->eq_n; sp.partial = at<float>(ws, p.o_partial); sp.is_int8 = 0; sp.order = 0;
  sp.row_keys = 1;
  if ((rc = p4v_run_sweep(sp, p.jobs.data(), d->kernel, st))) return rc;
  conv_reduce_kernel<<<p4v_cdiv(d->eq_n * p.O, 256), 256, 0, st>>>(sp.partial, p.P, p.tiles_o, p.tiles_l, d->eq_n, p.O, at<double>(ws, p.o_scores));
  p4v_count_launch();
  P4V_CUDA_OK(cudaGetLastError());
  SelectArgs f{};
  f.sums = at<double>(ws, p.o_scores); f.n_cand = d->eq_n; f.n_keys = p.O; f.n_groups = p.O; f.keys_per_group = 1;
  f.inv_count = 1.0 / (double)p.L;                          // mean over the output positions, sum over the images (conv.py:548-549)
  f.gscale = at<float>(ws, p.o_gscale); f.factors = at<float>(ws, p.o_factors);
  f.d0 = at<float>(ws, p.o_d0); f.d = at<float>(ws, p.o_d); f.d_stride = 1; f.d_col = 0;
  f.best = at<int>(ws, p.o_best); f.score_log = score_log; f.has_next = 0;
  if ((rc = p4v_select_step(f, st))) return rc;
  P4V_CUDA_OK(cudaMemcpyAsync(w_interval, at<float>(ws, p.o_d), (size_t)p.O * 4, cudaMemcpyDeviceToDevice, st));
  return 0;
}
