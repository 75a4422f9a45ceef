// C-ABI for the head-wise MatMul scale-factor search (PTQSLBatchingQuantMatMul and the
// split-of-softmax variant).  Problem p = image * heads + head; the row operand is A[p]
// (S1 x S2), the column operand is B[p]^T (S3 x S2); one K segment (n_V = n_H = 1).
#include <algorithm>
#include <vector>

#include "../../include/ptq4vit_b200.h"
#include "plan.cuh"
#include "prep.cuh"

namespace {

struct MStep { int job_off, nfj, ncj, nfg, ncg, meta_fix, meta_cand; };

struct MMPlan {
  p4v_matmul_desc d;
  bool i8, sos;
  int ew, P, H, S1, S2, S3, tiles_m, tiles_n, A_qmax, B_qmax;
  int kb;        // padded K bytes of one part in the search operand type
  int kb16;      // padded K bytes in bf16 (split-search images)
  int KB_A, KB_B;            // row bytes of Acur / Bcur  (sos: Acur = [hi|lo])
  int KB_As, KB_Bs;          // split search: Acand = [hi|lo] bf16, Bsplit = [b1|b2|b3] bf16
  std::vector<P4VJob> jobs; std::vector<GroupMeta> metas;
  std::vector<P4VSeg> segA, segB, segAs, segBs;
  MStep stepA, stepB, stepS, fwd;
  std::vector<float> factors, split_factors;
  int n_split;
  size_t o_factors, o_sfactors, o_keys, o_dA0, o_dA, o_dB0, o_dB, o_ones, o_aux, o_split, o_gscale, o_scores, o_best,
      o_fix, o_candA, o_candB, o_jobs, o_metas, o_segA, o_segB, o_segAs, o_segBs, o_partial, o_Acur, o_Bcur, o_Acand,
      o_Bcand, o_Ascand, o_Bsplit, total;
};

int build_plan(const p4v_matmul_desc* d, MMPlan& p, bool with_search) {
  P4V_REQUIRE(d != nullptr, "null desc");
  p.d = *d;
  P4V_REQUIRE(d->batch > 0 && d->heads > 0 && d->S1 > 0 && d->S2 > 0 && d->S3 > 0, "matmul: empty shape");
  P4V_REQUIRE(d->A_bit >= 2 && d->A_bit <= 8 && d->B_bit >= 2 && d->B_bit <= 8, "matmul: bit widths must be in [2,8]");
  P4V_REQUIRE(d->eq_n >= 1 && d->eq_n <= P4V_MAX_CAND, "matmul: eq_n must be in [1,%d]", P4V_MAX_CAND);
  p.sos = d->sos != 0;
  p.H = d->heads; p.P = d->batch * d->heads; p.S1 = d->S1; p.S2 = d->S2; p.S3 = d->S3;
  p.A_qmax = 1 << (d->A_bit - 1); p.B_qmax = 1 << (d->B_bit - 1);
  p.tiles_m = p4v_cdiv(p.S1, P4V_TILE); p.tiles_n = p4v_cdiv(p.S3, P4V_TILE);
  p.i8 = use_int8(d->operand, p.S2);
  p.ew = p.i8 ? 1 : 2;
  p.kb = (int)align_up((size_t)p.S2 * p.ew, 32);
  p.kb16 = (int)align_up((size_t)p.S2 * 2, 32);
  p.KB_A = p.sos ? 2 * p.kb : p.kb; p.KB_B = p.kb;
  p.KB_As = 2 * p.kb16; p.KB_Bs = 3 * p.kb16;
  const float qa1 = (float)(p.A_qmax - 1);

  p.segA.clear(); p.segB.clear(); p.segAs.clear(); p.segBs.clear();
  if (p.sos) {
    p.segA.push_back(P4VSeg{0, p.S2, 0, 0, 0.f, 0.f, qa1, 1, qa1, 0, 0});
    p.segA.push_back(P4VSeg{0, p.S2, p.kb * P4V_TILE, 0, 0.f, 0.f, qa1, 2, qa1, 0, 0});
    p.segAs.push_back(P4VSeg{0, p.S2, 0, 0, 0.f, 0.f, qa1, 1, qa1, 0, 0});
    p.segAs.push_back(P4VSeg{0, p.S2, p.kb16 * P4V_TILE, 0, 0.f, 0.f, qa1, 2, qa1, 0, 0});
    for (int t = 0; t < 3; ++t) p.segBs.push_back(P4VSeg{0, p.S2, t * p.kb16 * P4V_TILE, 0, 0.f, 0.f, 0.f, 0, 0.f, t + 1, 0});
  } else {
    p.segA.push_back(P4VSeg{0, p.S2, 0, 0, 0.f, (float)-p.A_qmax, (float)(p.A_qmax - 1), 0, 0.f, 0, 0});
  }
  p.segB.push_back(P4VSeg{0, p.S2, 0, 0, 0.f, (float)-p.B_qmax, (float)(p.B_qmax - 1), 0, 0.f, 0, 0});

  p.factors = candidate_factors(d->eq_alpha, d->eq_beta, d->eq_n);
  p.n_split = 20;                                         // matmul.py:636
  p.split_factors.resize(p.n_split);
  for (int i = 0; i < p.n_split; ++i) p.split_factors[i] = (float)(1.0 / (double)(1u << i));

  p.jobs.clear(); p.metas.clear();
  p.stepA = p.stepB = p.stepS = p.fwd = MStep{};
  auto begin = [&](MStep& s) { s = MStep{}; s.job_off = (int)p.jobs.size(); s.meta_fix = (int)p.metas.size(); };
  if (with_search) {
    if (!p.sos) {   // A step: candidates on the row operand
      begin(p.stepA); p.stepA.meta_cand = (int)p.metas.size();
      push_jobs(p.jobs, 0, 0, p.kb, P4V_JOB_RCAND, 0, true, true, p.stepA.ncj);
      p.metas.push_back(GroupMeta{0, 0, 0, 0}); p.stepA.ncg = 1;
    } else {        // split search: (hi,lo)_c x exact 3-term bf16 split of the unquantised B
      begin(p.stepS); p.stepS.meta_cand = (int)p.metas.size();
      for (int part = 0; part < 2; ++part) {
        for (int t = 0; t < 3; ++t)
          push_jobs(p.jobs, part * p.kb16, t * p.kb16, p.kb16, P4V_JOB_RCAND, part, t == 0, t == 2, p.stepS.ncj);
        p.metas.push_back(GroupMeta{0, 0, 0, 0});        // both parts use aux[0] = 1/(qmax-1); lo also the candidate split
        ++p.stepS.ncg;
      }
    }
    begin(p.stepB); p.stepB.meta_cand = (int)p.metas.size();
    if (!p.sos) {
      push_jobs(p.jobs, 0, 0, p.kb, P4V_JOB_CCAND, 0, true, true, p.stepB.ncj);
      p.metas.push_back(GroupMeta{0, 0, 0, 0}); p.stepB.ncg = 1;
    } else {
      for (int part = 0; part < 2; ++part) {
        push_jobs(p.jobs, part * p.kb, 0, p.kb, P4V_JOB_CCAND, part, true, true, p.stepB.ncj);
        p.metas.push_back(GroupMeta{0, (short)part, 0, 0}); ++p.stepB.ncg;     // aux[0] = 1/(qmax-1), aux[1] = A_interval
      }
    }
    mark_resident(p.jobs, p.stepB.job_off + p.stepB.nfj, p.stepB.ncj);   // the B step's row operand (A) is candidate independent
  }
  begin(p.fwd);
  if (!p.sos) { push_jobs(p.jobs, 0, 0, p.kb, 0, 0, true, true, p.fwd.nfj); p.metas.push_back(GroupMeta{0, 0, 0, 0}); p.fwd.nfg = 1; }
  else for (int part = 0; part < 2; ++part) {
    push_jobs(p.jobs, part * p.kb, 0, p.kb, 0, part, true, true, p.fwd.nfj);
    p.metas.push_back(GroupMeta{0, (short)part, 0, 0}); ++p.fwd.nfg;
  }
  p.fwd.meta_cand = (int)p.metas.size();
  P4V_REQUIRE((int)p.jobs.size() <= 4 * P4V_MAX_JOBS && p.stepS.ncj <= P4V_MAX_JOBS && p.stepB.ncj <= P4V_MAX_JOBS &&
              p.stepA.ncj <= P4V_MAX_JOBS && p.fwd.nfj <= P4V_MAX_JOBS, "matmul: S2 too large");

  Carver w;
  const int n_c = std::max(d->eq_n, p.n_split);
  p.o_factors = w.take((d->eq_n + 1) * 4); p.o_sfactors = w.take(p.n_split * 4);
  p.o_keys = w.take((2 * p.H + 1) * 4);
  p.o_dA0 = w.take(p.H * 4); p.o_dA = w.take(p.H * 4); p.o_dB0 = w.take(p.H * 4); p.o_dB = w.take(p.H * 4);
  p.o_ones = w.take(p.H * 4); p.o_aux = w.take(2 * 4); p.o_split = w.take(4); p.o_gscale = w.take(4);
  p.o_scores = w.take((size_t)n_c * p.H * 8); p.o_best = w.take(p.H * 4);
  p.o_fix = w.take((size_t)2 * p.H * 4); p.o_candA = w.take((size_t)n_c * p.H * 4); p.o_candB = w.take((size_t)2 * p.H * 4);
  p.o_jobs = w.take(p.jobs.size() * sizeof(P4VJob)); p.o_metas = w.take(p.metas.size() * sizeof(GroupMeta));
  p.o_segA = w.take(p.segA.size() * sizeof(P4VSeg)); p.o_segB = w.take(p.segB.size() * sizeof(P4VSeg));
  p.o_segAs = w.take(std::max<size_t>(1, p.segAs.size()) * sizeof(P4VSeg));
  p.o_segBs = w.take(std::max<size_t>(1, p.segBs.size()) * sizeof(P4VSeg));
  const size_t tilesA = (size_t)p.P * p.tiles_m, tilesB = (size_t)p.P * p.tiles_n;
  p.o_partial = w.take(with_search ? tilesA * p.tiles_n * n_c * 32 * 4 : 4);
  p.o_Acur = w.take(tilesA * P4V_TILE * p.KB_A);
  p.o_Bcur = w.take(tilesB * P4V_TILE * p.KB_B);
  p.o_Acand = w.take(with_search && !p.sos ? (size_t)d->eq_n * tilesA * P4V_TILE * p.KB_A : 4);
  p.o_Bcand = w.take(with_search ? (size_t)d->eq_n * tilesB * P4V_TILE * p.KB_B : 4);
  p.o_Ascand = w.take(with_search && p.sos ? (size_t)p.n_split * tilesA * P4V_TILE * p.KB_As : 4);
  p.o_Bsplit = w.take(with_search && p.sos ? tilesB * P4V_TILE * p.KB_Bs : 4);
  p.total = w.total;
  return 0;
}

int upload_tables(const MMPlan& p, void* ws, cudaStream_t st) {
  int rc;
  if ((rc = upload(ws, p.o_factors, p.factors, st)) || (rc = upload(ws, p.o_sfactors, p.split_factors, st)) ||
      (rc = upload(ws, p.o_jobs, p.jobs, st)) || (rc = upload(ws, p.o_metas, p.metas, st)) ||
      (rc = upload(ws, p.o_segA, p.segA, st)) || (rc = upload(ws, p.o_segB, p.segB, st)) ||
      (rc = upload(ws, p.o_segAs, p.segAs, st)) || (rc = upload(ws, p.o_segBs, p.segBs, st)) ||
      (rc = upload(ws, p.o_ones, std::vector<float>(p.H, 1.f), st))) return rc;
  return 0;
}

// The operand images quant() writes: the current A / B images, their candidate planes, and the two bf16 images of the
// split search (A's split candidates, the exact three-term split of B).
enum Image { A_CUR, A_CAND, B_CUR, B_CAND, A_SPLIT_CAND, B_SPLIT };

int quant(const MMPlan& p, void* ws, Image which, const float* src, cudaStream_t st) {
  QuantImageArgs q{};
  const bool isA = which == A_CUR || which == A_CAND || which == A_SPLIT_CAND;
  q.src = src; q.P = p.P; q.prob_stride = isA ? (long long)p.S1 * p.S2 : (long long)p.S2 * p.S3;
  q.src_transposed = isA ? 0 : 1; q.ld = isA ? p.S2 : p.S3;
  q.rows = isA ? p.S1 : p.S3; q.tiles = isA ? p.tiles_m : p.tiles_n;
  q.rows_per_block = 0; q.d_mod = p.H; q.d_stride = 1;
  q.is_int8 = p.i8; q.n_planes = 1; q.factors = nullptr; q.split = at<float>(ws, p.o_split);
  int KB = 0;
  switch (which) {
    case A_CUR: q.dst = at<uint8_t>(ws, p.o_Acur); KB = p.KB_A; q.delta = at<float>(ws, p.o_dA); q.segs = at<P4VSeg>(ws, p.o_segA); q.nseg = (int)p.segA.size(); break;
    case A_CAND: q.dst = at<uint8_t>(ws, p.o_Acand); KB = p.KB_A; q.delta = at<float>(ws, p.o_dA0); q.segs = at<P4VSeg>(ws, p.o_segA); q.nseg = (int)p.segA.size();
            q.n_planes = p.d.eq_n; q.factors = at<float>(ws, p.o_factors); break;
    case B_CUR: q.dst = at<uint8_t>(ws, p.o_Bcur); KB = p.KB_B; q.delta = at<float>(ws, p.o_dB); q.segs = at<P4VSeg>(ws, p.o_segB); q.nseg = 1; break;
    case B_CAND: q.dst = at<uint8_t>(ws, p.o_Bcand); KB = p.KB_B; q.delta = at<float>(ws, p.o_dB0); q.segs = at<P4VSeg>(ws, p.o_segB); q.nseg = 1;
            q.n_planes = p.d.eq_n; q.factors = at<float>(ws, p.o_factors); break;
    case A_SPLIT_CAND: q.dst = at<uint8_t>(ws, p.o_Ascand); KB = p.KB_As; q.delta = at<float>(ws, p.o_dA0); q.segs = at<P4VSeg>(ws, p.o_segAs); q.nseg = 2;
            q.n_planes = p.n_split; q.factors = at<float>(ws, p.o_sfactors); q.is_int8 = 0; break;
    case B_SPLIT: q.dst = at<uint8_t>(ws, p.o_Bsplit); KB = p.KB_Bs; q.delta = at<float>(ws, p.o_dB0); q.segs = at<P4VSeg>(ws, p.o_segBs); q.nseg = 3; q.is_int8 = 0; break;
  }
  q.tile_bytes = (unsigned long long)P4V_TILE * KB;
  q.plane_stride = q.tile_bytes * q.tiles * p.P;
  return p4v_quant_image(q, st);
}

void fill_sweep(const MMPlan& p, void* ws, const MStep& s, SweepParams& sp) {
  sp = SweepParams{};
  sp.R_cur = at<uint8_t>(ws, p.o_Acur); sp.C_cur = at<uint8_t>(ws, p.o_Bcur);
  sp.R_cand = at<uint8_t>(ws, p.o_Acand); sp.C_cand = at<uint8_t>(ws, p.o_Bcand);
  sp.R_tile_bytes = sp.R_cand_tile_bytes = (unsigned long long)P4V_TILE * p.KB_A;
  sp.C_tile_bytes = sp.C_cand_tile_bytes = (unsigned long long)P4V_TILE * p.KB_B;
  sp.R_cand_stride = sp.R_cand_tile_bytes * p.tiles_m * p.P; sp.C_cand_stride = sp.C_cand_tile_bytes * p.tiles_n * p.P;
  sp.P = p.P; sp.M = p.S1; sp.N = p.S3; sp.tiles_m = p.tiles_m; sp.tiles_n = p.tiles_n;
  sp.ld = p.S3; sp.prob_stride = (long long)p.S1 * p.S3;
  sp.gscale = at<float>(ws, p.o_gscale);
  sp.jobs = at<P4VJob>(ws, p.o_jobs) + s.job_off;
  sp.n_fixed_jobs = s.nfj; sp.n_cand_jobs = s.ncj; sp.n_fixed_groups = s.nfg; sp.n_cand_groups = s.ncg;
  sp.fix_scale = at<float>(ws, p.o_fix); sp.candA = at<float>(ws, p.o_candA); sp.candB = at<float>(ws, p.o_candB);
  sp.nsg = p.H; sp.sg_mode = P4V_SG_PROBLEM;
  sp.n_cand = p.d.eq_n; sp.partial = at<float>(ws, p.o_partial); sp.is_int8 = p.i8;
}

int run_sweep(const MMPlan& p, const MStep& s, const SweepParams& sp, cudaStream_t st) {
  return p4v_run_sweep(sp, p.jobs.data() + s.job_off, p.d.kernel, st);
}

// kind 2: searched operand tables (d0, cur other) per head ; kind 3: other operand = aux[meta.a]
int tables(const MMPlan& p, void* ws, const MStep& s, int kind, const float* d_search0, const float* d_fixed_w,
           const float* d_other, const float* factors, int n_cand, cudaStream_t st) {
  StepTablesArgs t{};
  t.kind = kind; t.target = 0;
  t.dW = d_fixed_w; t.dW0 = d_search0; t.n_V = p.H; t.n_H = 1; t.crb_rows = P4V_CG;
  t.dX = d_other; t.dX0 = d_other; t.n_a = 1; t.d_neg = 0.f;
  t.factors = factors; t.n_cand = n_cand;
  t.fixed_meta = at<GroupMeta>(ws, p.o_metas) + s.meta_fix; t.n_fixed_groups = s.nfg;
  t.cand_meta = at<GroupMeta>(ws, p.o_metas) + s.meta_cand; t.n_cand_groups = s.ncg;
  t.nsg = p.H;
  t.fix_scale = at<float>(ws, p.o_fix); t.candA = at<float>(ws, p.o_candA); t.candB = at<float>(ws, p.o_candB);
  return p4v_step_tables(t, st);
}

__global__ void sos_aux_kernel(const float* split, float qm1, float* aux, float* A_interval_out) {
  aux[0] = __fdiv_rn(1.f, qm1);
  aux[1] = __fdiv_rn(split[0], qm1);       // A_interval = split / (A_qmax - 1)   (matmul.py:629)
  if (A_interval_out) A_interval_out[0] = aux[1];
}
__global__ void set_scalar_kernel(float* p, float v) { p[0] = v; }

int reduce_finish(const MMPlan& p, void* ws, const SweepParams& sp, int n_cand, int n_groups, double inv_count,
                  const float* factors, const float* d0, float* d, float* score_log, cudaStream_t st) {
  ReduceArgs r{};
  r.partial = sp.partial; r.n_cand = n_cand; r.P = p.P; r.tiles_m = p.tiles_m; r.tiles_n = p.tiles_n; r.order = sp.order;
  r.mode = P4V_SG_PROBLEM; r.n_keys = p.H; r.sums = at<double>(ws, p.o_scores);
  int rc = p4v_reduce_scores(r, st);
  if (rc) return rc;
  SelectArgs f{};     // no image commit: the current image is re-quantised from the fp32 source with the chosen step size
  f.sums = r.sums; f.n_cand = n_cand; f.n_keys = p.H; f.n_groups = n_groups; f.keys_per_group = n_groups == 1 ? p.H : 1;
  f.inv_count = inv_count; f.gscale = at<float>(ws, p.o_gscale); f.factors = factors;
  f.d0 = d0; f.d = d; f.d_stride = 1; f.d_col = 0; f.best = at<int>(ws, p.o_best); f.score_log = score_log;
  f.has_next = 0;
  return p4v_select_step(f, st);
}

int search_A(const MMPlan& p, void* ws, const float* A, const float* Y, const float* G, float* log, cudaStream_t st) {
  int rc;
  if ((rc = tables(p, ws, p.stepA, 2, at<float>(ws, p.o_dA0), at<float>(ws, p.o_dA), at<float>(ws, p.o_dB),
                   at<float>(ws, p.o_factors), p.d.eq_n, st))) return rc;
  SweepParams sp; fill_sweep(p, ws, p.stepA, sp);
  sp.Y = Y; sp.Gr = G; sp.order = 1;
  if ((rc = run_sweep(p, p.stepA, sp, st))) return rc;
  if ((rc = reduce_finish(p, ws, sp, p.d.eq_n, p.H, 1.0 / ((double)p.S1 * p.S3), at<float>(ws, p.o_factors),
                          at<float>(ws, p.o_dA0), at<float>(ws, p.o_dA), log, st))) return rc;
  return quant(p, ws, A_CUR, A, st);
}

int search_B(const MMPlan& p, void* ws, const float* B, const float* Y, const float* G, float* log, cudaStream_t st) {
  int rc;
  if ((rc = tables(p, ws, p.stepB, p.sos ? 3 : 2, at<float>(ws, p.o_dB0), at<float>(ws, p.o_dB),
                   p.sos ? at<float>(ws, p.o_aux) : at<float>(ws, p.o_dA), at<float>(ws, p.o_factors), p.d.eq_n, st))) return rc;
  SweepParams sp; fill_sweep(p, ws, p.stepB, sp);
  sp.Y = Y; sp.Gr = G; sp.order = 0;
  if ((rc = run_sweep(p, p.stepB, sp, st))) return rc;
  if ((rc = reduce_finish(p, ws, sp, p.d.eq_n, p.H, 1.0 / ((double)p.S1 * p.S3), at<float>(ws, p.o_factors),
                          at<float>(ws, p.o_dB0), at<float>(ws, p.o_dB), log, st))) return rc;
  return quant(p, ws, B_CUR, B, st);
}

int search_split(const MMPlan& p, void* ws, const float* A, const float* Y, const float* G, float* log, cudaStream_t st) {
  int rc;
  // candA[c][head] = split_c * 1, candB[g][head] = aux[0] = 1/(qmax-1); the high part ignores candA
  if ((rc = tables(p, ws, p.stepS, 3, at<float>(ws, p.o_ones), at<float>(ws, p.o_ones), at<float>(ws, p.o_aux),
                   at<float>(ws, p.o_sfactors), p.n_split, st))) return rc;
  SweepParams sp; fill_sweep(p, ws, p.stepS, sp);
  sp.Y = Y; sp.Gr = G; sp.order = 1; sp.n_cand = p.n_split; sp.is_int8 = 0; sp.cand_noA_mask = 1ull;
  sp.R_cand = at<uint8_t>(ws, p.o_Ascand); sp.R_cand_tile_bytes = (unsigned long long)P4V_TILE * p.KB_As;
  sp.R_cand_stride = sp.R_cand_tile_bytes * p.tiles_m * p.P;
  sp.C_cur = at<uint8_t>(ws, p.o_Bsplit); sp.C_tile_bytes = (unsigned long long)P4V_TILE * p.KB_Bs;
  if ((rc = run_sweep(p, p.stepS, sp, st))) return rc;
  // global score: mean over heads and rows (matmul.py:620-621)
  if ((rc = reduce_finish(p, ws, sp, p.n_split, 1, 1.0 / ((double)p.H * p.S1 * p.S3), at<float>(ws, p.o_sfactors),
                          at<float>(ws, p.o_ones), at<float>(ws, p.o_split), log, st))) return rc;
  sos_aux_kernel<<<1, 1, 0, st>>>(at<float>(ws, p.o_split), (float)(p.A_qmax - 1), at<float>(ws, p.o_aux), nullptr);
  p4v_count_launch();
  P4V_CUDA_OK(cudaGetLastError());
  return quant(p, ws, A_CUR, A, st);
}

int begin(const MMPlan& p, void* ws, const float* A, const float* B, const float* G, cudaStream_t st) {
  int rc;
  if ((rc = upload_tables(p, ws, st))) return rc;
  int* keys = at<int>(ws, p.o_keys);
  if ((rc = p4v_keys_reset(keys, 2 * p.H + 1, st))) return rc;
  if ((rc = p4v_group_absmax(A, (long long)p.S1 * p.S2, p.P, p.H, keys, st))) return rc;
  if ((rc = p4v_group_absmax(B, (long long)p.S2 * p.S3, p.P, p.H, keys + p.H, st))) return rc;
  if ((rc = p4v_group_absmax(G, (long long)p.P * p.S1 * p.S3, 1, 1, keys + 2 * p.H, st))) return rc;
  if (p.d.init_layerwise) {       // matmul.py:430-432
    if ((rc = p4v_keys_broadcast_max(keys, p.H, st))) return rc;
    if ((rc = p4v_keys_broadcast_max(keys + p.H, p.H, st))) return rc;
  }
  if ((rc = p4v_keys_to_delta(keys, p.H, (float)p.A_qmax - 0.5f, at<float>(ws, p.o_dA0), at<float>(ws, p.o_dA), st))) return rc;
  if ((rc = p4v_keys_to_delta(keys + p.H, p.H, (float)p.B_qmax - 0.5f, at<float>(ws, p.o_dB0), at<float>(ws, p.o_dB), st))) return rc;
  if ((rc = p4v_make_gscale(keys + 2 * p.H, at<float>(ws, p.o_gscale), st))) return rc;
  if (p.sos) {
    set_scalar_kernel<<<1, 1, 0, st>>>(at<float>(ws, p.o_split), 0.01f);       // matmul.py:354-355 (dead: overwritten by the first search)
    sos_aux_kernel<<<1, 1, 0, st>>>(at<float>(ws, p.o_split), (float)(p.A_qmax - 1), at<float>(ws, p.o_aux), nullptr);
    P4V_CUDA_OK(cudaGetLastError());
    if ((rc = quant(p, ws, A_SPLIT_CAND, A, st))) return rc;
    if ((rc = quant(p, ws, B_SPLIT, B, st))) return rc;
  } else {
    if ((rc = quant(p, ws, A_CAND, A, st))) return rc;
  }
  if ((rc = quant(p, ws, A_CUR, A, st))) return rc;
  if ((rc = quant(p, ws, B_CUR, B, st))) return rc;
  if ((rc = quant(p, ws, B_CAND, B, st))) return rc;
  return 0;
}

}  // namespace

extern "C" int p4v_matmul_workspace_bytes(const p4v_matmul_desc* d, size_t* bytes) {
  return plan_workspace_bytes(build_plan, d, bytes, true);
}

extern "C" int p4v_matmul_score_log_floats(const p4v_matmul_desc* d, size_t* n) {
  P4V_REQUIRE(d && n, "null argument");
  *n = (size_t)d->search_round * ((d->sos ? (size_t)20 : (size_t)d->eq_n * d->heads) + (size_t)d->eq_n * d->heads);
  return 0;
}

extern "C" int p4v_matmul_calibrate(const p4v_matmul_desc* d, const float* A, const float* B, const float* raw_out,
                                    const float* raw_grad, void* workspace, size_t workspace_bytes, float* A_interval,
                                    float* B_interval, float* split, float* score_log, void* stream) {
  MMPlan p; int rc = build_plan(d, p, true);
  if (rc) return rc;
  P4V_REQUIRE(A && B && raw_out && raw_grad && workspace && A_interval && B_interval, "matmul_calibrate: null pointer");
  P4V_REQUIRE(!p.sos || split, "matmul_calibrate: sos needs the split output");
  P4V_REQUIRE(workspace_bytes >= p.total, "matmul_calibrate: workspace too small (%zu < %zu)", workspace_bytes, p.total);
  cudaStream_t st = (cudaStream_t)stream;
  if ((rc = begin(p, workspace, A, B, raw_grad, st))) return rc;
  for (int e = 0; e < d->search_round; ++e) {
    if (p.sos) {
      if ((rc = search_split(p, workspace, A, raw_out, raw_grad, score_log, st))) return rc;
      if (score_log) score_log += p.n_split;
    } else {
      if ((rc = search_A(p, workspace, A, raw_out, raw_grad, score_log, st))) return rc;
      if (score_log) score_log += (size_t)d->eq_n * p.H;
    }
    if ((rc = search_B(p, workspace, B, raw_out, raw_grad, score_log, st))) return rc;
    if (score_log) score_log += (size_t)d->eq_n * p.H;
  }
  if (p.sos) {
    P4V_CUDA_OK(cudaMemcpyAsync(split, at<float>(workspace, p.o_split), 4, cudaMemcpyDeviceToDevice, st));
    P4V_CUDA_OK(cudaMemcpyAsync(A_interval, at<float>(workspace, p.o_aux) + 1, 4, cudaMemcpyDeviceToDevice, st));
  } else {
    P4V_CUDA_OK(cudaMemcpyAsync(A_interval, at<float>(workspace, p.o_dA), (size_t)p.H * 4, cudaMemcpyDeviceToDevice, st));
  }
  P4V_CUDA_OK(cudaMemcpyAsync(B_interval, at<float>(workspace, p.o_dB), (size_t)p.H * 4, cudaMemcpyDeviceToDevice, st));
  return 0;
}

extern "C" int p4v_matmul_quant_forward_workspace_bytes(const p4v_matmul_desc* d, size_t* bytes) {
  return plan_workspace_bytes(build_plan, d, bytes, false);
}

extern "C" int p4v_matmul_quant_forward(const p4v_matmul_desc* d, const float* A, const float* B, const float* A_interval,
                                        const float* B_interval, const float* split, void* workspace, size_t workspace_bytes,
                                        float* out, void* stream) {
  MMPlan p; int rc = build_plan(d, p, false);
  if (rc) return rc;
  P4V_REQUIRE(A && B && A_interval && B_interval && workspace && out, "matmul_quant_forward: null pointer");
  P4V_REQUIRE(!p.sos || split, "matmul_quant_forward: sos needs split");
  P4V_REQUIRE(workspace_bytes >= p.total, "matmul_quant_forward: workspace too small (%zu < %zu)", workspace_bytes, p.total);
  cudaStream_t st = (cudaStream_t)stream;
  if ((rc = upload_tables(p, workspace, st))) return rc;
  P4V_CUDA_OK(cudaMemcpyAsync(at<float>(workspace, p.o_dB), B_interval, (size_t)p.H * 4, cudaMemcpyDeviceToDevice, st));
  if (p.sos) {
    P4V_CUDA_OK(cudaMemcpyAsync(at<float>(workspace, p.o_split), split, 4, cudaMemcpyDeviceToDevice, st));
    sos_aux_kernel<<<1, 1, 0, st>>>(at<float>(workspace, p.o_split), (float)(p.A_qmax - 1), at<float>(workspace, p.o_aux), nullptr);
    P4V_CUDA_OK(cudaGetLastError());
  } else {
    P4V_CUDA_OK(cudaMemcpyAsync(at<float>(workspace, p.o_dA), A_interval, (size_t)p.H * 4, cudaMemcpyDeviceToDevice, st));
  }
  if ((rc = quant(p, workspace, A_CUR, A, st))) return rc;
  if ((rc = quant(p, workspace, B_CUR, B, st))) return rc;
  // fixed scale per head: plain dA*dB ; sos: dB * aux[part]
  if ((rc = tables(p, workspace, p.fwd, p.sos ? 3 : 2, at<float>(workspace, p.o_dB0),
                   p.sos ? at<float>(workspace, p.o_dB) : at<float>(workspace, p.o_dA),
                   p.sos ? at<float>(workspace, p.o_aux) : at<float>(workspace, p.o_dB), at<float>(workspace, p.o_factors), 0, st))) return rc;
  SweepParams sp; fill_sweep(p, workspace, p.fwd, sp);
  sp.out = out; sp.n_cand = 1; sp.order = 0; sp.R_cand = nullptr; sp.C_cand = nullptr;
  return run_sweep(p, p.fwd, sp, st);
}
