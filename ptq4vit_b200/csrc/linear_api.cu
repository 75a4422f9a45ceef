// C-ABI for the Linear scale-factor search: host-side planning (segments, jobs,
// workspace carving) + the per-step launch sequence.  See include/ptq4vit_b200.h.
#include <algorithm>
#include <cstdlib>
#include <vector>

#include "../../include/ptq4vit_b200.h"
#include "plan.cuh"
#include "prep.cuh"
#include "gram.cuh"

namespace {

struct BSeg { int k0, klen, h, a, kb; int woff, xoff_p, xoff_n, xcoff; };   // offsets: bytes in the padded row
struct Step { int job_off, nfj, ncj, nfg, ncg, meta_fix, meta_cand, commit_off, ncommit, commit_chunks; };

struct LinPlan {
  p4v_linear_desc d;
  bool i8, twin;
  int ew, M, K, O, tiles_m, tiles_o, nsg, crb_rows, crb_cols, crb_acts, w_qmax, a_qmax;
  float d_neg;
  std::vector<BSeg> segs;
  int KB_W, KB_X, KB_Xc;
  std::vector<P4VJob> jobs; std::vector<GroupMeta> metas; std::vector<CommitSeg> commits;
  std::vector<P4VSeg> segsW, segsX, segsXc, segsG;
  std::vector<Step> wsteps, xsteps;
  Step fwd;   // quant_forward: every segment is a fixed group
  // normal-equation W search (gram.cu)
  bool gram; int g_ks, g_Mp, g_npairs, g_tiles_p, g_ldH, g_nmblk; unsigned g_term_bytes;
  size_t o_E, o_XqT, o_G2T, o_Z, o_H, o_Upart, o_E2part, o_U, o_E2, o_dprev, o_D, o_segsG;
  int g_osplit, g_opb;
  std::vector<float> factors;
  int max_groups;
  // workspace offsets
  size_t o_factors, o_keys, o_dW0, o_dW, o_dX0, o_dX, o_gscale, o_scores, o_best, o_fix, o_candA, o_candB, o_jobs,
      o_metas, o_segsW, o_segsX, o_segsXc, o_commits, o_partial, o_Wcur, o_Xcur, o_Wcand, o_Xcand, total;
};

// Merge runs of single-job accumulator groups whose K slabs are adjacent in BOTH operand images into one
// stage load with several sub-accumulators (one bulk copy / one stage handshake for up to 128 bytes of K).
void batch_jobs(LinPlan& p, int first, int& count) {
  std::vector<P4VJob> out;
  for (int j = 0; j < count; ++j) {
    const P4VJob jb = p.jobs[first + j];
    const bool single = (jb.flags & P4V_JOB_FIRST) && (jb.flags & P4V_JOB_LAST) && !(jb.flags & (P4V_JOB_RRES | P4V_JOB_CCAND));
    if (single && !out.empty()) {
      P4VJob& prev = out.back();
      const unsigned n = p4v_job_nsub(prev);
      const bool prev_single = (prev.flags & P4V_JOB_FIRST) && (prev.flags & P4V_JOB_LAST);
      if (prev_single && prev.flags == jb.flags && prev.kb == jb.kb && (n + 1) * jb.kb <= P4V_JOB_KB &&
          prev.r_off + n * jb.kb * P4V_TILE == jb.r_off && prev.c_off + n * jb.kb * P4V_TILE == jb.c_off &&
          prev.group + n == jb.group) {
        prev.nsub = (uint8_t)(n + 1);
        continue;
      }
    }
    out.push_back(jb);
  }
  std::copy(out.begin(), out.end(), p.jobs.begin() + first);
  p.jobs.erase(p.jobs.begin() + first + out.size(), p.jobs.begin() + first + count);
  count = (int)out.size();
}

int build_plan(const p4v_linear_desc* d, LinPlan& p, bool with_search) {
  P4V_REQUIRE(d != nullptr, "null desc");
  p.d = *d;
  p.M = d->rows; p.K = d->in_features; p.O = d->out_features;
  P4V_REQUIRE(p.M > 0 && p.K > 0 && p.O > 0, "linear: empty shape (rows=%d in=%d out=%d)", p.M, p.K, p.O);
  P4V_REQUIRE(d->n_V >= 1 && d->n_H >= 1 && d->n_a >= 1, "linear: n_V/n_H/n_a must be >= 1");
  P4V_REQUIRE(p.K % d->n_H == 0 && p.K % d->n_a == 0 && p.O % d->n_V == 0,
              "linear: in_features must divide by n_H and n_a, out_features by n_V (reference views, linear.py:117-119)");
  P4V_REQUIRE(d->tokens >= 1 && p.M % d->tokens == 0, "linear: rows must be a multiple of tokens");
  P4V_REQUIRE(d->w_bit >= 2 && d->w_bit <= 8 && d->a_bit >= 2 && d->a_bit <= 8, "linear: bit widths must be in [2,8]");
  P4V_REQUIRE(d->eq_n >= 1 && d->eq_n <= P4V_MAX_CAND, "linear: eq_n must be in [1,%d]", P4V_MAX_CAND);
  p.crb_rows = p.O / d->n_V; p.crb_cols = p.K / d->n_H; p.crb_acts = p.K / d->n_a;
  P4V_REQUIRE(d->n_V == 1 || p.crb_rows % P4V_CG == 0, "linear: out_features/n_V must be a multiple of 16 (got %d)", p.crb_rows);
  p.w_qmax = 1 << (d->w_bit - 1); p.a_qmax = 1 << (d->a_bit - 1);
  p.twin = d->post_gelu != 0;
  p.d_neg = (float)(0.16997124254703522 / (double)p.a_qmax);
  p.tiles_m = p4v_cdiv(p.M, P4V_TILE); p.tiles_o = p4v_cdiv(p.O, P4V_TILE);
  p.nsg = p.tiles_o * P4V_TILE_CG;

  // K segments = intersections of the weight column blocks and the activation chunks
  std::vector<int> cuts;
  for (int h = 0; h <= d->n_H; ++h) cuts.push_back(h * p.crb_cols);
  for (int a = 0; a <= d->n_a; ++a) cuts.push_back(a * p.crb_acts);
  std::sort(cuts.begin(), cuts.end());
  cuts.erase(std::unique(cuts.begin(), cuts.end()), cuts.end());
  int min_len = p.K;
  for (size_t i = 0; i + 1 < cuts.size(); ++i) min_len = std::min(min_len, cuts[i + 1] - cuts[i]);
  p.i8 = use_int8(d->operand, min_len);
  p.ew = p.i8 ? 1 : 2;
  p.segs.clear();
  int off = 0;
  for (size_t i = 0; i + 1 < cuts.size(); ++i) {
    BSeg s{};
    s.k0 = cuts[i]; s.klen = cuts[i + 1] - cuts[i];
    s.h = s.k0 / p.crb_cols; s.a = s.k0 / p.crb_acts;
    s.kb = (int)align_up((size_t)s.klen * p.ew, 32);
    s.woff = off; s.xoff_p = off; s.xcoff = off;
    off += s.kb;
    p.segs.push_back(s);
  }
  p.KB_W = off; p.KB_Xc = off;
  p.KB_X = p.twin ? 2 * off : off;
  for (auto& s : p.segs) s.xoff_n = p.twin ? off + s.xoff_p : -1;
  P4V_REQUIRE((size_t)p.KB_X * P4V_TILE < (1ull << 32), "linear: in_features too large");

  // quantisation segment tables
  p.segsW.clear(); p.segsX.clear(); p.segsXc.clear(); p.segsG.clear();
  for (auto& s : p.segs) {
    P4VSeg w{s.k0, s.klen, s.woff * P4V_TILE, s.h, 0.f, (float)-p.w_qmax, (float)(p.w_qmax - 1), 0, 0.f, 0, 0};
    p.segsW.push_back(w);
    P4VSeg x{s.k0, s.klen, s.xoff_p * P4V_TILE, s.a, 0.f, p.twin ? 0.f : (float)-p.a_qmax, (float)(p.a_qmax - 1), 0, 0.f, 0, 0};
    p.segsX.push_back(x);
    P4VSeg xc = x; xc.dst_off = s.xcoff * P4V_TILE;
    p.segsXc.push_back(xc);
  }
  if (p.twin)
    for (auto& s : p.segs) {
      P4VSeg n{s.k0, s.klen, s.xoff_n * P4V_TILE, s.a, p.d_neg, (float)-p.a_qmax, 0.f, 0, 0.f, 0, 0};
      p.segsX.push_back(n);
    }

  p.factors = candidate_factors(d->eq_alpha, d->eq_beta, d->eq_n);

  // steps
  p.jobs.clear(); p.metas.clear(); p.commits.clear(); p.wsteps.clear(); p.xsteps.clear();
  p.max_groups = 1;
  auto begin_step = [&](Step& st) { st = Step{}; st.job_off = (int)p.jobs.size(); st.commit_off = (int)p.commits.size(); };
  auto fixed_group = [&](Step& st, const BSeg& s, bool neg) {
    push_jobs(p.jobs, neg ? s.xoff_n : s.xoff_p, s.woff, s.kb, 0, st.nfg, true, true, st.nfj);
    p.metas.push_back(GroupMeta{(short)s.h, (short)s.a, (short)(neg ? 1 : 0), 0});
    ++st.nfg;
  };
  if (with_search) {
    for (int h = 0; h < d->n_H; ++h) {
      Step st; begin_step(st);
      st.meta_fix = (int)p.metas.size();
      for (auto& s : p.segs) if (s.h != h) { fixed_group(st, s, false); if (p.twin) fixed_group(st, s, true); }
      st.meta_cand = (int)p.metas.size();
      for (auto& s : p.segs) if (s.h == h) {
        push_jobs(p.jobs, s.xoff_p, s.woff, s.kb, P4V_JOB_CCAND, st.ncg, true, true, st.ncj);
        p.metas.push_back(GroupMeta{(short)s.h, (short)s.a, 0, 0}); ++st.ncg;
        if (p.twin) {
          push_jobs(p.jobs, s.xoff_n, s.woff, s.kb, P4V_JOB_CCAND, st.ncg, true, true, st.ncj);
          p.metas.push_back(GroupMeta{(short)s.h, (short)s.a, 1, 0}); ++st.ncg;
        }
        p.commits.push_back(CommitSeg{s.woff * P4V_TILE, s.woff * P4V_TILE, s.kb});
        st.commit_chunks += s.kb / 16; ++st.ncommit;
      }
      mark_resident(p.jobs, st.job_off + st.nfj, st.ncj);
      batch_jobs(p, st.job_off, st.nfj);
      p.wsteps.push_back(st);
    }
    for (int a = 0; a < d->n_a; ++a) {
      Step st; begin_step(st);
      st.meta_fix = (int)p.metas.size();
      for (auto& s : p.segs) { if (s.a != a) fixed_group(st, s, false); if (p.twin) fixed_group(st, s, true); }
      st.meta_cand = (int)p.metas.size();
      for (auto& s : p.segs) if (s.a == a) {
        push_jobs(p.jobs, s.xcoff, s.woff, s.kb, P4V_JOB_RCAND, st.ncg, true, true, st.ncj);
        p.metas.push_back(GroupMeta{(short)s.h, (short)s.a, 0, 0}); ++st.ncg;
        p.commits.push_back(CommitSeg{s.xcoff * P4V_TILE, s.xoff_p * P4V_TILE, s.kb});
        st.commit_chunks += s.kb / 16; ++st.ncommit;
      }
      {   // candidates change the row operand only: keep the tile's weight image resident when it fits
        int ncj = st.ncj; batch_jobs(p, st.job_off + st.nfj, ncj); st.ncj = ncj;
        batch_jobs(p, st.job_off, st.nfj);
        if ((size_t)p.KB_W * P4V_TILE <= 100 * 1024)
          for (int j = 0; j < st.nfj + st.ncj; ++j) p.jobs[st.job_off + j].flags |= P4V_JOB_CRES;
      }
      p.xsteps.push_back(st);
    }
  }
  {
    Step st; begin_step(st);
    st.meta_fix = (int)p.metas.size();
    for (auto& s : p.segs) { fixed_group(st, s, false); if (p.twin) fixed_group(st, s, true); }
    st.meta_cand = (int)p.metas.size();
    batch_jobs(p, st.job_off, st.nfj);
    p.fwd = st;
  }
  auto check = [&](const Step& st) {
    return st.nfj + st.ncj <= P4V_MAX_JOBS && st.nfg <= P4V_MAX_GROUPS && st.ncg <= P4V_MAX_GROUPS;
  };
  for (auto& st : p.wsteps) { P4V_REQUIRE(check(st), "linear: too many K segments for one step (n_H/n_a/in_features)"); p.max_groups = std::max(p.max_groups, std::max(st.nfg, st.ncg)); }
  for (auto& st : p.xsteps) { P4V_REQUIRE(check(st), "linear: too many K segments for one step (n_H/n_a/in_features)"); p.max_groups = std::max(p.max_groups, std::max(st.nfg, st.ncg)); }
  P4V_REQUIRE(check(p.fwd), "linear: too many K segments for quant_forward");
  p.max_groups = std::max(p.max_groups, p.fwd.nfg);

  // workspace carving
  Carver w;
  const int n_c = d->eq_n;
  p.o_factors = w.take((n_c + 1) * 4);
  p.o_keys = w.take((d->n_V * d->n_H + d->n_a + 1) * 4);
  p.o_dW0 = w.take(d->n_V * d->n_H * 4); p.o_dW = w.take(d->n_V * d->n_H * 4);
  p.o_dX0 = w.take(d->n_a * 4); p.o_dX = w.take(d->n_a * 4);
  p.o_gscale = w.take(4);
  p.o_scores = w.take((size_t)n_c * (p.nsg + d->n_V * (size_t)(1 + p4v_cdiv(p.crb_rows, 2))) * 8);
  p.o_best = w.take(std::max(d->n_V, 1) * 4);
  p.o_fix = w.take((size_t)p.max_groups * p.nsg * 4);
  p.o_candA = w.take((size_t)n_c * p.nsg * 4);
  p.o_candB = w.take((size_t)p.max_groups * p.nsg * 4);
  p.o_jobs = w.take(p.jobs.size() * sizeof(P4VJob));
  p.o_metas = w.take(p.metas.size() * sizeof(GroupMeta));
  p.o_segsW = w.take(p.segsW.size() * sizeof(P4VSeg));
  p.o_segsX = w.take(p.segsX.size() * sizeof(P4VSeg));
  p.o_segsXc = w.take(p.segsXc.size() * sizeof(P4VSeg));
  p.o_commits = w.take(std::max<size_t>(1, p.commits.size()) * sizeof(CommitSeg));
  p.o_partial = w.take(with_search ? (size_t)p.tiles_m * p.tiles_o * n_c * 32 * 4 : 4);
  p.o_Wcur = w.take((size_t)p.tiles_o * P4V_TILE * p.KB_W);
  p.o_Xcur = w.take((size_t)p.tiles_m * P4V_TILE * p.KB_X);
  p.o_Wcand = w.take(with_search ? (size_t)n_c * p.tiles_o * P4V_TILE * p.KB_W : 4);
  p.o_Xcand = w.take(with_search ? (size_t)n_c * p.tiles_m * P4V_TILE * p.KB_Xc : 4);
  // normal-equation W search: narrow column blocks inside one activation chunk, plain (non twin) activations
  p.gram = false;
  {
    const char* env = getenv("P4V_GRAM");
    const bool want = with_search && (env ? atoi(env) != 0 : true) && d->kernel == P4V_KERNEL_TCGEN05;
    const unsigned term = (unsigned)align_up((size_t)p.M * 2, 32);
    if (want && !p.twin && p.crb_cols <= 64 && p.crb_cols % 4 == 0 && p.crb_acts % p.crb_cols == 0) {
      p.gram = true;
      p.g_ks = p.crb_cols; p.g_term_bytes = term;
      p.g_Mp = (int)align_up((size_t)p.M, 16) + 16;
      p.g_npairs = p.g_ks * (p.g_ks + 1) / 2;
      p.g_tiles_p = p4v_cdiv(p.g_npairs * d->n_H, GRAM_PT); p.g_ldH = p.g_tiles_p * GRAM_PT;   // all column blocks side by side
      p.g_nmblk = p4v_gram_update_splits(p.O, p.M);
      const size_t KBg = 2 * (size_t)term;
      p.o_E = w.take((size_t)p.M * p.O * 4);
      p.o_XqT = w.take((size_t)p.K * p.g_Mp);
      p.o_G2T = w.take((size_t)p.tiles_o * P4V_TILE * KBg);
      p.o_Z = w.take((size_t)p.g_tiles_p * GRAM_PT * KBg);
      p.o_H = w.take((size_t)p.O * p.g_ldH * 4);
      p.o_Upart = w.take((size_t)p.g_nmblk * p.O * p.g_ks * 4);
      p.o_E2part = w.take((size_t)p.g_nmblk * p.O * 4);
      p.o_U = w.take((size_t)p.O * p.g_ks * 4); p.o_E2 = w.take((size_t)p.O * 4);
      p.g_osplit = std::max(1, p4v_cdiv(p.crb_rows, 2)); p.g_opb = p4v_cdiv(p.crb_rows, p.g_osplit);
      p.o_dprev = w.take((size_t)d->n_V * 4);
      p.o_D = w.take((size_t)p.O * 64 * 4);
      // (gs*g)^2 as two exact bf16 terms side by side in each row
      p.segsG = {{0, p.M, 0, 0, 0.f, 0.f, 0.f, 0, 0.f, 1, 1}, {0, p.M, (int)(term * P4V_TILE), 0, 0.f, 0.f, 0.f, 0, 0.f, 2, 1}};
      p.o_segsG = w.take(p.segsG.size() * sizeof(P4VSeg));
    }
  }
  p.total = w.total;
  return 0;
}

int upload_tables(const LinPlan& p, void* ws, cudaStream_t st) {
  int rc;
  if ((rc = upload(ws, p.o_factors, p.factors, st)) || (rc = upload(ws, p.o_jobs, p.jobs, st)) ||
      (rc = upload(ws, p.o_metas, p.metas, st)) || (rc = upload(ws, p.o_segsW, p.segsW, st)) ||
      (rc = upload(ws, p.o_segsX, p.segsX, st)) || (rc = upload(ws, p.o_segsXc, p.segsXc, st)) ||
      (rc = upload(ws, p.o_commits, p.commits, st)) || (rc = upload(ws, p.o_segsG, p.segsG, st))) return rc;
  return 0;
}

int quant_W(const LinPlan& p, void* ws, const float* W, const float* delta, bool cand, cudaStream_t st) {
  QuantImageArgs q{};
  q.src = W; q.ld = p.K; q.prob_stride = 0; q.src_transposed = 0;
  q.P = 1; q.rows = p.O; q.tiles = p.tiles_o;
  q.dst = at<uint8_t>(ws, cand ? p.o_Wcand : p.o_Wcur);
  q.tile_bytes = (unsigned long long)P4V_TILE * p.KB_W; q.plane_stride = q.tile_bytes * p.tiles_o;
  q.n_planes = cand ? p.d.eq_n : 1;
  q.factors = cand ? at<float>(ws, p.o_factors) : nullptr;
  q.delta = delta; q.rows_per_block = p.crb_rows; q.d_stride = p.d.n_H; q.d_mod = 1;
  q.segs = at<P4VSeg>(ws, p.o_segsW); q.nseg = (int)p.segsW.size(); q.is_int8 = p.i8;
  return p4v_quant_image(q, st);
}

int quant_X(const LinPlan& p, void* ws, const float* x, const float* delta, bool cand, cudaStream_t st) {
  QuantImageArgs q{};
  q.src = x; q.ld = p.K; q.prob_stride = 0; q.src_transposed = 0;
  q.P = 1; q.rows = p.M; q.tiles = p.tiles_m;
  q.dst = at<uint8_t>(ws, cand ? p.o_Xcand : p.o_Xcur);
  q.tile_bytes = (unsigned long long)P4V_TILE * (cand ? p.KB_Xc : p.KB_X); q.plane_stride = q.tile_bytes * p.tiles_m;
  q.n_planes = cand ? p.d.eq_n : 1;
  q.factors = cand ? at<float>(ws, p.o_factors) : nullptr;
  q.delta = delta; q.rows_per_block = p.M + P4V_TILE; q.d_stride = 0; q.d_mod = 1;   // single row block
  q.segs = at<P4VSeg>(ws, cand ? p.o_segsXc : p.o_segsX); q.nseg = (int)(cand ? p.segsXc.size() : p.segsX.size());
  q.is_int8 = p.i8;
  return p4v_quant_image(q, st);
}

void fill_sweep(const LinPlan& p, void* ws, const Step& s, SweepParams& sp) {
  sp = SweepParams{};
  sp.R_cur = at<uint8_t>(ws, p.o_Xcur); sp.R_cand = at<uint8_t>(ws, p.o_Xcand);
  sp.C_cur = at<uint8_t>(ws, p.o_Wcur); sp.C_cand = at<uint8_t>(ws, p.o_Wcand);
  sp.R_tile_bytes = (unsigned long long)P4V_TILE * p.KB_X; sp.C_tile_bytes = (unsigned long long)P4V_TILE * p.KB_W;
  sp.R_cand_tile_bytes = (unsigned long long)P4V_TILE * p.KB_Xc; sp.C_cand_tile_bytes = sp.C_tile_bytes;
  sp.R_cand_stride = sp.R_cand_tile_bytes * p.tiles_m; sp.C_cand_stride = sp.C_cand_tile_bytes * p.tiles_o;
  sp.P = 1; sp.M = p.M; sp.N = p.O; sp.tiles_m = p.tiles_m; sp.tiles_n = p.tiles_o;
  sp.ld = p.O; sp.prob_stride = 0;
  sp.gscale = at<float>(ws, p.o_gscale);
  sp.jobs = at<P4VJob>(ws, p.o_jobs) + s.job_off;
  sp.n_fixed_jobs = s.nfj; sp.n_cand_jobs = s.ncj; sp.n_fixed_groups = s.nfg; sp.n_cand_groups = s.ncg;
  sp.fix_scale = at<float>(ws, p.o_fix); sp.candA = at<float>(ws, p.o_candA); sp.candB = at<float>(ws, p.o_candB);
  sp.nsg = p.nsg; sp.sg_mode = P4V_SG_COLUMN;
  sp.n_cand = p.d.eq_n;
  sp.partial = at<float>(ws, p.o_partial);
  sp.is_int8 = p.i8;
}

int run_sweep(const LinPlan& p, const Step& s, const SweepParams& sp, cudaStream_t st) {
  return p4v_run_sweep(sp, p.jobs.data() + s.job_off, p.d.kernel, st);
}

StepTablesArgs tables_args(const LinPlan& p, void* ws, const Step& s, int kind, int target) {
  StepTablesArgs t{};
  t.kind = kind < 0 ? 0 : kind; t.target = target;
  t.dW = at<float>(ws, p.o_dW); t.dW0 = at<float>(ws, p.o_dW0); t.n_V = p.d.n_V; t.n_H = p.d.n_H; t.crb_rows = p.crb_rows;
  t.dX = at<float>(ws, p.o_dX); t.dX0 = at<float>(ws, p.o_dX0); t.n_a = p.d.n_a; t.d_neg = p.d_neg;
  t.factors = at<float>(ws, p.o_factors); t.n_cand = kind < 0 ? 0 : p.d.eq_n;
  t.fixed_meta = at<GroupMeta>(ws, p.o_metas) + s.meta_fix; t.n_fixed_groups = s.nfg;
  t.cand_meta = at<GroupMeta>(ws, p.o_metas) + s.meta_cand; t.n_cand_groups = s.ncg;
  t.nsg = p.nsg;
  t.fix_scale = at<float>(ws, p.o_fix); t.candA = at<float>(ws, p.o_candA); t.candB = at<float>(ws, p.o_candB);
  return t;
}

int tables_for(const LinPlan& p, void* ws, const Step& s, int kind, int target, cudaStream_t st) {
  return p4v_step_tables(tables_args(p, ws, s, kind, target), st);
}

// One search step: a W step (column block idx) or an X step (activation chunk idx).
struct StepRef { bool is_w; int idx; };

const Step& step_of(const LinPlan& p, StepRef r) { return r.is_w ? p.wsteps[r.idx] : p.xsteps[r.idx]; }

// Best candidate per row block (W step) / for the chunk (X step) from the score sums: the new step sizes.  The caller
// sets how the score keys map to the groups (n_keys, keys_per_group) and what else the select does (d_prev, has_next).
SelectArgs select_args(const LinPlan& p, void* ws, StepRef cur, float* score_log) {
  SelectArgs f{};
  f.sums = at<double>(ws, p.o_scores); f.n_cand = p.d.eq_n; f.n_groups = cur.is_w ? p.d.n_V : 1;
  f.inv_count = 1.0 / ((double)p.d.tokens * (double)(cur.is_w ? p.crb_rows : p.O));
  f.gscale = at<float>(ws, p.o_gscale); f.factors = at<float>(ws, p.o_factors);
  if (cur.is_w) { f.d0 = at<float>(ws, p.o_dW0); f.d = at<float>(ws, p.o_dW); f.d_stride = p.d.n_H; f.d_col = cur.idx; }
  else          { f.d0 = at<float>(ws, p.o_dX0); f.d = at<float>(ws, p.o_dX); f.d_stride = 0; f.d_col = cur.idx; }
  f.best = at<int>(ws, p.o_best); f.score_log = score_log;
  return f;
}

// Copy the chosen candidate's slabs of the step into the current operand image.
CommitArgs commit_args(const LinPlan& p, void* ws, StepRef cur) {
  const bool is_w = cur.is_w;
  const Step& s = step_of(p, cur);
  CommitArgs c{};
  c.best = at<int>(ws, p.o_best); c.n_groups = is_w ? p.d.n_V : 1;
  c.cand = at<uint8_t>(ws, is_w ? p.o_Wcand : p.o_Xcand);
  c.cand_tile_bytes = (unsigned long long)P4V_TILE * (is_w ? p.KB_W : p.KB_Xc);
  c.cand_plane_stride = c.cand_tile_bytes * (is_w ? p.tiles_o : p.tiles_m);
  c.cur = at<uint8_t>(ws, is_w ? p.o_Wcur : p.o_Xcur);
  c.cur_tile_bytes = (unsigned long long)P4V_TILE * (is_w ? p.KB_W : p.KB_X);
  c.P = 1; c.tiles = is_w ? p.tiles_o : p.tiles_m;
  c.rows_per_group = is_w ? p.crb_rows : 0; c.problem_groups = 0;
  c.segs = at<CommitSeg>(ws, p.o_commits) + s.commit_off; c.nseg = s.ncommit; c.commit_chunks = s.commit_chunks;
  return c;
}

// One search step: [scale tables] -> sweep -> reduce -> select (+ tables of the next step) -> commit.
int search_step(const LinPlan& p, void* ws, StepRef cur, const StepRef* next, bool tables_ready, const float* bias,
                const float* y, const float* g, float* score_log, cudaStream_t st) {
  const bool is_w = cur.is_w;
  const Step& s = step_of(p, cur);
  int rc;
  if (!tables_ready && (rc = tables_for(p, ws, s, is_w ? 0 : 1, cur.idx, st))) return rc;
  SweepParams sp; fill_sweep(p, ws, s, sp);
  sp.Y = y; sp.Gr = g; sp.bias = p.d.has_bias ? bias : nullptr;
  sp.order = is_w ? 0 : 1;
  if ((rc = run_sweep(p, s, sp, st))) return rc;
  ReduceArgs r{};
  r.partial = sp.partial; r.n_cand = p.d.eq_n; r.P = 1; r.tiles_m = p.tiles_m; r.tiles_n = p.tiles_o; r.order = sp.order;
  r.mode = P4V_SG_COLUMN; r.n_keys = p.nsg; r.sums = at<double>(ws, p.o_scores);
  if ((rc = p4v_reduce_scores(r, st))) return rc;
  SelectArgs f = select_args(p, ws, cur, score_log);
  f.n_keys = p.nsg;
  f.keys_per_group = (is_w && p.d.n_V > 1) ? p.crb_rows / P4V_CG : p.nsg;
  f.has_next = next != nullptr;
  if (next) f.next = tables_args(p, ws, step_of(p, *next), next->is_w ? 0 : 1, next->idx);
  if ((rc = p4v_select_step(f, st))) return rc;
  return p4v_commit_step(commit_args(p, ws, cur), st);
}

// The search steps of seq in order.  The scale tables of seq[0] are built first; those of every later step come with
// the select of the step before it.  The score log gets one [eq_n][groups] table per step.
int run_steps(const LinPlan& p, void* ws, const std::vector<StepRef>& seq, const float* bias, const float* y, const float* g,
              float* score_log, cudaStream_t st) {
  for (size_t i = 0; i < seq.size(); ++i) {
    int rc = search_step(p, ws, seq[i], i + 1 < seq.size() ? &seq[i + 1] : nullptr, i > 0, bias, y, g, score_log, st);
    if (rc) return rc;
    if (score_log) score_log += seq[i].is_w ? (size_t)p.d.eq_n * p.d.n_V : (size_t)p.d.eq_n;
  }
  return 0;
}

void add_steps(std::vector<StepRef>& seq, bool is_w, int begin, int end) {
  for (int i = begin; i < end; ++i) seq.push_back(StepRef{is_w, i});
}

// Whole W search of one round in normal-equation form (gram.cu): residual once, then per column block
// (pair image + Gram GEMM for every column block, once) and per column block update pass -> candidate evaluation -> select -> commit.
int gram_wsearch(const LinPlan& p, void* ws, const float* x, const float* W, const float* bias, const float* y, const float* g,
                 int h_begin, int h_end, float* score_log, cudaStream_t st) {
  int rc;
  const float w_lo = (float)-p.w_qmax, w_hi = (float)(p.w_qmax - 1);
  // e = y - yhat(current step sizes), exact integer products (every segment as a fixed group)
  if ((rc = tables_for(p, ws, p.fwd, -1, 0, st))) return rc;
  {
    SweepParams sp; fill_sweep(p, ws, p.fwd, sp);
    sp.Y = y; sp.Gr = g; sp.bias = p.d.has_bias ? bias : nullptr;
    sp.out = at<float>(ws, p.o_E); sp.out_residual = 1; sp.n_cand = 1; sp.order = 0; sp.R_cand = nullptr; sp.C_cand = nullptr;
    if ((rc = run_sweep(p, p.fwd, sp, st))) return rc;
  }
  if ((rc = p4v_xq_transpose(x, p.M, p.K, p.g_Mp, at<float>(ws, p.o_dX), p.crb_acts, (float)-p.a_qmax, (float)(p.a_qmax - 1),
                             at<int8_t>(ws, p.o_XqT), st))) return rc;
  // H for every column block of the range: one pair image + one tensor-core GEMM (the activations do not change
  // during the weight steps of a round)
  {
    const int nblk = h_end - h_begin;
    const unsigned long long z_tile = (unsigned long long)GRAM_PT * 2 * p.g_term_bytes;
    const int tiles_p = p4v_cdiv(p.g_npairs * nblk, GRAM_PT);
    if ((rc = p4v_pair_image(at<int8_t>(ws, p.o_XqT), p.g_Mp, p.M, h_begin * p.g_ks, p.g_ks, p.g_npairs, nblk, tiles_p, z_tile,
                             p.g_term_bytes, at<uint8_t>(ws, p.o_Z), st))) return rc;
    GramGemmArgs gg{};
    gg.R = at<uint8_t>(ws, p.o_G2T); gg.R_tile_bytes = (unsigned long long)P4V_TILE * 2 * p.g_term_bytes;
    gg.C = at<uint8_t>(ws, p.o_Z); gg.C_tile_bytes = z_tile; gg.term_bytes = p.g_term_bytes;
    gg.tiles_o = p.tiles_o; gg.tiles_p = tiles_p; gg.O = p.O; gg.H = at<float>(ws, p.o_H); gg.ldH = p.g_ldH;
    if ((rc = p4v_gram_gemm(gg, st))) return rc;
  }
  for (int h = h_begin; h < h_end; ++h) {
    GramUpdateArgs u{};
    u.E = at<float>(ws, p.o_E); u.G = g; u.gscale = at<float>(ws, p.o_gscale);
    u.W = W; u.M = p.M; u.O = p.O; u.K = p.K; u.XqT = at<int8_t>(ws, p.o_XqT); u.Mp = p.g_Mp;
    u.dX = at<float>(ws, p.o_dX); u.crb_acts = p.crb_acts;
    u.dW = at<float>(ws, p.o_dW); u.dW_prev = at<float>(ws, p.o_dprev); u.n_V = p.d.n_V; u.n_H = p.d.n_H; u.crb_rows = p.crb_rows;
    u.h_prev = h > h_begin ? h - 1 : -1; u.k_prev = (h - 1) * p.g_ks; u.k_next = h * p.g_ks; u.ks = p.g_ks;
    u.w_lo = w_lo; u.w_hi = w_hi; u.Upart = at<float>(ws, p.o_Upart); u.E2part = at<float>(ws, p.o_E2part);
    u.D = at<float>(ws, p.o_D); u.n_split = p.g_nmblk;
    if ((rc = p4v_gram_update(u, st))) return rc;
    GramEvalArgs ev{};
    ev.H = at<float>(ws, p.o_H) + (size_t)(h - h_begin) * p.g_npairs; ev.ldH = p.g_ldH; ev.npairs = p.g_npairs;
    if ((rc = p4v_gram_reduce(u.Upart, u.E2part, p.g_nmblk, p.O, p.g_ks, at<float>(ws, p.o_U), at<float>(ws, p.o_E2), st))) return rc;
    ev.U = at<float>(ws, p.o_U); ev.E2 = at<float>(ws, p.o_E2);
    ev.W = W; ev.O = p.O; ev.K = p.K; ev.k_first = h * p.g_ks; ev.ks = p.g_ks;
    ev.dW = at<float>(ws, p.o_dW); ev.dW0 = at<float>(ws, p.o_dW0); ev.n_H = p.d.n_H; ev.h = h;
    ev.dX = at<float>(ws, p.o_dX); ev.crb_acts = p.crb_acts;
    ev.factors = at<float>(ws, p.o_factors); ev.n_cand = p.d.eq_n;
    ev.n_groups = p.d.n_V; ev.rows_per_group = p.crb_rows; ev.osplit = p.g_osplit; ev.rows_per_block = p.g_opb;
    ev.w_lo = w_lo; ev.w_hi = w_hi;
    ev.sums = at<double>(ws, p.o_scores) + (size_t)p.d.eq_n * p.d.n_V; ev.n_keys = p.d.n_V * p.g_osplit;
    ev.sums2 = at<double>(ws, p.o_scores);
    if ((rc = p4v_gram_eval(ev, st))) return rc;
    SelectArgs f = select_args(p, ws, StepRef{true, h}, score_log);   // ev.sums2: one key per row block
    f.n_keys = p.d.n_V; f.keys_per_group = 1; f.d_prev = at<float>(ws, p.o_dprev);
    if ((rc = p4v_select_step(f, st))) return rc;
    if ((rc = p4v_commit_step(commit_args(p, ws, StepRef{true, h}), st))) return rc;
    if (score_log) score_log += (size_t)p.d.eq_n * p.d.n_V;
  }
  return 0;
}

int begin_impl(const LinPlan& p, const float* x, const float* W, const float* g, void* ws, cudaStream_t st) {
  int rc;
  if ((rc = upload_tables(p, ws, st))) return rc;
  int* keys = at<int>(ws, p.o_keys);
  const int nW = p.d.n_V * p.d.n_H;
  if ((rc = p4v_keys_reset(keys, nW + p.d.n_a + 1, st))) return rc;
  if ((rc = p4v_block_max(W, p.K, p.O, p.crb_rows, p.d.n_V, p.crb_cols, p.d.n_H, 1, keys, st))) return rc;
  if ((rc = p4v_block_max(x, p.K, p.M, p.M, 1, p.crb_acts, p.d.n_a, p.twin ? 0 : 1, keys + nW, st))) return rc;
  if ((rc = p4v_block_max(g, p.O, p.M, p.M, 1, p.O, 1, 1, keys + nW + p.d.n_a, st))) return rc;
  if (p.d.init_layerwise) {       // linear.py:382-383, :393-394: one step size for the whole weight / activation tensor
    if ((rc = p4v_keys_broadcast_max(keys, nW, st))) return rc;
    if ((rc = p4v_keys_broadcast_max(keys + nW, p.d.n_a, st))) return rc;
  }
  if ((rc = p4v_keys_to_delta(keys, nW, (float)p.w_qmax - 0.5f, at<float>(ws, p.o_dW0), at<float>(ws, p.o_dW), st))) return rc;
  if ((rc = p4v_keys_to_delta(keys + nW, p.d.n_a, (float)p.a_qmax - 0.5f, at<float>(ws, p.o_dX0), at<float>(ws, p.o_dX), st))) return rc;
  if ((rc = p4v_make_gscale(keys + nW + p.d.n_a, at<float>(ws, p.o_gscale), st))) return rc;
  if (p.gram) {          // (gs*g)^2 as two exact bf16 terms, transposed: rows = output channels, K = tokens
    QuantImageArgs q{};
    q.src = g; q.ld = p.O; q.prob_stride = 0; q.src_transposed = 1;
    q.P = 1; q.rows = p.O; q.tiles = p.tiles_o;
    q.dst = at<uint8_t>(ws, p.o_G2T); q.tile_bytes = (unsigned long long)P4V_TILE * 2 * p.g_term_bytes; q.plane_stride = 0;
    q.n_planes = 1; q.factors = nullptr; q.delta = at<float>(ws, p.o_dW0); q.rows_per_block = p.O + P4V_TILE; q.d_stride = 0; q.d_mod = 1;
    q.segs = at<P4VSeg>(ws, p.o_segsG); q.nseg = 2; q.is_int8 = 0; q.presc = at<float>(ws, p.o_gscale);
    if ((rc = p4v_quant_image(q, st))) return rc;
  }
  if ((rc = quant_W(p, ws, W, at<float>(ws, p.o_dW0), false, st))) return rc;
  if ((rc = quant_W(p, ws, W, at<float>(ws, p.o_dW0), true, st))) return rc;
  if ((rc = quant_X(p, ws, x, at<float>(ws, p.o_dX0), false, st))) return rc;
  if ((rc = quant_X(p, ws, x, at<float>(ws, p.o_dX0), true, st))) return rc;
  return 0;
}

}  // namespace

extern "C" int p4v_linear_workspace_bytes(const p4v_linear_desc* d, size_t* bytes) {
  return plan_workspace_bytes(build_plan, d, bytes, true);
}

extern "C" int p4v_linear_score_log_floats(const p4v_linear_desc* d, size_t* n) {
  P4V_REQUIRE(d && n, "null argument");
  *n = (size_t)d->search_round * ((size_t)d->n_H * d->eq_n * d->n_V + (size_t)d->n_a * d->eq_n);
  return 0;
}

extern "C" int p4v_linear_begin(const p4v_linear_desc* d, const float* x, const float* weight, const float* bias,
                                const float* raw_out, const float* raw_grad, void* workspace, size_t workspace_bytes, void* stream) {
  (void)bias; (void)raw_out;
  LinPlan p; int rc = build_plan(d, p, true);
  if (rc) return rc;
  P4V_REQUIRE(x && weight && raw_grad && workspace, "linear_begin: null pointer");
  P4V_REQUIRE(workspace_bytes >= p.total, "linear_begin: workspace too small (%zu < %zu)", workspace_bytes, p.total);
  return begin_impl(p, x, weight, raw_grad, workspace, (cudaStream_t)stream);
}

extern "C" int p4v_linear_search_w(const p4v_linear_desc* d, const float* bias, const float* raw_out, const float* raw_grad,
                                   void* workspace, int32_t h_begin, int32_t h_end, float* score_log, void* stream) {
  LinPlan p; int rc = build_plan(d, p, true);
  if (rc) return rc;
  P4V_REQUIRE(raw_out && raw_grad && workspace, "linear_search_w: null pointer");
  P4V_REQUIRE(0 <= h_begin && h_begin <= h_end && h_end <= d->n_H, "linear_search_w: bad block range");
  std::vector<StepRef> seq;
  add_steps(seq, true, h_begin, h_end);
  return run_steps(p, workspace, seq, bias, raw_out, raw_grad, score_log, (cudaStream_t)stream);
}

extern "C" int p4v_linear_search_a(const p4v_linear_desc* d, const float* bias, const float* raw_out, const float* raw_grad,
                                   void* workspace, int32_t a_begin, int32_t a_end, float* score_log, void* stream) {
  LinPlan p; int rc = build_plan(d, p, true);
  if (rc) return rc;
  P4V_REQUIRE(raw_out && raw_grad && workspace, "linear_search_a: null pointer");
  P4V_REQUIRE(0 <= a_begin && a_begin <= a_end && a_end <= d->n_a, "linear_search_a: bad chunk range");
  std::vector<StepRef> seq;
  add_steps(seq, false, a_begin, a_end);
  return run_steps(p, workspace, seq, bias, raw_out, raw_grad, score_log, (cudaStream_t)stream);
}

extern "C" int p4v_linear_intervals(const p4v_linear_desc* d, void* workspace, float* w_interval, float* a_interval, void* stream) {
  LinPlan p; int rc = build_plan(d, p, true);
  if (rc) return rc;
  P4V_REQUIRE(workspace && w_interval && a_interval, "linear_intervals: null pointer");
  P4V_CUDA_OK(cudaMemcpyAsync(w_interval, at<float>(workspace, p.o_dW), (size_t)d->n_V * d->n_H * 4, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  P4V_CUDA_OK(cudaMemcpyAsync(a_interval, at<float>(workspace, p.o_dX), (size_t)d->n_a * 4, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return 0;
}

extern "C" int p4v_linear_calibrate(const p4v_linear_desc* d, const float* x, const float* weight, const float* bias,
                                    const float* raw_out, const float* raw_grad, void* workspace, size_t workspace_bytes,
                                    float* w_interval, float* a_interval, float* score_log, void* stream) {
  LinPlan p; int rc = build_plan(d, p, true);
  if (rc) return rc;
  P4V_REQUIRE(x && weight && raw_out && raw_grad && workspace && w_interval && a_interval, "linear_calibrate: null pointer");
  P4V_REQUIRE(!d->has_bias || bias, "linear_calibrate: has_bias set but bias is null");
  P4V_REQUIRE(workspace_bytes >= p.total, "linear_calibrate: workspace too small (%zu < %zu)", workspace_bytes, p.total);
  cudaStream_t st = (cudaStream_t)stream;
  if ((rc = begin_impl(p, x, weight, raw_grad, workspace, st))) return rc;
  if (p.gram) {
    std::vector<StepRef> xseq;
    add_steps(xseq, false, 0, d->n_a);
    for (int e = 0; e < d->search_round; ++e) {
      if ((rc = gram_wsearch(p, workspace, x, weight, bias, raw_out, raw_grad, 0, d->n_H, score_log, st))) return rc;
      if (score_log) score_log += (size_t)d->n_H * d->eq_n * d->n_V;
      if ((rc = run_steps(p, workspace, xseq, bias, raw_out, raw_grad, score_log, st))) return rc;
      if (score_log) score_log += (size_t)d->n_a * d->eq_n;
    }
  } else {   // one sequence over all rounds: every select prepares the next step's tables, across W/X boundaries too
    std::vector<StepRef> seq;
    for (int e = 0; e < d->search_round; ++e) {
      add_steps(seq, true, 0, d->n_H);
      add_steps(seq, false, 0, d->n_a);
    }
    if ((rc = run_steps(p, workspace, seq, bias, raw_out, raw_grad, score_log, st))) return rc;
  }
  P4V_CUDA_OK(cudaMemcpyAsync(w_interval, at<float>(workspace, p.o_dW), (size_t)d->n_V * d->n_H * 4, cudaMemcpyDeviceToDevice, st));
  P4V_CUDA_OK(cudaMemcpyAsync(a_interval, at<float>(workspace, p.o_dX), (size_t)d->n_a * 4, cudaMemcpyDeviceToDevice, st));
  return 0;
}

extern "C" int p4v_linear_quant_forward_workspace_bytes(const p4v_linear_desc* d, size_t* bytes) {
  return plan_workspace_bytes(build_plan, d, bytes, false);
}

extern "C" int p4v_linear_quant_forward(const p4v_linear_desc* d, const float* x, const float* weight, const float* bias,
                                        const float* w_interval, const float* a_interval, void* workspace,
                                        size_t workspace_bytes, float* out, void* stream) {
  LinPlan p; int rc = build_plan(d, p, false);
  if (rc) return rc;
  P4V_REQUIRE(x && weight && w_interval && a_interval && workspace && out, "linear_quant_forward: null pointer");
  P4V_REQUIRE(workspace_bytes >= p.total, "linear_quant_forward: workspace too small (%zu < %zu)", workspace_bytes, p.total);
  cudaStream_t st = (cudaStream_t)stream;
  if ((rc = upload_tables(p, workspace, st))) return rc;
  P4V_CUDA_OK(cudaMemcpyAsync(at<float>(workspace, p.o_dW), w_interval, (size_t)d->n_V * d->n_H * 4, cudaMemcpyDeviceToDevice, st));
  P4V_CUDA_OK(cudaMemcpyAsync(at<float>(workspace, p.o_dX), a_interval, (size_t)d->n_a * 4, cudaMemcpyDeviceToDevice, st));
  if ((rc = quant_W(p, workspace, weight, at<float>(workspace, p.o_dW), false, st))) return rc;
  if ((rc = quant_X(p, workspace, x, at<float>(workspace, p.o_dX), false, st))) return rc;
  if ((rc = tables_for(p, workspace, p.fwd, -1, 0, st))) return rc;
  SweepParams sp; fill_sweep(p, workspace, p.fwd, sp);
  sp.bias = d->has_bias ? bias : nullptr;
  sp.out = out; sp.n_cand = 1; sp.order = 0;
  sp.R_cand = nullptr; sp.C_cand = nullptr;
  return run_sweep(p, p.fwd, sp, st);
}
