// Host-side planning pieces shared by the Linear, MatMul and conv searches: workspace carving, the candidate factor
// grid, the job splitter, the operand type choice and the table upload.  Host code only.
#pragma once
#include <algorithm>
#include <vector>

#include "../../include/ptq4vit_b200.h"
#include "common.cuh"

inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }
template <class T> T* at(void* ws, size_t off) { return reinterpret_cast<T*>(static_cast<uint8_t*>(ws) + off); }

// Consecutive workspace slices, each starting on a 256-byte boundary: take() returns a slice's offset, total is the
// workspace size so far.
struct Carver {
  size_t total = 0;
  size_t take(size_t bytes) { const size_t r = total; total = align_up(total + bytes, 256); return r; }
};

// The eq_n + 1 candidate factors alpha + i * (beta - alpha) / n: Python floats in the reference, rounded to fp32 when
// they become a tensor (linear.py:544-545).  The grid is compared bit for bit with the reference's: keep the
// expression and its order of operations.
inline std::vector<float> candidate_factors(double alpha, double beta, int n) {
  std::vector<float> f(n + 1);
  for (int i = 0; i <= n; ++i) f[i] = (float)(alpha + i * (beta - alpha) / n);
  return f;
}

// One K slab of an accumulator group as jobs of at most P4V_JOB_KB bytes (offsets: bytes in the padded rows of the
// two operand images).  first / last: the slab opens / closes the group's accumulation; a group may chain several
// slabs (the three terms of an exact bf16 split).  count is advanced by the number of jobs added.
inline void push_jobs(std::vector<P4VJob>& jobs, int r_off, int c_off, int kb, uint8_t flags, int group, bool first, bool last,
                      int& count) {
  for (int b = 0; b < kb; b += P4V_JOB_KB) {
    P4VJob j{};
    const int len = std::min(P4V_JOB_KB, kb - b);
    j.r_off = (uint32_t)(r_off + b) * P4V_TILE;
    j.c_off = (uint32_t)(c_off + b) * P4V_TILE;
    j.kb = (uint8_t)len;
    j.flags = flags | ((first && b == 0) ? P4V_JOB_FIRST : 0) | ((last && b + len >= kb) ? P4V_JOB_LAST : 0);
    j.group = (uint8_t)group;
    jobs.push_back(j);
    ++count;
  }
}

// Candidate jobs jobs[first, first + count) whose row operand does not depend on the candidate: keep that operand
// resident in shared memory when it fits in 60 KB.  Left as they are if any of them reads a candidate row plane.
inline void mark_resident(std::vector<P4VJob>& jobs, int first, int count) {
  uint32_t total = 0;
  for (int j = 0; j < count; ++j) total += (uint32_t)jobs[first + j].kb * P4V_TILE;
  if (total == 0 || total > 60 * 1024) return;
  uint32_t off = 0;
  for (int j = 0; j < count; ++j) {
    P4VJob& jb = jobs[first + j];
    if (jb.flags & P4V_JOB_RCAND) return;
    jb.flags |= P4V_JOB_RRES; jb.res_off = off; off += (uint32_t)jb.kb * P4V_TILE;
  }
}

// Operand images in int8 or integer-valued bf16 (desc.operand; automatic: int8 unless the shortest K slab is under 64
// elements -- short slabs are epilogue bound, and bf16 saves the int->float converts there, measured).
inline bool use_int8(int operand, int shortest_slab) {
  if (operand == P4V_OPERAND_INT8) return true;
  if (operand == P4V_OPERAND_BF16) return false;
  return shortest_slab >= 64;
}

// Host table -> its workspace slice, enqueued on st.  An empty table uploads nothing.
template <class T> int upload(void* ws, size_t off, const std::vector<T>& v, cudaStream_t st) {
  if (!v.empty()) P4V_CUDA_OK(cudaMemcpyAsync(at<void>(ws, off), v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice, st));
  return 0;
}

// Body of the *_workspace_bytes entry points: the bytes of device workspace the plan of d carves.
template <class Plan, class Desc, class... Args>
int plan_workspace_bytes(int (*build_plan)(const Desc*, Plan&, Args...), const Desc* d, size_t* bytes, Args... args) {
  Plan p;
  int rc = build_plan(d, p, args...);
  if (rc) return rc;
  P4V_REQUIRE(bytes != nullptr, "null output");
  *bytes = p.total;
  return 0;
}
