// Pieces shared by the CUDA-core scoring kernels (score.cu) and the tcgen05 full-sort path
// (mma_topk.cu): the 64-bit top-k key, the warp-cooperative sorted-list insertion and the query
// transform q(head, relation) of the five scorers.  TransH and TransD have no scorer of their own:
// they score as TransE on rows projected by kge_transh_project / kge_transd_project.
#pragma once

#include "common.cuh"

namespace {

constexpr int KMAX = 128;  // largest k of the sorted-list epilogue (warp_insert); larger k take score.cu's buffers

__device__ __forceinline__ uint64_t make_key(float score, uint32_t id) {
  uint32_t b = __float_as_uint(score);
  b = (b & 0x80000000u) ? ~b : (b | 0x80000000u);  // order-preserving map of fp32 to uint32
  return ((uint64_t)b << 32) | (uint64_t)(0xFFFFFFFFu - id);  // larger key = better (score desc, id asc)
}
__device__ __forceinline__ float key_score(uint64_t key) {
  uint32_t b = (uint32_t)(key >> 32);
  b = (b & 0x80000000u) ? (b & 0x7FFFFFFFu) : ~b;
  return __uint_as_float(b);
}
__device__ __forceinline__ int64_t key_id(uint64_t key) { return (int64_t)(0xFFFFFFFFu - (uint32_t)key); }

// Insert `c` into the descending list (capacity k) cooperatively by one warp.  `len` is warp-uniform.
__device__ __forceinline__ void warp_insert(uint64_t* list, int& len, int k, uint64_t c, int lane) {
  if (len == k && c <= list[k - 1]) return;
  int pos = 0;
  for (int base = 0; base < len; base += 32) {
    const int i = base + lane;
    const bool gt = (i < len) && (list[i] > c);
    pos += __popc(__ballot_sync(0xffffffffu, gt));
  }
  const int newlen = len < k ? len + 1 : k;
  uint64_t moved[KMAX / 32];
#pragma unroll
  for (int q = 0; q < KMAX / 32; ++q) {
    const int i = q * 32 + lane;
    moved[q] = (i > pos && i < newlen) ? list[i - 1] : 0ull;
  }
  __syncwarp();
#pragma unroll
  for (int q = 0; q < KMAX / 32; ++q) {
    const int i = q * 32 + lane;
    if (i > pos && i < newlen) list[i] = moved[q];
  }
  if (lane == 0) list[pos] = c;
  len = newlen;
  __syncwarp();
}

__device__ __forceinline__ float fracf_signed(float x) { return x - truncf(x); }   // torch.frac

struct ScoreArgs {
  kge_model_t m;
  const int64_t* heads;
  const int64_t* rels;   // NULL: the user->item relation row
  const int64_t* tails;  // predict only
  int64_t n;
  int head_is_user;
  int rel_row;  // row used when rels == NULL
};


// q(head, relation) at column c of the embedding (both parts for the complex models):
//   TransE   q = h + r                     (transe.py:55-57)
//   DistMult q = h * r                     (distmult.py:50-51)
//   RotatE   q = rot(h, theta) = (re | im) (rotate.py:61-66)
//   ComplEx  q = (hr*rr | hi*rr + hr*ri - hi*ri)   (complex.py:53-62 regrouped by tail part)
//   TorusE   q = frac(h) + frac(r)         (toruse.py:66-76; torch.frac keeps the sign: x - trunc(x))
__device__ __forceinline__ void query_value(const ScoreArgs& a, int64_t qrow, int c, float& q0, float& q1) {
  const int d = a.m.d;
  const int model = a.m.model;
  const kge_table_t& HT = a.head_is_user ? a.m.user : a.m.entity;
  const int64_t h_id = __ldg(a.heads + qrow);
  const int64_t r_id = a.rels ? __ldg(a.rels + qrow) : (int64_t)a.rel_row;
  const float h0 = __ldg(HT.w[0] + h_id * d + c);
  const float r0 = __ldg(a.m.relation.w[0] + r_id * d + c);
  q1 = 0.f;
  if (model == KGE_TRANSE) {
    q0 = h0 + r0;
  } else if (model == KGE_TORUSE) {
    q0 = fracf_signed(h0) + fracf_signed(r0);
  } else if (model == KGE_DISTMULT) {
    q0 = h0 * r0;
  } else if (model == KGE_ROTATE) {
    const float h1 = __ldg(HT.w[1] + h_id * d + c);
    float sn, cs;
    sincosf(r0, &sn, &cs);
    q0 = cs * h0 - sn * h1;
    q1 = cs * h1 + sn * h0;
  } else {
    const float h1 = __ldg(HT.w[1] + h_id * d + c);
    const float r1 = __ldg(a.m.relation.w[1] + r_id * d + c);
    q0 = h0 * r0;
    q1 = h1 * r0 + h0 * r1 - h1 * r1;
  }
}

// How a (query, target) pair of rows is contracted -- 0 dot product, 1 squared distance (score = margin - sqrt),
// 2 torus distance sum(min(x^2, 1 - x^2)) on frac()ed rows (score = -4 * sum).  Zero padding contributes 0 in all three.
constexpr int MODE_DOT = 0, MODE_DIST = 1, MODE_TORUS = 2;

// The sequential fp32 chain of score.cu's tile kernel over one part of one (query, target) pair: columns ascending,
// one accumulation per column, continuing from `acc`.  `qp` = the part's d query values, `t` = the target's row of
// that part (raw: the torus frac() is applied here as the tile kernel applies it when it stages targets).  Scores
// built on it are bit-identical to the tile kernel's.  The loads of a 64-column block are all issued before the chain
// consumes them.
template <int MODE>
__device__ __forceinline__ float exact_chain(const float* qp, const float* __restrict__ t, int d, float acc) {
  if ((d & 3) == 0) {
    for (int c0 = 0; c0 < d; c0 += 64) {
      float4 tv[16];
#pragma unroll
      for (int x = 0; x < 16; ++x)
        if (c0 + 4 * x < d) tv[x] = __ldg(reinterpret_cast<const float4*>(t + c0) + x);
#pragma unroll
      for (int x = 0; x < 16; ++x) {
        if (c0 + 4 * x < d) {
          const int c = c0 + 4 * x;
          const float4 qv = *reinterpret_cast<const float4*>(qp + c);
          float4 v = tv[x];
          if (MODE == MODE_TORUS) v = make_float4(fracf_signed(v.x), fracf_signed(v.y), fracf_signed(v.z), fracf_signed(v.w));
          if (MODE == MODE_TORUS) {
            const float e0 = qv.x - v.x, e1 = qv.y - v.y, e2 = qv.z - v.z, e3 = qv.w - v.w;
            const float s0 = e0 * e0, s1 = e1 * e1, s2 = e2 * e2, s3 = e3 * e3;
            acc += fminf(s0, 1.f - s0);
            acc += fminf(s1, 1.f - s1);
            acc += fminf(s2, 1.f - s2);
            acc += fminf(s3, 1.f - s3);
          } else if (MODE == MODE_DIST) {
            const float e0 = qv.x - v.x, e1 = qv.y - v.y, e2 = qv.z - v.z, e3 = qv.w - v.w;
            acc = fmaf(e0, e0, acc);
            acc = fmaf(e1, e1, acc);
            acc = fmaf(e2, e2, acc);
            acc = fmaf(e3, e3, acc);
          } else {
            acc = fmaf(qv.x, v.x, acc);
            acc = fmaf(qv.y, v.y, acc);
            acc = fmaf(qv.z, v.z, acc);
            acc = fmaf(qv.w, v.w, acc);
          }
        }
      }
    }
  } else {
#pragma unroll 8
    for (int c = 0; c < d; ++c) {
      float v = __ldg(t + c);
      if (MODE == MODE_TORUS) v = fracf_signed(v);
      const float e0 = qp[c] - v;
      if (MODE == MODE_TORUS) {
        const float s0 = e0 * e0;
        acc += fminf(s0, 1.f - s0);
      } else if (MODE == MODE_DIST) {
        acc = fmaf(e0, e0, acc);
      } else {
        acc = fmaf(qp[c], v, acc);
      }
    }
  }
  return acc;
}

}  // namespace
