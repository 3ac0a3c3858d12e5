// Fused KGE training step for sm_100a: gather -> score -> loss -> analytic gradient scatter,
// then exact row-lazy Adam on the touched rows.
//
// Replaces, per step (paths under /root/reference/hopwise/):
//   model/knowledge_graph_embedding_recommender/{transe.py:75-98, distmult.py:68-95,
//   rotate.py:98-131, complex.py:95-128}   (calculate_loss: 8-16 gathers, cat, scorer, loss)
//   trainer/trainer.py:261                  (loss.backward(): dense [rows, d] gradients)
//   trainer/trainer.py:264 + torch.optim.Adam (dense update of every table)
//
// Data layout in HBM: the tables stay exactly where torch keeps them (fp32 [rows, d], one
// matrix per re/im part), so state_dict() is zero-copy.  Next to every table live m, v (Adam
// moments), g (a gradient accumulator that is all-zero between steps: only touched rows are ever
// written and the update kernel zeroes them again) and row_state[rows] = {last_step, touch_step}
// (8 bytes per row).  Nothing of size [rows, d] is traversed per step.
//
// Kernel A (train_fwd_kernel): a group of G lanes owns one positive triple.  Ids of the whole
// triple are read first, then the 8-byte row states and the 128-bit row fragments of head,
// relation, positive and first negative tail are all issued before anything is consumed (one
// memory latency per triple; further negatives are prefetched one ahead).  Gradients leave as
// RED.ADD.F32x4; a touched row is marked by a plain store of the step number.  The user->item
// relation row is shared by every rec triple, so its gradient is accumulated in registers,
// reduced per CTA in shared memory and flushed once per CTA.  With two triples per warp, the KG
// relation rows go the same way, through per-warp copies in shared memory (WARP_RACC).
// Kernel B (adam_apply_kernel): lanes scan row_state (8 B per row, coalesced), ballot the rows
// marked in this step and a lane group updates each: replay the zero-gradient steps the row
// skipped (dense Adam keeps moving a row after its last gradient), apply the real step, zero g.
#include <math.h>
#include <stdarg.h>
#include <stdio.h>

#include <type_traits>

#include "common.cuh"

namespace {

struct AdamDev {
  float lr, b1, b2, eps, omb1, omb2;
  int step;  // update being produced
  int cap;
  int opt;   // enum kge_optimizer
  const float2* table;  // {lr/(1-b1^j), 1/sqrt(1-b2^j)}
  int tlen;
};
struct TrainArgs {
  kge_model_t m;
  kge_batch_t b;
  AdamDev adam;
  float w_rec, w_kg;        // weight of one (positive, negative) pair in the scalar loss
  float wpos_rec, wpos_kg;  // BCE models: weight of the positive term (= w * k)
  int with_grad;
  float* loss;
};

__device__ __forceinline__ float2 adam_consts(const AdamDev& A, int j) {
  if (j < A.tlen) return __ldg(A.table + j);
  return make_float2(A.lr, 1.f);
}

// Zero-gradient Adam steps s+1 .. t_end on one row fragment (torch.optim.Adam with g = 0:
// m.lerp_(0, 1-b1); v.mul_(b2); p.addcdiv_(m, sqrt(v)/sqrt(1-b2^j) + eps, -lr/(1-b1^j))).
// After `cap` steps m has decayed by b1^cap (7e-10 at cap 200) and the remaining movement is
// below fp32 resolution of the weights; m and v then decay in closed form.
template <int E>
__device__ __forceinline__ void adam_replay(float (&p)[E], float (&m)[E], float (&v)[E], int s, int t_end,
                                            const AdamDev& A) {
  const int n = t_end - s;
  if (n <= 0) return;
  const int nrep = n < A.cap ? n : A.cap;
  for (int j = s + 1; j <= s + nrep; ++j) {
    const float2 c = adam_consts(A, j);
#pragma unroll
    for (int e = 0; e < E; ++e) {
      m[e] -= A.omb1 * m[e];
      v[e] *= A.b2;
      const float den = sqrt_approx(v[e]) * c.y + A.eps;
      p[e] -= c.x * __fdividef(m[e], den);
    }
  }
  if (n > nrep) {
    const float f1 = powf(A.b1, (float)(n - nrep)), f2 = powf(A.b2, (float)(n - nrep));
#pragma unroll
    for (int e = 0; e < E; ++e) {
      m[e] *= f1;
      v[e] *= f2;
    }
  }
}

// {last_step, touch_step} of a row; tables without optimiser state read as never updated.
__device__ __forceinline__ int2 row_state(const kge_table_t& T, int64_t row) {
  if (!T.row_state) return make_int2(-1, -1);
  return *(reinterpret_cast<const int2*>(T.row_state) + row);
}

// Mark a row as touched in `step` (an idempotent plain store); skipped when the loaded state shows it.
__device__ __forceinline__ void touch_row(const kge_table_t& T, int64_t row, int seen_touch, int step, int gl) {
  // (tables without row states -- dense Adam on every element, owner-sharded over the switch -- keep no marks)
  if (gl != 0 || seen_touch == step || !T.row_state) return;
  T.row_state[2 * row + 1] = step;
}

// Bring a fragment that was loaded from w up to step-1 when the row lags behind (rare path).
// With `mark` (a training pass) the lagging row is also marked as touched, even if it will receive no gradient:
// the Adam kernel then brings it up to date with a zero-gradient step (exactly what dense Adam does to it), so
// the lag of a row that keeps being referenced by inactive triples stays bounded -- without this every forward
// pass would replay the same (growing, up to the cap) run of skipped steps for it again.
template <int VEC, int G, int NCH>
__device__ __forceinline__ void catch_up(const kge_table_t& T, int part, int64_t row, int2 st, int d, int gl,
                                         const AdamDev& A, float (&x)[VEC * NCH], int mark) {
  const int last = st.x;
  if (last >= 0 && last < A.step - 1 && A.opt == KGE_OPT_ADAM) {   // (only Adam moves a row that has no gradient)
    float m[VEC * NCH], v[VEC * NCH];
    frag_load<VEC, G, NCH>(T.m[part], row, d, gl, m);
    frag_load<VEC, G, NCH>(T.v[part], row, d, gl, v);
    adam_replay<VEC * NCH>(x, m, v, last, A.step - 1, A);
    if (mark && part == 0) touch_row(T, row, st.y, A.step, gl);   // (last >= 0: the table has states)
  }
}


__device__ __forceinline__ float softplusf(float z) { return fmaxf(z, 0.f) + log1pf(expf(-fabsf(z))); }
__device__ __forceinline__ float sigmoidf(float z) { return 1.f / (1.f + expf(-z)); }

template <int MODEL, int VEC, int G, int NCH>
struct FwdBounds {
  static constexpr int E = VEC * NCH;
  static constexpr int PH = (MODEL == KGE_ROTATE || MODEL == KGE_COMPLEX || MODEL == KGE_TRANSD) ? 2 : 1;
  // resident CTAs per SM the register budget is shaped for (more warps = more loads in flight)
  // (the two-triples-per-warp shape, G = 16 with two fragments per lane, wants its 8-element fragments of h, r, both
  // tails and three gradients in registers: measured 0.320 ms at two CTAs per SM vs 0.381 ms at three, cfg2)
  static constexpr int MIN_CTAS = (VEC == 4 && G == 16 && NCH == 2) ? 2
                                  : (E * PH <= 4) ? 4 : (E * PH <= 8 ? 3 : (E * PH <= 16 ? 2 : 1));
};

// Shared memory of the WARP_RACC path: every warp's private [R][PR][d] relation-gradient copy, then one flag per
// relation row that this CTA gave a gradient.
constexpr int kFwdWarps = 8;   // train_fwd_kernel runs 256 threads per CTA
inline size_t warp_racc_smem_bytes(int64_t rows, int parts, int d) {
  return (size_t)kFwdWarps * rows * parts * d * sizeof(float) + (size_t)rows * sizeof(int);
}

// WARP_RACC (two triples per warp only, G = 16): relation gradients of both halves are summed in per-warp copies in
// shared memory with plain loads and stores and leave once per CTA, one float4 RED per 4 columns of each touched
// row -- instead of one RED per triple onto the few lines of the ~20 KG relation rows, which every L2 slice holding
// them has to serialise.  (A CTA-wide copy would need float atomics on shared memory: a CAS loop on sm_100a.)
template <int MODEL, int VEC, int G, int NCH, bool WARP_RACC = false>
__global__ void __launch_bounds__(256, FwdBounds<MODEL, VEC, G, NCH>::MIN_CTAS) train_fwd_kernel(const TrainArgs a) {
  constexpr int E = VEC * NCH;
  constexpr int PH = (MODEL == KGE_ROTATE || MODEL == KGE_COMPLEX || MODEL == KGE_TRANSD) ? 2 : 1;  // head / tail parts
  constexpr int PR = (MODEL == KGE_COMPLEX || MODEL == KGE_TRANSH || MODEL == KGE_TRANSD) ? 2 : 1;   // relation parts
  static_assert(!WARP_RACC || (VEC == 4 && G == 16), "per-warp relation copies pair the two half-warp groups");
  // without WARP_RACC: [PR][d] user->item relation gradient of this CTA; with it: warp_racc_smem_bytes
  extern __shared__ __align__(16) float s_racc[];
  __shared__ float s_loss[8];

  const int d = a.m.d;
  const int gl = (threadIdx.x & 31) % G;
  const int groups_per_cta = blockDim.x / G;
  const int64_t n_groups = (int64_t)gridDim.x * groups_per_cta;
  const int step = a.adam.step;
  const float margin = a.m.margin;
  const kge_table_t& ET = a.m.entity;
  const kge_table_t& RT = a.m.relation;

  const int n_rel = (int)RT.rows;
  const int nv = d >> 2;
  // WARP_RACC: this warp's copy, as float4 [R][PR][nv]; the touched flags follow the copies of all warps
  float4* s_wrg = reinterpret_cast<float4*>(s_racc) + (size_t)(threadIdx.x >> 5) * n_rel * PR * nv;
  int* s_rtouch = reinterpret_cast<int*>(s_racc + (size_t)kFwdWarps * n_rel * PR * d);
  if constexpr (WARP_RACC) {
    float4* s4 = reinterpret_cast<float4*>(s_racc);
    for (int i = threadIdx.x; i < kFwdWarps * n_rel * PR * nv; i += blockDim.x) s4[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int i = threadIdx.x; i < n_rel; i += blockDim.x) s_rtouch[i] = 0;
  } else {
    for (int i = threadIdx.x; i < PR * d; i += blockDim.x) s_racc[i] = 0.f;
  }
  __syncthreads();
  // (adds a group's relation-gradient fragment into row `row` of its warp's copy)
  auto warp_copy_add = [&](int row, const float (&x)[PR][E]) {
#pragma unroll
    for (int p = 0; p < PR; ++p)
#pragma unroll
      for (int j = 0; j < NCH; ++j) {
        const int c = gl + j * G;
        if (c < nv) {
          float4& s = s_wrg[(row * PR + p) * nv + c];
          float4 v = s;
          v.x += x[p][4 * j]; v.y += x[p][4 * j + 1]; v.z += x[p][4 * j + 2]; v.w += x[p][4 * j + 3];
          s = v;
        }
      }
  };

  float lsum = 0.f;
  float racc[PR][E];
#pragma unroll
  for (int p = 0; p < PR; ++p)
#pragma unroll
    for (int e = 0; e < E; ++e) racc[p][e] = 0.f;
  bool rec_seen = false;

  // The recommendation half and the KG half run as two loops over one body: with the half known at compile
  // time the table / id-array selections fold away (they cost ~100 instructions per triple as run-time selects).
  auto run_half = [&](auto rec_tag) {
  constexpr bool is_rec = decltype(rec_tag)::value;
  const int64_t n_seg = is_rec ? a.b.n_rec : a.b.n_kg;
  const int64_t* negs = is_rec ? a.b.neg_item : a.b.neg_tail;
  for (int64_t i = (int64_t)blockIdx.x * groups_per_cta + threadIdx.x / G; i < n_seg; i += n_groups) {
    const int K = is_rec ? a.b.k_rec : a.b.k_kg;
    const kge_table_t& HT = is_rec ? a.m.user : a.m.entity;
    const float w = is_rec ? a.w_rec : a.w_kg;
    const float wpos = is_rec ? a.wpos_rec : a.wpos_kg;

    // ---- one memory latency: ids, then every row state and row fragment of the triple ---------------
    // (requesting the ids one iteration ahead changes nothing measurable: cfg2 0.3202 vs 0.3198 ms forward -- the
    // id vectors stream through L1/L2 -- and costs the one-triple-per-warp shapes ~100 B of spills)
    const int64_t h_id = is_rec ? __ldg(a.b.user + i) : __ldg(a.b.head + i);
    const int64_t r_id = is_rec ? (int64_t)a.m.ui_relation : __ldg(a.b.relation + i);
    const int64_t tp_id = is_rec ? __ldg(a.b.item + i) : __ldg(a.b.tail + i);
    int64_t tn_id = __ldg(negs + i);
    const int2 sh = row_state(HT, h_id), sr = row_state(RT, r_id), stp = row_state(ET, tp_id);
    int2 stn = row_state(ET, tn_id);
    float h[PH][E], r[PR][E], tp[PH][E], tnx[PH][E];
#pragma unroll
    for (int p = 0; p < PH; ++p) frag_load<VEC, G, NCH>(HT.w[p], h_id, d, gl, h[p]);
#pragma unroll
    for (int p = 0; p < PR; ++p) frag_load<VEC, G, NCH>(RT.w[p], r_id, d, gl, r[p]);
#pragma unroll
    for (int p = 0; p < PH; ++p) frag_load<VEC, G, NCH>(ET.w[p], tp_id, d, gl, tp[p]);
#pragma unroll
    for (int p = 0; p < PH; ++p) frag_load<VEC, G, NCH>(ET.w[p], tn_id, d, gl, tnx[p]);
#pragma unroll
    for (int p = 0; p < PH; ++p) catch_up<VEC, G, NCH>(HT, p, h_id, sh, d, gl, a.adam, h[p], a.with_grad);
#pragma unroll
    for (int p = 0; p < PR; ++p) catch_up<VEC, G, NCH>(RT, p, r_id, sr, d, gl, a.adam, r[p], a.with_grad);
#pragma unroll
    for (int p = 0; p < PH; ++p) catch_up<VEC, G, NCH>(ET, p, tp_id, stp, d, gl, a.adam, tp[p], a.with_grad);

    // gradient fragments of the anchor, relation and positive tail
    float gh[PH][E], gr[PR][E], gtp[PH][E];
#pragma unroll
    for (int p = 0; p < PH; ++p)
#pragma unroll
      for (int e = 0; e < E; ++e) { gh[p][e] = 0.f; gtp[p][e] = 0.f; }
#pragma unroll
    for (int p = 0; p < PR; ++p)
#pragma unroll
      for (int e = 0; e < E; ++e) gr[p][e] = 0.f;
    bool any_grad = false;
    float inst_loss = 0.f;

    // ---- model-specific precomputation on (h, r, positive tail) -------------------------------------
    // TransE:   c0 = x = h + r, c1 = w * unit(x - tp + eps), s_pos = ||x - tp + eps||  (transe.py:96)
    // DistMult: c0 = q = h * r, s_pos = q . tp                                         (distmult.py:90-93)
    // RotatE:   c0 = cos, c1 = sin of the phases, (c2, c3) = rot(h)                    (rotate.py:118-131)
    // ComplEx:  c0 = A = hr*rr, c1 = B = hi*rr + hr*ri - hi*ri                          (complex.py:115-128)
    float c0[E], c1[E], c2[E], c3[E];
    float acc0[E], acc1[E];  // per-triple accumulators over the tails
    float s_pos = 0.f;
#pragma unroll
    for (int e = 0; e < E; ++e) { c0[e] = c1[e] = c2[e] = c3[e] = 0.f; acc0[e] = acc1[e] = 0.f; }
    float nact = 0.f;
    float s_w = 0.f;   // TransH: sum of the hyperplane vector's components
    float s_h = 0.f, s_tp = 0.f;   // TransD: <h, h_p>, <tp, tp_p>
    if (MODEL == KGE_TRANSD) {
      // transd.py:86-91: proj(e) = e + r_p * <e, e_p> (parts: [0] embedding, [1] transfer vector).  Then TransE on the
      // projected rows: c0 = x = proj(h) + r, c1 = w * unit(x - proj(tp) + eps).  Products and dot products by explicit
      // fmas in one order, so that the projections of equal rows are equal bit for bit wherever they are formed.
      float a0 = 0.f, a1 = 0.f;
#pragma unroll
      for (int e = 0; e < E; ++e) {
        a0 = __fmaf_rn(h[0][e], h[PH - 1][e], a0);
        a1 = __fmaf_rn(tp[0][e], tp[PH - 1][e], a1);
      }
      s_h = group_sum<G>(a0);
      s_tp = group_sum<G>(a1);
      float sp = 0.f;
#pragma unroll
      for (int e = 0; e < E; ++e) {
        c0[e] = __fmaf_rn(r[PR - 1][e], s_h, h[0][e]) + r[0][e];
        const float tproj = __fmaf_rn(r[PR - 1][e], s_tp, tp[0][e]);
        const float dp = frag_valid<VEC, G, NCH>(d, gl, e) ? (__fsub_rn(c0[e], tproj) + 1e-6f) : 0.f;
        c1[e] = dp;
        sp = __fmaf_rn(dp, dp, sp);
      }
      s_pos = sqrtf(group_sum<G>(sp));
      const float inv_p = s_pos > 0.f ? 1.f / s_pos : 0.f;
#pragma unroll
      for (int e = 0; e < E; ++e) c1[e] = __fmul_rn(w, __fmul_rn(c1[e], inv_p));
    } else if (MODEL == KGE_TRANSH) {
      // transh.py:73-74: project(e) = e - (e * sum(w)) * w = e * (1 - sum(w) * w); c2 holds the factor.  Then TransE on
      // the projected rows: c0 = x = h*c2 + r, c1 = w * unit(x - tp*c2 + eps), s_pos = ||x - tp*c2 + eps||
      float sw = 0.f;
#pragma unroll
      for (int e = 0; e < E; ++e) sw += r[PR - 1][e];   // (padding lanes hold zeros)
      s_w = group_sum<G>(sw);
      float sp = 0.f;
#pragma unroll
      for (int e = 0; e < E; ++e) {
        // (explicit roundings: the compiler rematerialises this factor at its uses, and a product contracted into
        // the subtraction at one use only would give the positive and the negative tail different factors)
        c2[e] = __fsub_rn(1.f, __fmul_rn(s_w, r[PR - 1][e]));
        c0[e] = __fmaf_rn(h[0][e], c2[e], r[0][e]);
        // (projected tails as explicit products: the positive and the negative residual must be formed by identical
        // operations -- a product contracted into the subtraction on one side only leaves a 1-ulp residue where a
        // row is both the positive and the negative of a pair, and Adam turns 5e-10 of gradient into 4e-5 of weight)
        const float dp = frag_valid<VEC, G, NCH>(d, gl, e) ? (__fsub_rn(c0[e], __fmul_rn(tp[0][e], c2[e])) + 1e-6f) : 0.f;
        c1[e] = dp;
        sp = __fmaf_rn(dp, dp, sp);
      }
      s_pos = sqrtf(group_sum<G>(sp));
      const float inv_p = s_pos > 0.f ? 1.f / s_pos : 0.f;
#pragma unroll
      for (int e = 0; e < E; ++e) c1[e] = __fmul_rn(w, __fmul_rn(c1[e], inv_p));
    } else if (MODEL == KGE_TRANSE) {
      float sp = 0.f;
#pragma unroll
      for (int e = 0; e < E; ++e) {
        c0[e] = h[0][e] + r[0][e];
        const float dp = frag_valid<VEC, G, NCH>(d, gl, e) ? (c0[e] - tp[0][e] + 1e-6f) : 0.f;
        c1[e] = dp;
        sp = __fmaf_rn(dp, dp, sp);
      }
      s_pos = sqrtf(group_sum<G>(sp));
      const float inv_p = s_pos > 0.f ? 1.f / s_pos : 0.f;
      // positive and negative terms are formed by the same operations so that a pair whose
      // negative equals its positive cancels exactly, as it does under autograd (explicit _rn
      // intrinsics: the compiler must not contract one side's product into the subtraction)
#pragma unroll
      for (int e = 0; e < E; ++e) c1[e] = __fmul_rn(w, __fmul_rn(c1[e], inv_p));
    } else if (MODEL == KGE_DISTMULT) {
      float sp = 0.f;
#pragma unroll
      for (int e = 0; e < E; ++e) {
        c0[e] = h[0][e] * r[0][e];
        sp += c0[e] * tp[0][e];
      }
      s_pos = group_sum<G>(sp);
    } else if (MODEL == KGE_ROTATE) {
#pragma unroll
      for (int e = 0; e < E; ++e) {
        sincosf(r[0][e], &c1[e], &c0[e]);
        c2[e] = c0[e] * h[0][e] - c1[e] * h[PH - 1][e];
        c3[e] = c0[e] * h[PH - 1][e] + c1[e] * h[0][e];
      }
    } else {
#pragma unroll
      for (int e = 0; e < E; ++e) {
        c0[e] = h[0][e] * r[0][e];
        c1[e] = h[PH - 1][e] * r[0][e] + h[0][e] * r[PR - 1][e] - h[PH - 1][e] * r[PR - 1][e];
      }
    }

    // ---- tails: j = -1 is the positive (BCE models only), then K negatives, prefetched one ahead ------
    const int j0 = (MODEL == KGE_ROTATE || MODEL == KGE_COMPLEX) ? -1 : 0;
    for (int j = j0; j < K; ++j) {
      const bool pos = j < 0;
      float t[PH][E];
      int64_t t_id;
      int2 st;
      if (pos) {
        t_id = tp_id;
        st = stp;
#pragma unroll
        for (int p = 0; p < PH; ++p)
#pragma unroll
          for (int e = 0; e < E; ++e) t[p][e] = tp[p][e];
      } else {
        t_id = tn_id;
        st = stn;
#pragma unroll
        for (int p = 0; p < PH; ++p)
#pragma unroll
          for (int e = 0; e < E; ++e) t[p][e] = tnx[p][e];
        if (j + 1 < K) {  // prefetch the next negative while this one is consumed
          tn_id = __ldg(negs + (int64_t)(j + 1) * n_seg + i);
          stn = row_state(ET, tn_id);
#pragma unroll
          for (int p = 0; p < PH; ++p) frag_load<VEC, G, NCH>(ET.w[p], tn_id, d, gl, tnx[p]);
        }
#pragma unroll
        for (int p = 0; p < PH; ++p) catch_up<VEC, G, NCH>(ET, p, t_id, st, d, gl, a.adam, t[p], a.with_grad);
      }

      if (MODEL == KGE_TRANSD) {
        float a0 = 0.f;
#pragma unroll
        for (int e = 0; e < E; ++e) a0 = __fmaf_rn(t[0][e], t[PH - 1][e], a0);
        const float s_tn = group_sum<G>(a0);
        float dnv[E];
        float sn = 0.f;
#pragma unroll
        for (int e = 0; e < E; ++e) {
          const float tproj = __fmaf_rn(r[PR - 1][e], s_tn, t[0][e]);
          dnv[e] = frag_valid<VEC, G, NCH>(d, gl, e) ? (__fsub_rn(c0[e], tproj) + 1e-6f) : 0.f;
          sn = __fmaf_rn(dnv[e], dnv[e], sn);
        }
        const float nn_ = sqrtf(group_sum<G>(sn));
        const float z = margin + s_pos - nn_;
        if (z >= 0.f) {
          inst_loss += z * w;
          if (a.with_grad) {
            const float inv_n = nn_ > 0.f ? 1.f / nn_ : 0.f;
            nact += 1.f;
            float dotn = 0.f;
#pragma unroll
            for (int e = 0; e < E; ++e) {
              dnv[e] = __fmul_rn(w, __fmul_rn(dnv[e], inv_n));   // gradient of the PROJECTED negative tail
              gh[0][e] += __fsub_rn(c1[e], dnv[e]);              // ... of x = proj(h) + r
              gtp[0][e] -= c1[e];                                // ... of the projected positive tail
              acc1[e] = __fmaf_rn(dnv[e], s_tn, acc1[e]);        // ... of r_p, this tail's share
              dotn = __fmaf_rn(dnv[e], r[PR - 1][e], dotn);
            }
            dotn = group_sum<G>(dotn);
            float gv[E];
#pragma unroll
            for (int e = 0; e < E; ++e) {   // back through proj(t) = t + r_p * <t, t_p>
              gv[e] = t[0][e] * dotn;
              dnv[e] = __fmaf_rn(t[PH - 1][e], dotn, dnv[e]);
            }
            frag_atomic_add<VEC, G, NCH>(ET.g[0], t_id, d, gl, dnv);
            frag_atomic_add<VEC, G, NCH>(ET.g[PH - 1], t_id, d, gl, gv);
            touch_row(ET, t_id, st.y, step, gl);
          }
        }
      } else if (MODEL == KGE_TRANSH) {
        float dnv[E];
        float sn = 0.f;
#pragma unroll
        for (int e = 0; e < E; ++e) {
          dnv[e] = frag_valid<VEC, G, NCH>(d, gl, e) ? (__fsub_rn(c0[e], __fmul_rn(t[0][e], c2[e])) + 1e-6f) : 0.f;
          sn = __fmaf_rn(dnv[e], dnv[e], sn);
        }
        const float nn_ = sqrtf(group_sum<G>(sn));
        const float z = margin + s_pos - nn_;
        if (z >= 0.f) {
          inst_loss += z * w;
          if (a.with_grad) {
            const float inv_n = nn_ > 0.f ? 1.f / nn_ : 0.f;
            nact += 1.f;
#pragma unroll
            for (int e = 0; e < E; ++e) {
              const float gneg = __fmul_rn(w, __fmul_rn(dnv[e], inv_n));   // gradient of the PROJECTED negative tail
              gh[0][e] += __fsub_rn(c1[e], gneg);                          // ... of x = proj(h) + r
              gtp[0][e] -= c1[e];                                          // ... of the projected positive tail
              acc0[e] = __fmaf_rn(gneg, t[0][e], acc0[e]);                 // ... of the factor c2, this tail's share
              t[0][e] = gneg * c2[e];                                      // back through the projection
            }
            frag_atomic_add<VEC, G, NCH>(ET.g[0], t_id, d, gl, t[0]);
            touch_row(ET, t_id, st.y, step, gl);
          }
        }
      } else if (MODEL == KGE_TRANSE) {
        float sn = 0.f;
#pragma unroll
        for (int e = 0; e < E; ++e) {
          const float dn = frag_valid<VEC, G, NCH>(d, gl, e) ? (c0[e] - t[0][e] + 1e-6f) : 0.f;
          t[0][e] = dn;
          sn = __fmaf_rn(dn, dn, sn);
        }
        const float nn_ = sqrtf(group_sum<G>(sn));
        const float z = margin + s_pos - nn_;
        if (z >= 0.f) {
          inst_loss += z * w;
          if (a.with_grad) {
            const float inv_n = nn_ > 0.f ? 1.f / nn_ : 0.f;
            nact += 1.f;
#pragma unroll
            for (int e = 0; e < E; ++e) {
              t[0][e] = __fmul_rn(w, __fmul_rn(t[0][e], inv_n));  // gradient of the negative tail
              gh[0][e] += __fsub_rn(c1[e], t[0][e]);
              gtp[0][e] -= c1[e];
            }
            frag_atomic_add<VEC, G, NCH>(ET.g[0], t_id, d, gl, t[0]);
            touch_row(ET, t_id, st.y, step, gl);
          }
        }
      } else if (MODEL == KGE_DISTMULT) {
        float sn = 0.f;
#pragma unroll
        for (int e = 0; e < E; ++e) sn += c0[e] * t[0][e];
        sn = group_sum<G>(sn);
        const float z = margin - s_pos + sn;
        if (z >= 0.f) {
          inst_loss += z * w;
          if (a.with_grad) {
            nact += 1.f;
            float gtn[E];
#pragma unroll
            for (int e = 0; e < E; ++e) {
              acc0[e] += w * (t[0][e] - tp[0][e]);
              gtn[e] = w * c0[e];
            }
            frag_atomic_add<VEC, G, NCH>(ET.g[0], t_id, d, gl, gtn);
            touch_row(ET, t_id, st.y, step, gl);
          }
        }
      } else if (MODEL == KGE_ROTATE) {
        // score = margin - || rot(h, theta) - t ||_2 over the stacked (re, im) vector
        float ss = 0.f;
#pragma unroll
        for (int e = 0; e < E; ++e) {
          t[0][e] = c2[e] - t[0][e];  // residual; padding lanes are 0 - 0
          t[PH - 1][e] = c3[e] - t[PH - 1][e];
          ss += t[0][e] * t[0][e] + t[PH - 1][e] * t[PH - 1][e];
        }
        const float nrm = sqrtf(group_sum<G>(ss));
        const float sc = margin - nrm;
        float dl;
        if (pos) { inst_loss += wpos * softplusf(-sc); dl = -wpos * sigmoidf(-sc); }
        else     { inst_loss += w * softplusf(sc);     dl =  w * sigmoidf(sc); }
        if (a.with_grad) {
          any_grad = true;
          const float f = nrm > 0.f ? -dl / nrm : 0.f;  // dL/d(residual) = dl * (-e / nrm)
#pragma unroll
          for (int e = 0; e < E; ++e) {
            t[0][e] *= f;
            t[PH - 1][e] *= f;
            acc0[e] += t[0][e];
            acc1[e] += t[PH - 1][e];
            t[0][e] = -t[0][e];  // gradient of the tail
            t[PH - 1][e] = -t[PH - 1][e];
          }
          if (pos) {
#pragma unroll
            for (int p = 0; p < PH; ++p)
#pragma unroll
              for (int e = 0; e < E; ++e) gtp[p][e] = t[p][e];
          } else {
#pragma unroll
            for (int p = 0; p < PH; ++p) frag_atomic_add<VEC, G, NCH>(ET.g[p], t_id, d, gl, t[p]);
            touch_row(ET, t_id, st.y, step, gl);
          }
        }
      } else {
        // ComplEx as written in the reference: s = sum tr*A + ti*B
        float ss = 0.f;
#pragma unroll
        for (int e = 0; e < E; ++e) ss += t[0][e] * c0[e] + t[PH - 1][e] * c1[e];
        const float sc = group_sum<G>(ss);
        float dl;
        if (pos) { inst_loss += wpos * softplusf(-sc); dl = -wpos * sigmoidf(-sc); }
        else     { inst_loss += w * softplusf(sc);     dl =  w * sigmoidf(sc); }
        if (a.with_grad) {
          any_grad = true;
#pragma unroll
          for (int e = 0; e < E; ++e) {
            acc0[e] += dl * t[0][e];
            acc1[e] += dl * t[PH - 1][e];
            t[0][e] = dl * c0[e];
            t[PH - 1][e] = dl * c1[e];
          }
          if (pos) {
#pragma unroll
            for (int p = 0; p < PH; ++p)
#pragma unroll
              for (int e = 0; e < E; ++e) gtp[p][e] = t[p][e];
          } else {
#pragma unroll
            for (int p = 0; p < PH; ++p) frag_atomic_add<VEC, G, NCH>(ET.g[p], t_id, d, gl, t[p]);
            touch_row(ET, t_id, st.y, step, gl);
          }
        }
      }
    }

    // ---- gradients of head, relation and positive tail from the accumulators ------------------------
    if (MODEL == KGE_TRANSD) {
      if (nact > 0.f) {
        any_grad = true;
        // gh[0] / gtp[0] hold the gradients of x and of the projected positive tail; back through
        // proj(e) = e + r_p * <e, e_p>:  g_e = g + e_p * <g, r_p>,  g_ep = e * <g, r_p>,  g_rp += g * <e, e_p>
        float dh = 0.f, dt = 0.f;
#pragma unroll
        for (int e = 0; e < E; ++e) {
          dh = __fmaf_rn(gh[0][e], r[PR - 1][e], dh);
          dt = __fmaf_rn(gtp[0][e], r[PR - 1][e], dt);
        }
        dh = group_sum<G>(dh);
        dt = group_sum<G>(dt);
#pragma unroll
        for (int e = 0; e < E; ++e) {
          gr[0][e] = gh[0][e];
          gr[PR - 1][e] = __fmaf_rn(gh[0][e], s_h, __fmaf_rn(gtp[0][e], s_tp, acc1[e]));
          gh[PH - 1][e] = h[0][e] * dh;
          gh[0][e] = __fmaf_rn(h[PH - 1][e], dh, gh[0][e]);
          gtp[PH - 1][e] = tp[0][e] * dt;
          gtp[0][e] = __fmaf_rn(tp[PH - 1][e], dt, gtp[0][e]);
        }
      }
    } else if (MODEL == KGE_TRANSH) {
      if (nact > 0.f) {
        any_grad = true;
        // gh / gtp hold the gradients of x and of the projected positive tail.  The factor c2 = 1 - s_w * w gets
        // g_c = g_x*h + g_tp'*tp + sum_j g_tn'_j*tn_j (acc0), and d c2_j / d w_i = -w_j - s_w * [i == j], so
        // g_w = -s_w * g_c - <g_c, w> on every component.
        float dot = 0.f;
#pragma unroll
        for (int e = 0; e < E; ++e) {
          acc0[e] = __fmaf_rn(gh[0][e], h[0][e], __fmaf_rn(gtp[0][e], tp[0][e], acc0[e]));
          dot = __fmaf_rn(acc0[e], r[PR - 1][e], dot);
        }
        dot = group_sum<G>(dot);
#pragma unroll
        for (int e = 0; e < E; ++e) {
          gr[0][e] = gh[0][e];
          gr[PR - 1][e] = frag_valid<VEC, G, NCH>(d, gl, e) ? (-s_w * acc0[e] - dot) : 0.f;
          gh[0][e] *= c2[e];
          gtp[0][e] *= c2[e];
        }
      }
    } else if (MODEL == KGE_TRANSE) {
      if (nact > 0.f) {
        any_grad = true;
#pragma unroll
        for (int e = 0; e < E; ++e) gr[0][e] = gh[0][e];
      }
    } else if (MODEL == KGE_DISTMULT) {
      if (nact > 0.f) {
        any_grad = true;
#pragma unroll
        for (int e = 0; e < E; ++e) {
          gh[0][e] = r[0][e] * acc0[e];
          gr[0][e] = h[0][e] * acc0[e];
          gtp[0][e] = -nact * w * c0[e];
        }
      }
    } else if (MODEL == KGE_ROTATE) {
      if (any_grad) {
#pragma unroll
        for (int e = 0; e < E; ++e) {
          gh[0][e] = c0[e] * acc0[e] + c1[e] * acc1[e];
          gh[PH - 1][e] = -c1[e] * acc0[e] + c0[e] * acc1[e];
          gr[0][e] = -acc0[e] * c3[e] + acc1[e] * c2[e];
        }
      }
    } else {
      if (any_grad) {
#pragma unroll
        for (int e = 0; e < E; ++e) {
          gh[0][e] = r[0][e] * acc0[e] + r[PR - 1][e] * acc1[e];
          gh[PH - 1][e] = r[0][e] * acc1[e] - r[PR - 1][e] * acc1[e];
          gr[0][e] = h[0][e] * acc0[e] + h[PH - 1][e] * acc1[e];
          gr[PR - 1][e] = h[0][e] * acc1[e] - h[PH - 1][e] * acc1[e];
        }
      }
    }

    if (gl == 0) lsum += inst_loss;

    if (any_grad) {
#pragma unroll
      for (int p = 0; p < PH; ++p) {
        frag_atomic_add<VEC, G, NCH>(HT.g[p], h_id, d, gl, gh[p]);
        frag_atomic_add<VEC, G, NCH>(ET.g[p], tp_id, d, gl, gtp[p]);
      }
      touch_row(HT, h_id, sh.y, step, gl);
      touch_row(ET, tp_id, stp.y, step, gl);
      if (is_rec) {
        rec_seen = true;
#pragma unroll
        for (int p = 0; p < PR; ++p)
#pragma unroll
          for (int e = 0; e < E; ++e) racc[p][e] += gr[p][e];
      } else if (!WARP_RACC) {
#pragma unroll
        for (int p = 0; p < PR; ++p) frag_atomic_add<VEC, G, NCH>(RT.g[p], r_id, d, gl, gr[p]);
        touch_row(RT, r_id, sr.y, step, gl);
      }
    }

    if constexpr (WARP_RACC && !is_rec) {
      // The two groups of the warp run triples i and i + 1 (i even).  Lane l and lane l + 16 hold the same columns:
      // when both triples name the same relation, group 1 hands its fragment to group 0, which writes alone.
      const bool pair = (i | 1) < n_seg;   // (group 1 has left the loop when this is false)
      __syncwarp(pair ? 0xffffffffu : 0x0000ffffu);   // orders the other group's add of the previous iteration
      bool write = any_grad;
      if (pair) {
        const int r_other = __shfl_xor_sync(0xffffffffu, (int)r_id, 16);
        if (r_other == (int)r_id) {
          const bool any_other = __shfl_xor_sync(0xffffffffu, any_grad ? 1 : 0, 16) != 0;
#pragma unroll
          for (int p = 0; p < PR; ++p)
#pragma unroll
            for (int e = 0; e < E; ++e) gr[p][e] += __shfl_xor_sync(0xffffffffu, gr[p][e], 16);
          write = (threadIdx.x & 16) == 0 && (any_grad || any_other);
        }
      }
      if (write) {
        warp_copy_add((int)r_id, gr);
        if (gl == 0) s_rtouch[r_id] = 1;
      }
    }
  }

  };
  run_half(std::true_type{});
  if constexpr (WARP_RACC) {
    // the user->item relation gradient of this warp: both groups hold the same columns
#pragma unroll
    for (int p = 0; p < PR; ++p)
#pragma unroll
      for (int e = 0; e < E; ++e) racc[p][e] += __shfl_xor_sync(0xffffffffu, racc[p][e], 16);
    if (__any_sync(0xffffffffu, rec_seen) && (threadIdx.x & 16) == 0) {
      warp_copy_add(a.m.ui_relation, racc);
      if (gl == 0) s_rtouch[a.m.ui_relation] = 1;
    }
  }
  run_half(std::false_type{});

  // ---- CTA epilogue: relation gradients and the loss --------------------------------------------
  if constexpr (WARP_RACC) {
    // sum the warp copies of every row this CTA touched: one float4 RED per 4 columns, one mark per row
    __syncthreads();
    const float4* s4 = reinterpret_cast<const float4*>(s_racc);
    const int row_len = PR * nv;
    const int warp_stride = n_rel * row_len;
    for (int k = threadIdx.x; k < warp_stride; k += blockDim.x) {
      const int row = k / row_len;
      if (!s_rtouch[row]) continue;
      const int p = (k - row * row_len) / nv, c = k - row * row_len - p * nv;
      float4 s = s4[k];
#pragma unroll
      for (int w = 1; w < kFwdWarps; ++w) {
        const float4 v = s4[w * warp_stride + k];
        s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
      }
      atomicAdd(reinterpret_cast<float4*>((p == 0 ? RT.g[0] : RT.g[PR - 1]) + (int64_t)row * d) + c, s);
    }
    for (int row = threadIdx.x; row < n_rel; row += blockDim.x)
      if (s_rtouch[row]) touch_row(RT, row, -1, step, 0);
  } else {
    if (rec_seen) {
#pragma unroll
      for (int p = 0; p < PR; ++p) {
#pragma unroll
        for (int e = 0; e < E; ++e) {
          const int j = e / VEC;
          const int col = (gl + j * G) * VEC + (e % VEC);
          if (col < d) atomicAdd(&s_racc[p * d + col], racc[p][e]);
        }
      }
    }
    const int any_rec = __syncthreads_or(rec_seen ? 1 : 0);
    if (any_rec) {
      for (int i = threadIdx.x; i < PR * d; i += blockDim.x) {
        const int p = i / d, col = i - p * d;
        atomicAdd(RT.g[p] + (int64_t)a.m.ui_relation * d + col, s_racc[i]);
      }
      if (threadIdx.x == 0) touch_row(RT, a.m.ui_relation, -1, step, 0);
    }
  }
  lsum = warp_sum(lsum);
  if ((threadIdx.x & 31) == 0) s_loss[threadIdx.x >> 5] = lsum;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int i = 0; i < (int)(blockDim.x >> 5); ++i) t += s_loss[i];
    if (t != 0.f) atomicAdd(a.loss, t);
  }
}

// ---- scanning the row states -------------------------------------------------------------------
// Lanes read the 8-byte states of 32 consecutive rows, ballot the rows selected by `pred` and the
// lane groups of the warp then work on the selected rows, 32/G at a time.  `body(row, last_step)`
// runs converged within a group.
// `win` (4..32) rows per warp window: small windows spread a densely touched small table over
// more warps, 32 keeps the scan of a large sparse table cheap.
template <int G, typename Pred, typename Body>
__device__ __forceinline__ void for_selected_rows(const kge_table_t& T, int win, Pred pred, Body body) {
  constexpr int NG = 32 / G;
  const int lane = threadIdx.x & 31;
  const int grp = lane / G;
  const int64_t warp_global = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t base = warp_global * win; base < T.rows; base += n_warps * win) {
    const int64_t row = base + lane;
    const bool mine = lane < win && row < T.rows;
    int2 st = make_int2(-1, -1);
    if (mine) st = *(reinterpret_cast<const int2*>(T.row_state) + row);
    unsigned mask = __ballot_sync(0xffffffffu, mine && pred(st));
    while (mask) {
      unsigned m = mask;  // group `grp` takes the grp-th set bit
      for (int q = 0; q < grp; ++q) m &= m - 1;
      const int bit = m ? (__ffs(m) - 1) : -1;
      const int last = __shfl_sync(0xffffffffu, st.x, bit < 0 ? 0 : bit);
      if (bit >= 0) body(base + bit, last);
      for (int q = 0; q < NG && mask; ++q) mask &= mask - 1;
      __syncwarp();
    }
  }
}

struct ApplyArgs {
  kge_model_t m;
  AdamDev adam;
  float scale;
  const float* scale_dev;  // optional device-side factor (the incoming grad of the loss)
  int win[3];              // scan window per table
};

template <int VEC, int G, int NCH>
__device__ __forceinline__ void adam_row(const kge_table_t& T, int64_t row, int last, int d, int gl, const AdamDev& A,
                                         float scale) {
  constexpr int E = VEC * NCH;
  const float2 c = adam_consts(A, A.step);
  // RMSprop: the second moment of a row that skipped n steps decayed by alpha^n meanwhile (torch multiplies it by
  // alpha once per step, gradient or not); a row never touched before has v = 0
  const float lag_decay = (A.opt == KGE_OPT_RMSPROP && last >= 0 && last < A.step - 1)
                              ? powf(A.b2, (float)(A.step - 1 - last)) : 1.f;
  for (int part = 0; part < T.parts; ++part) {
    float p[E], m[E], v[E], g[E];
    frag_load<VEC, G, NCH>(T.w[part], row, d, gl, p);
    if (A.opt == KGE_OPT_ADAM) frag_load<VEC, G, NCH>(T.m[part], row, d, gl, m);
    if (A.opt != KGE_OPT_SGD) frag_load<VEC, G, NCH>(T.v[part], row, d, gl, v);
    frag_load_cg<VEC, G, NCH>(T.g[part], row, d, gl, g);
    float z[E];
    if (A.opt == KGE_OPT_ADAM) {
      if (last >= 0 && last < A.step - 1) adam_replay<E>(p, m, v, last, A.step - 1, A);
#pragma unroll
      for (int e = 0; e < E; ++e) {
        const float ge = g[e] * scale;
        m[e] += A.omb1 * (ge - m[e]);
        v[e] = v[e] * A.b2 + A.omb2 * ge * ge;
        const float den = sqrt_nonneg(v[e]) * c.y + A.eps;
        p[e] -= c.x * div_pos_den(m[e], den);
        z[e] = 0.f;
      }
      frag_store<VEC, G, NCH>(T.m[part], row, d, gl, m);
    } else {
#pragma unroll
      for (int e = 0; e < E; ++e) {
        const float ge = g[e] * scale;
        if (A.opt == KGE_OPT_SGD) {
          p[e] -= A.lr * ge;
        } else {
          v[e] = A.opt == KGE_OPT_ADAGRAD ? __fmaf_rn(ge, ge, v[e]) : __fmaf_rn(A.omb2 * ge, ge, v[e] * lag_decay * A.b2);
          p[e] -= A.lr * div_pos_den(ge, sqrt_nonneg(v[e]) + A.eps);
        }
        z[e] = 0.f;
      }
    }
    frag_store<VEC, G, NCH>(T.w[part], row, d, gl, p);
    if (A.opt != KGE_OPT_SGD) frag_store<VEC, G, NCH>(T.v[part], row, d, gl, v);
    frag_store<VEC, G, NCH>(T.g[part], row, d, gl, z);
  }
  if (gl == 0) T.row_state[2 * row] = A.step;  // last_step; touch_step keeps `step` (stale from step+1 on)
}

template <int VEC, int G, int NCH>
__global__ void __launch_bounds__(256) adam_apply_kernel(const ApplyArgs a) {
  const int gl = (threadIdx.x & 31) % G;
  const int step = a.adam.step;
  const float scale = a.scale_dev ? a.scale * __ldg(a.scale_dev) : a.scale;
  auto marked = [step](int2 st) { return st.y == step; };
  // (the tables are kernel parameters: index them by name, a pointer array would copy them to local memory)
  for_selected_rows<G>(a.m.user, a.win[0], marked, [&](int64_t row, int last) {
    adam_row<VEC, G, NCH>(a.m.user, row, last, a.m.d, gl, a.adam, scale);
  });
  for_selected_rows<G>(a.m.entity, a.win[1], marked, [&](int64_t row, int last) {
    adam_row<VEC, G, NCH>(a.m.entity, row, last, a.m.d, gl, a.adam, scale);
  });
  for_selected_rows<G>(a.m.relation, a.win[2], marked, [&](int64_t row, int last) {
    adam_row<VEC, G, NCH>(a.m.relation, row, last, a.m.d, gl, a.adam, scale);
  });
}

// ---- dense catch-up of every row to adam.step (before weights are read by others) ------------
template <int VEC, int G, int NCH>
__global__ void __launch_bounds__(256) adam_flush_kernel(const kge_table_t T, int d, const AdamDev A, int win) {
  constexpr int E = VEC * NCH;
  const int gl = (threadIdx.x & 31) % G;
  const int step = A.step;
  for_selected_rows<G>(
      T, win, [step](int2 st) { return st.x >= 0 && st.x < step; },
      [&](int64_t row, int last) {
        for (int part = 0; part < T.parts; ++part) {
          float p[E], m[E], v[E];
          if (A.opt != KGE_OPT_ADAM) {   // the weights of an idle row do not move; RMSprop's second moment decays
            if (A.opt == KGE_OPT_RMSPROP) {
              frag_load<VEC, G, NCH>(T.v[part], row, d, gl, v);
              const float f = powf(A.b2, (float)(A.step - last));
#pragma unroll
              for (int e = 0; e < E; ++e) v[e] *= f;
              frag_store<VEC, G, NCH>(T.v[part], row, d, gl, v);
            }
            continue;
          }
          frag_load<VEC, G, NCH>(T.w[part], row, d, gl, p);
          frag_load<VEC, G, NCH>(T.m[part], row, d, gl, m);
          frag_load<VEC, G, NCH>(T.v[part], row, d, gl, v);
          adam_replay<E>(p, m, v, last, A.step, A);
          frag_store<VEC, G, NCH>(T.w[part], row, d, gl, p);
          frag_store<VEC, G, NCH>(T.m[part], row, d, gl, m);
          frag_store<VEC, G, NCH>(T.v[part], row, d, gl, v);
        }
        if (gl == 0) T.row_state[2 * row] = A.step;
      });
}

// ---- discard / pack / add (row-sparse exchange) --------------------------------------------------
// take: every row marked in `step` gives up its gradient row (zeroed, mark cleared); with outputs
// the rows are compacted into ids_out / rows_out (order unspecified) and *count_out is advanced.
template <int VEC, int G, int NCH>
__global__ void __launch_bounds__(256) grad_take_kernel(const kge_table_t T, int d, int step, int64_t* ids_out,
                                                        float* rows_out, int32_t* count_out) {
  constexpr int E = VEC * NCH;
  constexpr int NG = 32 / G;
  const int lane = threadIdx.x & 31, gl = lane % G, grp = lane / G;
  const int64_t warp_global = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t base = warp_global * 32; base < T.rows; base += n_warps * 32) {
    const int64_t row_l = base + lane;
    int touch = -1;
    if (row_l < T.rows) touch = T.row_state[2 * row_l + 1];
    unsigned mask = __ballot_sync(0xffffffffu, touch == step);
    if (!mask) continue;
    int slot0 = 0;
    if (count_out) {  // one returning atomic per 32 scanned rows that hold anything
      if (lane == 0) slot0 = atomicAdd(count_out, __popc(mask));
      slot0 = __shfl_sync(0xffffffffu, slot0, 0);
    }
    int taken = 0;
    while (mask) {
      unsigned m = mask;
      for (int q = 0; q < grp; ++q) m &= m - 1;
      const int bit = m ? (__ffs(m) - 1) : -1;
      if (bit >= 0) {
        const int64_t row = base + bit;
        const int64_t idx = slot0 + taken + grp;
        for (int part = 0; part < T.parts; ++part) {
          float g[E], z[E];
          frag_load_cg<VEC, G, NCH>(T.g[part], row, d, gl, g);
#pragma unroll
          for (int e = 0; e < E; ++e) z[e] = 0.f;
          frag_store<VEC, G, NCH>(T.g[part], row, d, gl, z);
          if (rows_out) frag_store<VEC, G, NCH>(rows_out + (int64_t)part * d, idx * T.parts, d, gl, g);
        }
        if (gl == 0) {
          T.row_state[2 * row + 1] = -1;
          if (ids_out) ids_out[idx] = row;
        }
      }
      for (int q = 0; q < NG && mask; ++q) {
        mask &= mask - 1;
        ++taken;
      }
      __syncwarp();
    }
  }
}

template <int VEC, int G, int NCH>
__global__ void __launch_bounds__(256) grad_add_kernel(const kge_table_t T, int d, int step, const int64_t* ids,
                                                       const float* rows, const int32_t* count_dev) {
  constexpr int E = VEC * NCH;
  const int gl = (threadIdx.x & 31) % G;
  const int groups_per_cta = blockDim.x / G;
  const int64_t n_groups = (int64_t)gridDim.x * groups_per_cta;
  const int64_t total = *count_dev;
  for (int64_t idx = (int64_t)blockIdx.x * groups_per_cta + threadIdx.x / G; idx < total; idx += n_groups) {
    const int64_t row = ids[idx];
    for (int part = 0; part < T.parts; ++part) {
      float g[E], x[E];
      frag_load_cg<VEC, G, NCH>(T.g[part], row, d, gl, g);
      frag_load<VEC, G, NCH>(rows + (int64_t)part * d, idx * T.parts, d, gl, x);
#pragma unroll
      for (int e = 0; e < E; ++e) g[e] += x[e];
      frag_store<VEC, G, NCH>(T.g[part], row, d, gl, g);
    }
    if (gl == 0) T.row_state[2 * row + 1] = step;
  }
}

AdamDev make_adam_dev(const kge_model_t* m, const kge_adam_t* a) {
  AdamDev A;
  A.lr = a->lr;
  A.b1 = a->beta1;
  A.b2 = a->beta2;
  A.eps = a->eps;
  A.omb1 = (float)(1.0 - (double)a->beta1);
  A.omb2 = (float)(1.0 - (double)a->beta2);
  A.step = a->step;
  A.opt = a->optimizer;
  A.cap = a->replay_cap > 0 ? a->replay_cap : 200;
  A.table = reinterpret_cast<const float2*>(m->adam_table);
  A.tlen = m->adam_table ? m->adam_table_len : 0;
  return A;
}

int grid_for(int64_t n_groups_needed, int groups_per_cta, int ctas_per_sm) {
  int64_t g = (n_groups_needed + groups_per_cta - 1) / groups_per_cta;
  const int64_t cap = (int64_t)kge_num_sms() * ctas_per_sm;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return (int)g;
}

// scan window: as large as still gives every resident warp (32 per SM) a window of its own
int scan_window(int64_t rows) {
  const int64_t warps = (int64_t)kge_num_sms() * 32;
  int win = 32;
  while (win > 4 && (rows + win - 1) / win < warps) win >>= 1;
  return win;
}
// grid for a scan over `rows` row states: `win` rows per warp iteration, 8 warps per CTA
int scan_grid(int64_t rows, int win, int ctas_per_sm) { return grid_for((rows + win - 1) / win, 8, ctas_per_sm); }

bool table_has_state(const kge_table_t& T, bool need_rows) {
  for (int p = 0; p < T.parts; ++p)
    if (!T.g[p] || (need_rows && (!T.m[p] || !T.v[p]))) return false;
  return !need_rows || T.row_state != nullptr;
}

// need_state: gradient accumulators; need_rows: also moments and row states (the row-lazy Adam kernels)
int check_model(const kge_model_t* m, bool need_state, bool need_rows = true) {
  KGE_REQUIRE(m, KGE_E_ARG, "model is NULL");
  KGE_REQUIRE(m->model >= KGE_TRANSE && m->model <= KGE_TRANSD, KGE_E_ARG, "unknown model kind %d", m->model);
  const int ph = (m->model == KGE_ROTATE || m->model == KGE_COMPLEX || m->model == KGE_TRANSD) ? 2 : 1;
  const int pr = (m->model == KGE_COMPLEX || m->model == KGE_TRANSH || m->model == KGE_TRANSD) ? 2 : 1;
  KGE_REQUIRE(m->user.parts == ph && m->entity.parts == ph && m->relation.parts == pr, KGE_E_ARG,
              "table parts do not match the model kind");
  for (int p = 0; p < ph; ++p) KGE_REQUIRE(m->user.w[p] && m->entity.w[p], KGE_E_ARG, "NULL weight table");
  for (int p = 0; p < pr; ++p) KGE_REQUIRE(m->relation.w[p], KGE_E_ARG, "NULL relation table");
  RowCfg c = {};
  KGE_REQUIRE(kge_pick_rowcfg(m->d, c), KGE_E_UNSUPPORTED,
              "embedding_size %d unsupported (1 to %d)", m->d, KGE_MAX_D);
  if (need_state) {
    KGE_REQUIRE(table_has_state(m->user, need_rows) && table_has_state(m->entity, need_rows) &&
                    table_has_state(m->relation, need_rows), KGE_E_STATE, "optimiser state buffers missing");
  }
  return 0;
}

}  // namespace

// =================================== C ABI ===================================================

extern "C" int kge_adam_table_fill(float lr, float beta1, float beta2, float* out_host, int32_t len) {
  // entries beyond the table are (lr, 1): both corrections are 1 to fp32 resolution there
  const double b = beta1 > beta2 ? beta1 : beta2;
  int need = 2;
  if (b > 0.0 && b < 1.0) need = (int)ceil(log(1e-10) / log(b)) + 2;
  if (!out_host) return need;
  for (int j = 0; j < len; ++j) {
    if (j == 0) { out_host[0] = lr; out_host[1] = 1.f; continue; }
    const double bc1 = 1.0 - pow((double)beta1, j), bc2 = 1.0 - pow((double)beta2, j);
    out_host[2 * j] = (float)((double)lr / bc1);
    out_host[2 * j + 1] = (float)(1.0 / sqrt(bc2));
  }
  return need;
}

extern "C" int kge_train_forward(const kge_model_t* model, const kge_batch_t* b, const kge_adam_t* adam,
                                 int with_grad, float* loss_out, kge_stream_t stream) {
  // (a training pass without row states accumulates gradients for a dense optimiser step: kge_owner_adam_step)
  const bool rows_given = model && (model->user.row_state || model->entity.row_state || model->relation.row_state);
  if (int e = check_model(model, with_grad != 0, rows_given)) return e;
  KGE_REQUIRE(b && adam && loss_out, KGE_E_ARG, "NULL batch / adam / loss_out");
  KGE_REQUIRE(b->n_rec >= 0 && b->n_kg >= 0 && b->k_rec >= 1 && b->k_kg >= 1, KGE_E_ARG, "bad batch sizes");
  KGE_REQUIRE(adam->step >= 1, KGE_E_ARG, "adam.step is 1-based");
  KGE_REQUIRE(adam->optimizer >= KGE_OPT_ADAM && adam->optimizer <= KGE_OPT_RMSPROP, KGE_E_ARG, "unknown optimizer %d",
              adam->optimizer);
  const int64_t n_total = b->n_rec + b->n_kg;
  if (n_total == 0) return 0;
  KGE_REQUIRE(b->n_rec == 0 || (b->user && b->item && b->neg_item), KGE_E_ARG, "NULL rec id array");
  KGE_REQUIRE(b->n_kg == 0 || (b->head && b->relation && b->tail && b->neg_tail), KGE_E_ARG, "NULL KG id array");
  const bool any_state = model->user.row_state || model->entity.row_state || model->relation.row_state;
  const bool all_state = model->user.row_state && model->entity.row_state && model->relation.row_state;
  KGE_REQUIRE(any_state == all_state, KGE_E_STATE, "row_state must be given for all tables or none");
  KGE_REQUIRE(!all_state || (model->user.m[0] && model->entity.m[0] && model->relation.m[0]), KGE_E_STATE,
              "row_state without moments");

  TrainArgs a;
  a.m = *model;
  a.b = *b;
  a.adam = make_adam_dev(model, adam);
  a.with_grad = with_grad;
  a.loss = loss_out;
  const double pr = (double)b->n_rec * b->k_rec, pk = (double)b->n_kg * b->k_kg;
  // (TorusE's training objective is TransE's: TripletMarginLoss on h + r, toruse.py:81-102)
  const int kind = model->model == KGE_TORUSE ? KGE_TRANSE : model->model;
  if (kind == KGE_TRANSE || kind == KGE_DISTMULT || kind == KGE_TRANSH || kind == KGE_TRANSD) {
    a.w_rec = a.w_kg = (float)(1.0 / (pr + pk));
    a.wpos_rec = a.wpos_kg = 0.f;
  } else {
    a.w_rec = pr > 0 ? (float)(0.5 / pr) : 0.f;
    a.w_kg = pk > 0 ? (float)(0.5 / pk) : 0.f;
    a.wpos_rec = pr > 0 ? (float)(0.5 / (double)b->n_rec) : 0.f;
    a.wpos_kg = pk > 0 ? (float)(0.5 / (double)b->n_kg) : 0.f;
  }
  RowCfg c = {};
  kge_pick_rowcfg(model->d, c);
  // Rows of 17..32 float4 (d = 68..128: cfg2's d = 100, cfg5's d = 128): two triples per warp -- half-warp groups,
  // two fragments per lane -- instead of one, when the tables (weights, moments, gradient accumulators: 16 B per
  // element) fit the L2.  There the step is bound by instruction issue, and the loop's scalar work (ids, row states,
  // loss bookkeeping, branches) is issued once per two triples: cfg2 0.395 -> 0.366 ms/step.  With tables beyond the
  // L2 the step is bound by bytes in flight, which the fatter threads (two CTAs per SM instead of four) halve: cfg5
  // 1.012 -> 1.055 ms/step, so that regime keeps one triple per warp.
  const double table_bytes = ((double)model->user.rows + (double)model->entity.rows) * model->d * 16.0;
  // (a batch that does not fill the resident warps even once -- the reference's 2048 + 2048 -- is bound by the
  // length of one warp's dependent instruction chain: one triple per warp halves it and doubles the warps)
  const bool two_per_warp = c.vec == 4 && c.g == 32 && c.nch == 1 && table_bytes < 96e6 &&
                            n_total >= (int64_t)kge_num_sms() * 256 &&
                            (kind == KGE_TRANSE || kind == KGE_DISTMULT);
  const int threads = 256;
  int grid = grid_for(n_total, threads / (two_per_warp ? 16 : c.g), 8);
  size_t smem = (size_t)model->relation.parts * model->d * sizeof(float);
  cudaStream_t st = (cudaStream_t)stream;
  // Two triples per warp with gradients: relation gradients go through per-warp copies in shared memory when those
  // fit at the residency the kernel's register budget is shaped for.  The grid is then sized to what is resident,
  // so that every CTA zeroes and flushes its copies once.
  bool warp_racc = false;
  if (two_per_warp && with_grad) {
    const size_t ws = warp_racc_smem_bytes(model->relation.rows, model->relation.parts, model->d);
    auto kern = kind == KGE_TRANSE ? train_fwd_kernel<KGE_TRANSE, 4, 16, 2, true>
                                   : train_fwd_kernel<KGE_DISTMULT, 4, 16, 2, true>;
    const int min_ctas = kind == KGE_TRANSE ? FwdBounds<KGE_TRANSE, 4, 16, 2>::MIN_CTAS
                                            : FwdBounds<KGE_DISTMULT, 4, 16, 2>::MIN_CTAS;
    int dev = 0, optin = 0, resident = 0;
    KGE_CUDA(cudaGetDevice(&dev));
    KGE_CUDA(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    if (ws <= (size_t)optin) {
      KGE_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ws));
      KGE_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&resident, kern, threads, ws));
    }
    if (resident >= min_ctas) {
      warp_racc = true;
      smem = ws;
      grid = grid_for(n_total, threads / 16, resident);
    }
  }
#define CALL(V, G, N)                                                                                   \
  switch (kind) {                                                                                       \
    case KGE_TRANSE: train_fwd_kernel<KGE_TRANSE, V, G, N><<<grid, threads, smem, st>>>(a); break;      \
    case KGE_DISTMULT: train_fwd_kernel<KGE_DISTMULT, V, G, N><<<grid, threads, smem, st>>>(a); break;  \
    case KGE_ROTATE: train_fwd_kernel<KGE_ROTATE, V, G, N><<<grid, threads, smem, st>>>(a); break;      \
    case KGE_TRANSH: train_fwd_kernel<KGE_TRANSH, V, G, N><<<grid, threads, smem, st>>>(a); break;      \
    case KGE_TRANSD: train_fwd_kernel<KGE_TRANSD, V, G, N><<<grid, threads, smem, st>>>(a); break;      \
    default: train_fwd_kernel<KGE_COMPLEX, V, G, N><<<grid, threads, smem, st>>>(a); break;             \
  }
  if (warp_racc) {
    if (kind == KGE_TRANSE) train_fwd_kernel<KGE_TRANSE, 4, 16, 2, true><<<grid, threads, smem, st>>>(a);
    else train_fwd_kernel<KGE_DISTMULT, 4, 16, 2, true><<<grid, threads, smem, st>>>(a);
  } else if (two_per_warp) {
    if (kind == KGE_TRANSE) train_fwd_kernel<KGE_TRANSE, 4, 16, 2><<<grid, threads, smem, st>>>(a);
    else train_fwd_kernel<KGE_DISTMULT, 4, 16, 2><<<grid, threads, smem, st>>>(a);
  } else {
    KGE_DISPATCH_ROWCFG(c, CALL);
  }
#undef CALL
  KGE_LAUNCH_CHECK();
  return 0;
}

extern "C" int kge_adam_apply(const kge_model_t* model, const kge_adam_t* adam, float grad_scale,
                              const float* grad_scale_dev, kge_stream_t stream) {
  if (int e = check_model(model, true)) return e;
  KGE_REQUIRE(adam && adam->step >= 1, KGE_E_ARG, "bad adam");
  ApplyArgs a;
  a.m = *model;
  a.adam = make_adam_dev(model, adam);
  a.scale = grad_scale;
  a.scale_dev = grad_scale_dev;
  RowCfg c = {};
  kge_pick_rowcfg(model->d, c);
  const int threads = 256;
  const int64_t max_rows = model->entity.rows > model->user.rows ? model->entity.rows : model->user.rows;
  a.win[0] = scan_window(model->user.rows);
  a.win[1] = scan_window(model->entity.rows);
  a.win[2] = 4;
  const int grid = scan_grid(max_rows, scan_window(max_rows), 4);
  cudaStream_t st = (cudaStream_t)stream;
#define CALL(V, G, N) adam_apply_kernel<V, G, N><<<grid, threads, 0, st>>>(a)
  KGE_DISPATCH_ROWCFG(c, CALL);
#undef CALL
  KGE_LAUNCH_CHECK();
  return 0;
}

extern "C" int kge_train_step(const kge_model_t* model, const kge_batch_t* b, const kge_adam_t* adam,
                              float grad_scale, float* loss_out, kge_stream_t stream) {
  if (int e = kge_train_forward(model, b, adam, 1, loss_out, stream)) return e;
  if (b->n_rec + b->n_kg == 0) return 0;
  return kge_adam_apply(model, adam, grad_scale, nullptr, stream);
}

extern "C" int kge_adam_flush(const kge_model_t* model, const kge_adam_t* adam, kge_stream_t stream) {
  if (int e = check_model(model, true)) return e;
  KGE_REQUIRE(adam && adam->step >= 0, KGE_E_ARG, "bad adam");
  if (adam->step == 0) return 0;
  AdamDev A = make_adam_dev(model, adam);
  RowCfg c = {};
  kge_pick_rowcfg(model->d, c);
  const int threads = 256;
  cudaStream_t st = (cudaStream_t)stream;
  const kge_table_t* tabs[3] = {&model->user, &model->entity, &model->relation};
  for (int t = 0; t < 3; ++t) {
    const int win = scan_window(tabs[t]->rows);
    const int grid = scan_grid(tabs[t]->rows, win, 8);
#define CALL(V, G, N) adam_flush_kernel<V, G, N><<<grid, threads, 0, st>>>(*tabs[t], model->d, A, win)
    KGE_DISPATCH_ROWCFG(c, CALL);
#undef CALL
    KGE_LAUNCH_CHECK();
  }
  return 0;
}

static int grad_take(const kge_model_t* model, int which, int step, int64_t* ids_out, float* rows_out,
                     int32_t* count_out, cudaStream_t st) {
  const kge_table_t* tabs[3] = {&model->user, &model->entity, &model->relation};
  const kge_table_t& T = *tabs[which];
  RowCfg c = {};
  kge_pick_rowcfg(model->d, c);
  const int threads = 256;
  const int grid = scan_grid(T.rows, 32, 4);
  if (count_out) KGE_CUDA(cudaMemsetAsync(count_out, 0, sizeof(int32_t), st));
#define CALL(V, G, N) \
  grad_take_kernel<V, G, N><<<grid, threads, 0, st>>>(T, model->d, step, ids_out, rows_out, count_out)
  KGE_DISPATCH_ROWCFG(c, CALL);
#undef CALL
  KGE_LAUNCH_CHECK();
  return 0;
}

extern "C" int kge_grad_discard(const kge_model_t* model, int32_t step, kge_stream_t stream) {
  if (int e = check_model(model, true)) return e;
  for (int t = 0; t < 3; ++t)
    if (int e = grad_take(model, t, step, nullptr, nullptr, nullptr, (cudaStream_t)stream)) return e;
  return 0;
}

extern "C" int kge_grad_pack(const kge_model_t* model, int32_t which, int32_t step, int64_t* ids_out,
                             float* rows_out, int32_t* count_out, kge_stream_t stream) {
  if (int e = check_model(model, true)) return e;
  KGE_REQUIRE(which >= 0 && which < 3 && ids_out && rows_out && count_out, KGE_E_ARG, "bad pack arguments");
  return grad_take(model, which, step, ids_out, rows_out, count_out, (cudaStream_t)stream);
}

extern "C" int kge_grad_add(const kge_model_t* model, int32_t which, int32_t step, const int64_t* ids,
                            const float* rows, const int32_t* count_dev, int64_t max_count, kge_stream_t stream) {
  if (int e = check_model(model, true)) return e;
  KGE_REQUIRE(which >= 0 && which < 3 && ids && rows && count_dev && max_count >= 0, KGE_E_ARG, "bad add arguments");
  if (max_count == 0) return 0;
  const kge_table_t* tabs[3] = {&model->user, &model->entity, &model->relation};
  RowCfg c = {};
  kge_pick_rowcfg(model->d, c);
  const int threads = 256;
  const int grid = grid_for(max_count, threads / c.g, 4);
#define CALL(V, G, N)                                                                                            \
  grad_add_kernel<V, G, N><<<grid, threads, 0, (cudaStream_t)stream>>>(*tabs[which], model->d, step, ids, rows, \
                                                                         count_dev)
  KGE_DISPATCH_ROWCFG(c, CALL);
#undef CALL
  KGE_LAUNCH_CHECK();
  return 0;
}
