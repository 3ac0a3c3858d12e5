// Scoring side of the KGE hot path for sm_100a: predict, dense full-sort scores and the fused
// full-sort + mask + per-user top-k, all on the CUDA cores in exact fp32.
//
// Replaces (paths under /root/reference/hopwise/):
//   model/knowledge_graph_embedding_recommender/{transe.py:100-154, distmult.py:97-146,
//   rotate.py:133-220, complex.py:130-219}         (predict / full_sort_predict and _kg twins)
//   trainer/trainer.py:716-735                     (scores[:, 0] = -inf; scores[history] = -inf)
//   evaluator/collector.py:176-177                 (torch.topk over [n, I])
//
// All five scorers are "transform the (head, relation) pair into one query vector q of
// Kdim = parts*d floats, then reduce against the target row t":
//   TransE   q = h + r                      score = -||q - t||
//   RotatE   q = rot(h, theta) (re | im)    score = margin - ||q - t||   (one L2 norm, rotate.py:61-69)
//   DistMult q = h * r                      score = q . t
//   ComplEx  q = (hr*rr | hi*rr + hr*ri - hi*ri)   score = q . t        (complex.py:53-62 as written)
//   TorusE   q = frac(h) + frac(r)          score = -4 * sum(min(x^2, 1 - x^2)), x = q - frac(t)
// so one tile kernel serves them all: a CTA owns BU query rows (q kept in shared memory for
// the whole sweep; BU = 32, or 16 when 32 rows of q do not fit) and streams target tiles of
// BT=128 rows through shared memory in K-chunks of 32 floats; each thread accumulates a
// (BU/8)x4 register block.  The epilogue either stores the dense [n, n_targets] scores (API
// parity: the unchanged trainer mutates that tensor) or keeps a per-row sorted top-k list of
// 64-bit (score, ~id) keys in shared memory, so the dense matrix never exists (800 GB at
// 1M x 200k).  Order: score descending, id ascending.  A third epilogue counts, for listed
// targets (the positives), the targets scoring above and equal to them over the whole masked
// row: the exact ranks GAUC reads (collector.py's rec.meanrank).
// TransH and TransD have no scorer here: transh_project_kernel / transd_project_kernel write projected rows, which
// the caller scores as TransE (check_score_model refuses both model kinds).
#include <math.h>

#include "common.cuh"
#include "score_common.cuh"

namespace {

constexpr int BT = 128;   // target rows per tile
constexpr int KC = 32;    // K chunk (floats)
constexpr int TS = KC + 4;  // padded row stride of the target tile: conflict-free LDS.128
constexpr int TILE_THREADS = 256;

// ---- predict: one lane group per (head, relation, tail) -------------------------------------
template <int MODEL, int VEC, int G, int NCH>
__global__ void __launch_bounds__(256) predict_kernel(const ScoreArgs a, float* __restrict__ out) {
  constexpr int E = VEC * NCH;
  constexpr int PH = (MODEL == KGE_ROTATE || MODEL == KGE_COMPLEX) ? 2 : 1;
  constexpr int PR = MODEL == KGE_COMPLEX ? 2 : 1;
  const int d = a.m.d;
  const int gl = (threadIdx.x & 31) % G;
  const int groups_per_cta = blockDim.x / G;
  const int64_t n_groups = (int64_t)gridDim.x * groups_per_cta;
  const kge_table_t& HT = a.head_is_user ? a.m.user : a.m.entity;
  for (int64_t i = (int64_t)blockIdx.x * groups_per_cta + threadIdx.x / G; i < a.n; i += n_groups) {
    const int64_t h_id = __ldg(a.heads + i);
    const int64_t r_id = a.rels ? __ldg(a.rels + i) : (int64_t)a.rel_row;
    const int64_t t_id = __ldg(a.tails + i);
    float h[PH][E], r[PR][E], t[PH][E];
#pragma unroll
    for (int p = 0; p < PH; ++p) {
      frag_load<VEC, G, NCH>(HT.w[p], h_id, d, gl, h[p]);
      frag_load<VEC, G, NCH>(a.m.entity.w[p], t_id, d, gl, t[p]);
    }
#pragma unroll
    for (int p = 0; p < PR; ++p) frag_load<VEC, G, NCH>(a.m.relation.w[p], r_id, d, gl, r[p]);
    float s = 0.f;
    if (MODEL == KGE_TRANSE) {
#pragma unroll
      for (int e = 0; e < E; ++e) {
        const float x = h[0][e] + r[0][e] - t[0][e];
        s += x * x;
      }
      s = -sqrtf(group_sum<G>(s));
    } else if (MODEL == KGE_TORUSE) {   // toruse.py:66-76 (padding lanes hold zeros: min(0, 1) = 0)
#pragma unroll
      for (int e = 0; e < E; ++e) {
        const float x = (fracf_signed(h[0][e]) + fracf_signed(r[0][e])) - fracf_signed(t[0][e]);
        const float x2 = x * x;
        s += fminf(x2, 1.f - x2);
      }
      s = -(4.f * group_sum<G>(s));
    } else if (MODEL == KGE_DISTMULT) {
#pragma unroll
      for (int e = 0; e < E; ++e) s += h[0][e] * r[0][e] * t[0][e];
      s = group_sum<G>(s);
    } else if (MODEL == KGE_ROTATE) {
#pragma unroll
      for (int e = 0; e < E; ++e) {
        float sn, cs;
        sincosf(r[0][e], &sn, &cs);
        const float re = (cs * h[0][e] - sn * h[1][e]) - t[0][e];
        const float im = (cs * h[1][e] + sn * h[0][e]) - t[1][e];
        s += re * re + im * im;
      }
      s = a.m.margin - sqrtf(group_sum<G>(s));
    } else {
#pragma unroll
      for (int e = 0; e < E; ++e) {
        const float A_ = h[0][e] * r[0][e];
        const float B_ = h[1][e] * r[0][e] + h[0][e] * r[1][e] - h[1][e] * r[1][e];
        s += t[0][e] * A_ + t[1][e] * B_;
      }
      s = group_sum<G>(s);
    }
    if (gl == 0) out[i] = s;
  }
}

// ---- TransD projection: out[i] = E[id_i] + RP[rel_i] * <E[id_i], EP[id_i]>  (transd.py:86-91) --------------------
template <int VEC, int G, int NCH>
__global__ void __launch_bounds__(256) transd_project_kernel(const float* __restrict__ emb, const float* __restrict__ vec,
                                                             const int64_t* __restrict__ ids, int64_t n, int d,
                                                             const float* __restrict__ rel_vec,
                                                             const int64_t* __restrict__ rel_ids, int64_t rel_row,
                                                             float* __restrict__ out) {
  constexpr int E = VEC * NCH;
  const int gl = (threadIdx.x & 31) % G;
  const int groups_per_cta = blockDim.x / G;
  const int64_t n_groups = (int64_t)gridDim.x * groups_per_cta;
  for (int64_t i = (int64_t)blockIdx.x * groups_per_cta + threadIdx.x / G; i < n; i += n_groups) {
    const int64_t row = ids ? __ldg(ids + i) : i;
    const int64_t rr = rel_ids ? __ldg(rel_ids + i) : rel_row;
    float e0[E], e1[E], rp[E];
    frag_load<VEC, G, NCH>(emb, row, d, gl, e0);
    frag_load<VEC, G, NCH>(vec, row, d, gl, e1);
    frag_load<VEC, G, NCH>(rel_vec, rr, d, gl, rp);
    float s = 0.f;
#pragma unroll
    for (int e = 0; e < E; ++e) s = __fmaf_rn(e0[e], e1[e], s);
    s = group_sum<G>(s);
#pragma unroll
    for (int e = 0; e < E; ++e) e0[e] = __fmaf_rn(rp[e], s, e0[e]);
    frag_store<VEC, G, NCH>(out, i, d, gl, e0);
  }
}

// ---- TransH projection: out[i] = E[id_i] * (1 - sum(w) * w), w = W[rel_i]  (transh.py:73-74) ---------------------
template <int VEC, int G, int NCH>
__global__ void __launch_bounds__(256) transh_project_kernel(const float* __restrict__ emb, const int64_t* __restrict__ ids,
                                                             int64_t n, int d, const float* __restrict__ norm_vec,
                                                             const int64_t* __restrict__ rel_ids, int64_t rel_row,
                                                             float* __restrict__ out) {
  constexpr int E = VEC * NCH;
  const int gl = (threadIdx.x & 31) % G;
  const int groups_per_cta = blockDim.x / G;
  const int64_t n_groups = (int64_t)gridDim.x * groups_per_cta;
  for (int64_t i = (int64_t)blockIdx.x * groups_per_cta + threadIdx.x / G; i < n; i += n_groups) {
    const int64_t row = ids ? __ldg(ids + i) : i;
    const int64_t rr = rel_ids ? __ldg(rel_ids + i) : rel_row;
    float e0[E], w[E];
    frag_load<VEC, G, NCH>(emb, row, d, gl, e0);
    frag_load<VEC, G, NCH>(norm_vec, rr, d, gl, w);
    float s = 0.f;
#pragma unroll
    for (int e = 0; e < E; ++e) s += w[e];
    s = group_sum<G>(s);
#pragma unroll
    for (int e = 0; e < E; ++e) e0[e] *= __fsub_rn(1.f, __fmul_rn(s, w[e]));
    frag_store<VEC, G, NCH>(out, i, d, gl, e0);
  }
}

// ---- the tile kernel ---------------------------------------------------------------------------
struct TileArgs {
  ScoreArgs s;
  int64_t n_targets;
  int kpad;            // padded floats per part = ceil(d / KC) * KC
  int tiles_per_split; // target tiles handled by one blockIdx.y
  // dense epilogue
  float* out;
  // top-k epilogue
  const int64_t* hist_off;
  const int64_t* hist_items;
  int mask_first;
  int k;
  uint64_t* part_keys;  // [n, n_splits, k]; large k: [n, n_splits, buf_cap]
  int n_splits;
  // Indirect rows (the tensor-core path's device-side fallback): the CTA works on entries [row_begin, min(*row_count,
  // row_end)) of row_map instead of rows [0, n); the row count is only known on the device, so the grid is sized for
  // a capacity, CTAs beyond the count leave at once and the others stride over the row blocks.  part_keys is
  // indexed by (entry - row_begin).
  const int32_t* row_map;
  const int32_t* row_count;
  int64_t row_begin, row_end;
  // rank epilogue (see rank_thresholds_kernel): the positives CSR, their scores sorted per row and the counters
  const int64_t* pos_off;
  const float* rank_thr;       // [n_pos] sorted ascending inside every row
  const float* rank_lo;        // [n] lowest finite threshold of the row (+inf: none)
  uint64_t* rank_bins;         // [2 * n_pos]
  uint64_t* rank_unmasked;     // [n]
  uint64_t* rank_ninf;         // [n]
  int64_t rank_cap;            // positives the workspace holds
  // large-k epilogue: keys one (row, split) buffer of part_keys holds (>= k + BT)
  int64_t buf_cap;
};

// Epilogue of the tile kernel: the dense scores, the per-row top-k, or the rank counts of listed targets.
// EPI_TOPK_LARGE is the top-k for k > KMAX (see large_k_cap).
constexpr int EPI_DENSE = 0, EPI_TOPK = 1, EPI_RANK = 2, EPI_TOPK_LARGE = 3;
constexpr int RANK_SM = 16;   // thresholds a row keeps in shared memory; rows with more count in global memory

// ---- large-k top-k (k > KMAX) -----------------------------------------------------------------------------------
// A sorted list of k keys per row no longer fits shared memory, so each (row, split) appends the keys that beat the
// row's threshold to a buffer of buf_cap = large_k_cap(k) keys in the workspace.  When a tile's keys would overflow
// it, the buffer is compacted to exactly its top k (keys are unique: the id is part of the key) and the threshold
// rises to the k-th key.  A merge kernel then selects each row's top k over its splits and sorts them.
__host__ __device__ __forceinline__ int64_t large_k_cap(int64_t k) { return (2 * k + 31) / 32 * 32; }   // >= k + BT

__device__ __forceinline__ uint64_t warp_min_u64(uint64_t x) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) x = min(x, (uint64_t)__shfl_xor_sync(0xffffffffu, x, o));
  return x;
}
__device__ __forceinline__ int64_t warp_sum_i64(int64_t x) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
  return x;
}

// The k-th largest non-zero key among keys[s * stride + i] (s < nseg, i < len), or 0 when fewer than k are non-zero;
// every lane of the warp returns it.  mma_topk.cu's warp_kth_largest on 64-bit keys in memory: the radix descent
// starts at the highest bit in which the keys differ and stops as soon as exactly k keys remain above the prefix.
__device__ __forceinline__ uint64_t warp_kth_largest_mem(const uint64_t* keys, int64_t nseg, int64_t len, int64_t stride,
                                                      int64_t k) {
  const int lane = threadIdx.x & 31;
  int64_t n_t = 0;
  uint64_t k_or = 0ull, k_and = ~0ull;
  for (int64_t s = 0; s < nseg; ++s)
    for (int64_t i = lane; i < len; i += 32) {
      const uint64_t x = keys[s * stride + i];
      if (x) {
        ++n_t;
        k_or |= x;
        k_and &= x;
      }
    }
  n_t = warp_sum_i64(n_t);
  if (n_t < k) return 0ull;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    k_or |= (uint64_t)__shfl_xor_sync(0xffffffffu, k_or, o);
    k_and &= (uint64_t)__shfl_xor_sync(0xffffffffu, k_and, o);
  }
  const uint64_t diff = k_or ^ k_and;
  if (diff == 0ull) return k_or;   // one key
  const int top = 63 - __clzll((long long)diff);
  uint64_t P = top == 63 ? 0ull : (k_and & ~((2ull << top) - 1ull));   // invariant: #(key >= max(P, 1)) = n_t >= k
  for (int bit = top; bit >= 0 && n_t > k; --bit) {
    const uint64_t c = P | (1ull << bit);
    int64_t n = 0;
    for (int64_t s = 0; s < nseg; ++s)
      for (int64_t i = lane; i < len; i += 32) n += keys[s * stride + i] >= c;
    n = warp_sum_i64(n);
    if (n >= k) {
      P = c;
      n_t = n;
    }
  }
  const uint64_t T = P ? P : 1ull;
  uint64_t mn = ~0ull;
  for (int64_t s = 0; s < nseg; ++s)
    for (int64_t i = lane; i < len; i += 32) {
      const uint64_t x = keys[s * stride + i];
      if (x >= T) mn = min(mn, x);
    }
  return warp_min_u64(mn);
}

// Keep the keys >= T (T > 0) of buf[0, len), in order, in place; returns the new length (lane-uniform).  Writes never
// overtake reads: a key moves to a position at or below its own, and the ballot orders a round's reads before its
// writes.
__device__ __forceinline__ int warp_keep_at_least(uint64_t* buf, int len, uint64_t T) {
  const int lane = threadIdx.x & 31;
  int w = 0;
  for (int base = 0; base < len; base += 32) {
    const int i = base + lane;
    const uint64_t x = i < len ? buf[i] : 0ull;
    const bool keep = x >= T;
    const unsigned b = __ballot_sync(0xffffffffu, keep);
    if (keep) buf[w + __popc(b & ((1u << lane) - 1u))] = x;
    w += __popc(b);
  }
  __syncwarp();
  return w;
}

// Sort buf[0, P) descending with the whole block (bitonic network; P a power of two).
__device__ __forceinline__ void block_bitonic_sort_desc(uint64_t* buf, int64_t P) {
  for (int64_t size = 2; size <= P; size <<= 1)
    for (int64_t stride = size >> 1; stride > 0; stride >>= 1) {
      for (int64_t i = threadIdx.x; i < P / 2; i += blockDim.x) {
        const int64_t lo = 2 * i - (i & (stride - 1)), hi = lo + stride;
        const uint64_t x = buf[lo], y = buf[hi];
        if ((lo & size) == 0 ? x < y : x > y) {
          buf[lo] = y;
          buf[hi] = x;
        }
      }
      __syncthreads();
    }
}

template <int BU>
__device__ __forceinline__ void build_queries(const ScoreArgs& a, const int64_t* rowid, int nrows, int kpad, float* Qs) {
  const int d = a.m.d;
  const int parts = (a.m.model == KGE_ROTATE || a.m.model == KGE_COMPLEX) ? 2 : 1;
  const int qstride = parts * kpad;
  for (int idx = threadIdx.x; idx < BU * kpad; idx += blockDim.x) {
    const int u = idx / kpad, c = idx - u * kpad;
    float q0 = 0.f, q1 = 0.f;
    if (u < nrows && c < d) query_value(a, rowid[u], c, q0, q1);
    Qs[u * qstride + c] = q0;
    if (parts == 2) Qs[u * qstride + kpad + c] = q1;
  }
}

// Stage target rows [t0, t0+BT) x columns [c0, c0+KC) of one part into Ts (zero padded).
template <bool FRAC>
__device__ __forceinline__ void load_target_chunk(const float* __restrict__ W, int d, int64_t n_targets, int64_t t0,
                                                  int c0, float* Ts) {
  if ((d & 3) == 0) {
    // 8 float4 per row chunk; consecutive lanes take consecutive rows -> conflict-free STS.128
    for (int idx = threadIdx.x; idx < BT * (KC / 4); idx += blockDim.x) {
      const int q = idx / BT, j = idx - q * BT;
      const int c = c0 + q * 4;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      const int64_t t = t0 + j;
      if (t < n_targets && c < d) v = __ldg(reinterpret_cast<const float4*>(W + t * d + c));
      if (FRAC) v = make_float4(fracf_signed(v.x), fracf_signed(v.y), fracf_signed(v.z), fracf_signed(v.w));
      *reinterpret_cast<float4*>(Ts + j * TS + q * 4) = v;
    }
  } else {
    for (int idx = threadIdx.x; idx < BT * KC; idx += blockDim.x) {
      const int j = idx / KC, q = idx - j * KC;
      const int c = c0 + q;
      const int64_t t = t0 + j;
      const float v = (t < n_targets && c < d) ? __ldg(W + t * d + c) : 0.f;
      Ts[j * TS + q] = FRAC ? fracf_signed(v) : v;
    }
  }
}

// MODE: how a (query, target) pair of rows is contracted (score_common.cuh).  EPI: what the sweep does with the scores.
// The rank epilogue asks for two CTAs per SM (128 registers): under the compiler's default budget it spills.
// BU: query rows per CTA (plan_tiles); warp w owns rows RU*w .. RU*w + RU-1 of the block.
template <int MODE, int EPI, int BU>
__global__ void __launch_bounds__(TILE_THREADS, (EPI == EPI_RANK || EPI == EPI_TOPK_LARGE) ? 2 : 0) fullsort_tile_kernel(const TileArgs a) {
  constexpr bool DIST = MODE == MODE_DIST;
  constexpr bool TOPK = EPI == EPI_TOPK, RANK = EPI == EPI_RANK, LARGE = EPI == EPI_TOPK_LARGE;
  constexpr bool SEL = TOPK || LARGE;         // a top-k epilogue: candidate keys staged per tile
  constexpr bool MASKED = EPI != EPI_DENSE;   // the trainer's masking: column 0 and the history -> -inf
  constexpr int RU = BU / (TILE_THREADS / 32);   // query rows of a thread's register block
  static_assert(BU == 32 || BU == 16, "query blocks of 32 or 16 rows");
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int model = a.s.m.model;
  const int parts = (model == KGE_ROTATE || model == KGE_COMPLEX) ? 2 : 1;
  const int d = a.s.m.d;
  const int kpad = a.kpad;
  const int qstride = parts * kpad;
  const int k = a.k;

  float* Qs = reinterpret_cast<float*>(smem_raw);  // [BU][qstride]
  float* Ts = Qs + BU * qstride;                   // [BT][TS]
  // top-k only
  uint64_t* lists = reinterpret_cast<uint64_t*>(Ts + BT * TS);  // [BU][k]
  uint64_t* cand = lists + (TOPK ? BU * k : 0);                 // [BU][BT]
  uint64_t* thr = cand + (SEL ? BU * BT : 0);                   // [BU]
  uint32_t* maskbits = reinterpret_cast<uint32_t*>(thr + (SEL ? BU : 0));  // [BU][BT/32] (top-k and rank)
  int* cnt = reinterpret_cast<int*>(maskbits + (MASKED ? BU * (BT / 32) : 0));  // [BU]
  int* llen = cnt + (SEL ? BU : 0);                                         // [BU] list / buffer length
  int64_t* cursor = reinterpret_cast<int64_t*>(llen + (SEL ? BU : 0));      // [BU] (8-byte aligned by layout)
  int64_t* rowid = cursor + (MASKED ? BU : 0);                              // [BU] query row of each slot
  // rank only
  int64_t* rbase = rowid + BU;                                              // [BU] pos_off of the row
  float* rthr = reinterpret_cast<float*>(rbase + (RANK ? BU : 0));         // [BU][RANK_SM] sorted thresholds
  uint32_t* rcnt = reinterpret_cast<uint32_t*>(rthr + (RANK ? BU * RANK_SM : 0));  // [BU][2 * RANK_SM] bins
  float* rlo = reinterpret_cast<float*>(rcnt + (RANK ? BU * 2 * RANK_SM : 0));    // [BU] lowest finite threshold
  int* rm = reinterpret_cast<int*>(rlo + (RANK ? BU : 0));                        // [BU] thresholds of the row
  if (RANK && a.pos_off[a.s.n] > a.rank_cap) return;   // (the workspace was sized for fewer positives)

  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int tu = warp;  // users RU*tu .. RU*tu+RU-1

  const int64_t n_tiles = (a.n_targets + BT - 1) / BT;
  const int64_t tile_lo = (int64_t)blockIdx.y * a.tiles_per_split;
  const int64_t tile_hi = min(n_tiles, tile_lo + a.tiles_per_split);
  const int64_t row_stop = a.row_map ? min((int64_t)__ldg(a.row_count), a.row_end) : a.s.n;

  for (int64_t row0 = a.row_begin + (int64_t)blockIdx.x * BU; row0 < row_stop; row0 += (int64_t)gridDim.x * BU) {
  const int nrows = (int)min((int64_t)BU, row_stop - row0);
  __syncthreads();   // (indirect rows: the previous row block of this CTA is done with shared memory)
  for (int u = threadIdx.x; u < BU; u += blockDim.x)
    rowid[u] = u < nrows ? (a.row_map ? (int64_t)__ldg(a.row_map + row0 + u) : row0 + u) : 0;
  __syncthreads();
  build_queries<BU>(a.s, rowid, nrows, kpad, Qs);
  if (RANK) {
    for (int u = threadIdx.x; u < BU; u += blockDim.x) {
      int64_t base = 0, m = 0;
      float lo = INFINITY;
      if (u < nrows) {
        base = a.pos_off[rowid[u]];
        m = a.pos_off[rowid[u] + 1] - base;
        lo = a.rank_lo[rowid[u]];
      }
      rbase[u] = base;
      rm[u] = (int)min(m, (int64_t)0x7fffffff);
      rlo[u] = lo;
      if (m <= RANK_SM) {
        for (int i = 0; i < m; ++i) rthr[u * RANK_SM + i] = a.rank_thr[base + i];
        for (int i = 0; i < 2 * RANK_SM; ++i) rcnt[u * 2 * RANK_SM + i] = 0u;
      }
    }
  }
  // unmasked targets and targets scoring -inf of the thread's RU rows (rank epilogue)
  uint32_t n_unm[RU] = {}, n_ninf[RU] = {};
  if (MASKED) {
    for (int u = threadIdx.x; u < BU; u += blockDim.x) {
      if (SEL) {
        thr[u] = 0ull;
        llen[u] = 0;
        cnt[u] = 0;
      }
      int64_t cur = 0;
      if (u < nrows && a.hist_off) {
        // first history entry >= tile_lo * BT (history sorted ascending per row)
        int64_t lo = a.hist_off[rowid[u]], hi = a.hist_off[rowid[u] + 1];
        const int64_t first = tile_lo * BT;
        while (lo < hi) {
          const int64_t mid = (lo + hi) >> 1;
          if (a.hist_items[mid] < first) lo = mid + 1; else hi = mid;
        }
        cur = lo;
      }
      cursor[u] = cur;
    }
  }
  __syncthreads();

  for (int64_t tile = tile_lo; tile < tile_hi; ++tile) {
    const int64_t t0 = tile * BT;
    float acc[RU][4];
#pragma unroll
    for (int x = 0; x < RU; ++x)
#pragma unroll
      for (int y = 0; y < 4; ++y) acc[x][y] = 0.f;

    if (MASKED) {
      // history bits of this tile
      for (int i = threadIdx.x; i < BU * (BT / 32); i += blockDim.x) maskbits[i] = 0u;
      __syncthreads();
      if (a.hist_off) {
        for (int u = warp; u < nrows; u += TILE_THREADS / 32) {
          const int64_t end = a.hist_off[rowid[u] + 1];
          int64_t cur = cursor[u];
          const int64_t limit = t0 + BT;
          while (true) {
            const int64_t idx = cur + lane;
            int64_t item = limit;
            if (idx < end) item = a.hist_items[idx];
            const bool in = item < limit;
            if (in && item >= t0) {
              const int off = (int)(item - t0);
              atomicOr(&maskbits[u * (BT / 32) + (off >> 5)], 1u << (off & 31));
            }
            const unsigned b = __ballot_sync(0xffffffffu, in);
            cur += __popc(b);
            if (b != 0xffffffffu) break;
          }
          if (lane == 0) cursor[u] = cur;
        }
      }
    }

    for (int p = 0; p < parts; ++p) {
      const float* W = a.s.m.entity.w[p];
      for (int c0 = 0; c0 < kpad; c0 += KC) {
        __syncthreads();  // previous chunk consumed
        load_target_chunk<MODE == MODE_TORUS>(W, d, a.n_targets, t0, c0, Ts);
        __syncthreads();
        const float* qbase = Qs + (RU * tu) * qstride + p * kpad + c0;
#pragma unroll
        for (int kk = 0; kk < KC; kk += 4) {
          float4 qv[RU], tv[4];
#pragma unroll
          for (int x = 0; x < RU; ++x) qv[x] = *reinterpret_cast<const float4*>(qbase + x * qstride + kk);
#pragma unroll
          for (int y = 0; y < 4; ++y) tv[y] = *reinterpret_cast<const float4*>(Ts + (lane + 32 * y) * TS + kk);
#pragma unroll
          for (int x = 0; x < RU; ++x)
#pragma unroll
            for (int y = 0; y < 4; ++y) {
              if (DIST) {
                const float e0 = qv[x].x - tv[y].x, e1 = qv[x].y - tv[y].y;
                const float e2 = qv[x].z - tv[y].z, e3 = qv[x].w - tv[y].w;
                acc[x][y] = fmaf(e0, e0, acc[x][y]);
                acc[x][y] = fmaf(e1, e1, acc[x][y]);
                acc[x][y] = fmaf(e2, e2, acc[x][y]);
                acc[x][y] = fmaf(e3, e3, acc[x][y]);
              } else if (MODE == MODE_TORUS) {
                const float e0 = qv[x].x - tv[y].x, e1 = qv[x].y - tv[y].y;
                const float e2 = qv[x].z - tv[y].z, e3 = qv[x].w - tv[y].w;
                const float s0 = e0 * e0, s1 = e1 * e1, s2 = e2 * e2, s3 = e3 * e3;
                acc[x][y] += fminf(s0, 1.f - s0);
                acc[x][y] += fminf(s1, 1.f - s1);
                acc[x][y] += fminf(s2, 1.f - s2);
                acc[x][y] += fminf(s3, 1.f - s3);
              } else {
                acc[x][y] = fmaf(qv[x].x, tv[y].x, acc[x][y]);
                acc[x][y] = fmaf(qv[x].y, tv[y].y, acc[x][y]);
                acc[x][y] = fmaf(qv[x].z, tv[y].z, acc[x][y]);
                acc[x][y] = fmaf(qv[x].w, tv[y].w, acc[x][y]);
              }
            }
        }
      }
    }

    // ---- epilogue of this tile ------------------------------------------------------------
    const float margin = (model == KGE_ROTATE) ? a.s.m.margin : 0.f;
#pragma unroll
    for (int x = 0; x < RU; ++x) {
      const int u = RU * tu + x;
      if (u >= nrows) continue;
#pragma unroll
      for (int y = 0; y < 4; ++y) {
        const int jo = lane + 32 * y;
        const int64_t j = t0 + jo;
        if (j >= a.n_targets) continue;
        float sc = DIST ? (margin - sqrtf(acc[x][y])) : (MODE == MODE_TORUS ? -(4.f * acc[x][y]) : acc[x][y]);
        if (!MASKED) {
          a.out[rowid[u] * a.n_targets + j] = sc;
          continue;
        }
        const bool masked = (a.mask_first && j == 0) || ((maskbits[u * (BT / 32) + (jo >> 5)] >> (jo & 31)) & 1u);
        if (masked) sc = -INFINITY;
        if (SEL) {
          const uint64_t key = make_key(sc, (uint32_t)j);
          if (key > thr[u]) {
            const int slot = atomicAdd(&cnt[u], 1);
            cand[u * BT + slot] = key;
          }
        } else {
          n_unm[x] += masked ? 0u : 1u;
          if (sc == -INFINITY) {
            ++n_ninf[x];
          } else if (sc >= rlo[u]) {
            // Most targets score below the row's lowest positive and stop at the compare above.  The others are
            // binned against the sorted thresholds w[0, m): with L = #{w < sc}, bin 2L counts scores equal to w[L]
            // and bin 2L - 1 the scores strictly between w[L - 1] and w[L] (or above w[m - 1] when L = m).
            const int m = rm[u];
            if (m <= RANK_SM) {
              const float* w = rthr + u * RANK_SM;
              int lo = 0, hi = m;
              while (lo < hi) {
                const int mid = (lo + hi) >> 1;
                if (w[mid] < sc) lo = mid + 1; else hi = mid;
              }
              atomicAdd(&rcnt[u * 2 * RANK_SM + ((lo < m && w[lo] == sc) ? 2 * lo : 2 * lo - 1)], 1u);
            } else {
              const int64_t base = rbase[u];
              const int64_t mm = a.pos_off[rowid[u] + 1] - base;
              const float* w = a.rank_thr + base;
              int64_t lo = 0, hi = mm;
              while (lo < hi) {
                const int64_t mid = (lo + hi) >> 1;
                if (w[mid] < sc) lo = mid + 1; else hi = mid;
              }
              atomicAdd(reinterpret_cast<unsigned long long*>(a.rank_bins + 2 * base +
                                                              ((lo < mm && w[lo] == sc) ? 2 * lo : 2 * lo - 1)),
                        1ull);
            }
          }
        }
      }
    }
    if (TOPK) {
      __syncthreads();
      for (int u = warp; u < nrows; u += TILE_THREADS / 32) {
        const int c = cnt[u];
        if (c == 0) continue;
        int len = llen[u];
        uint64_t* list = lists + u * k;
        for (int i = 0; i < c; ++i) warp_insert(list, len, k, cand[u * BT + i], lane);
        if (lane == 0) {
          llen[u] = len;
          cnt[u] = 0;
          thr[u] = (len == k) ? list[k - 1] : 0ull;
        }
      }
      // the next tile's first __syncthreads orders these writes before its reads
    }
    if (LARGE) {
      __syncthreads();
      for (int u = warp; u < nrows; u += TILE_THREADS / 32) {
        const int c = cnt[u];
        if (c == 0) continue;
        int len = llen[u];
        uint64_t t = thr[u];
        uint64_t* buf = a.part_keys + ((row0 + u) * a.n_splits + blockIdx.y) * a.buf_cap;
        if (len + c > a.buf_cap) {   // len > k: keep exactly the top k, whose last key becomes the threshold
          t = warp_kth_largest_mem(buf, 1, len, 0, k);
          len = warp_keep_at_least(buf, len, t);
        }
        for (int base = 0; base < c; base += 32) {
          const uint64_t key = base + lane < c ? cand[u * BT + base + lane] : 0ull;
          const bool keep = key > t;
          const unsigned b = __ballot_sync(0xffffffffu, keep);
          if (keep) buf[len + __popc(b & ((1u << lane) - 1u))] = key;
          len += __popc(b);
        }
        __syncwarp();
        if (lane == 0) {
          llen[u] = len;
          cnt[u] = 0;
          thr[u] = t;
        }
      }
    }
    if (RANK) __syncthreads();   // every warp is done with this tile's history bits before they are cleared
  }

  if (TOPK) {
    __syncthreads();
    for (int idx = threadIdx.x; idx < nrows * k; idx += blockDim.x) {
      const int u = idx / k, i = idx - u * k;
      const uint64_t key = (i < llen[u]) ? lists[u * k + i] : 0ull;
      a.part_keys[((row0 - a.row_begin + u) * a.n_splits + blockIdx.y) * k + i] = key;
    }
  }
  if (LARGE) {
    // each split leaves its top min(k, len) keys in the first k slots of its buffer, zero-padded
    __syncthreads();
    for (int u = warp; u < nrows; u += TILE_THREADS / 32) {
      int len = llen[u];
      uint64_t* buf = a.part_keys + ((row0 + u) * a.n_splits + blockIdx.y) * a.buf_cap;
      if (len > k) len = warp_keep_at_least(buf, len, warp_kth_largest_mem(buf, 1, len, 0, k));
      for (int i = len + lane; i < k; i += 32) buf[i] = 0ull;
    }
  }
  if (RANK) {
    // this split's counts, added exactly (integer atomics: the result does not depend on the order)
#pragma unroll
    for (int x = 0; x < RU; ++x) {
      const int u = RU * tu + x;
      const unsigned unm = __reduce_add_sync(0xffffffffu, n_unm[x]);
      const unsigned ninf = __reduce_add_sync(0xffffffffu, n_ninf[x]);
      if (lane == 0 && u < nrows) {
        atomicAdd(reinterpret_cast<unsigned long long*>(a.rank_unmasked + rowid[u]), (unsigned long long)unm);
        if (ninf) atomicAdd(reinterpret_cast<unsigned long long*>(a.rank_ninf + rowid[u]), (unsigned long long)ninf);
      }
    }
    __syncthreads();
    for (int idx = threadIdx.x; idx < nrows * 2 * RANK_SM; idx += blockDim.x) {
      const int u = idx / (2 * RANK_SM), s = idx - u * (2 * RANK_SM);
      const uint32_t c = rcnt[idx];
      if (rm[u] <= RANK_SM && s < 2 * rm[u] && c)
        atomicAdd(reinterpret_cast<unsigned long long*>(a.rank_bins + 2 * rbase[u] + s), (unsigned long long)c);
    }
  }
  if (!a.row_map) break;   // direct rows: the grid covers every row block
  }
}

// Merge the per-split lists of one row (one warp per row) and decode.
// With row_map: entry e in [row_begin, min(*row_count, row_end)) of the map, lists at (e - row_begin), output row
// row_map[e]; warps stride over the entries (the count is only known on the device).
__global__ void __launch_bounds__(256) topk_merge_kernel(const uint64_t* __restrict__ part_keys, int64_t n,
                                                         int n_splits, int k, int64_t* __restrict__ ids_out,
                                                         float* __restrict__ scores_out,
                                                         const int32_t* __restrict__ row_map,
                                                         const int32_t* __restrict__ row_count, int64_t row_begin,
                                                         int64_t row_end) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  uint64_t* lists = reinterpret_cast<uint64_t*>(smem_raw);  // [warps][k]
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t stop = row_map ? min((int64_t)__ldg(row_count), row_end) : n;
  const int64_t stride = row_map ? (int64_t)gridDim.x * (blockDim.x >> 5) : stop;   // direct rows: one pass
  for (int64_t ent = row_begin + (int64_t)blockIdx.x * (blockDim.x >> 5) + warp; ent < stop; ent += stride) {
  const int64_t row = row_map ? (int64_t)__ldg(row_map + ent) : ent;
  uint64_t* list = lists + warp * k;
  int len = 0;
  const uint64_t* src = part_keys + (ent - row_begin) * (int64_t)n_splits * k;
  if (n_splits == 1) {
    for (int i = lane; i < k; i += 32) list[i] = src[i];
    len = k;
    __syncwarp();
  } else {
    for (int i = 0; i < n_splits * k; ++i) {
      const uint64_t key = src[i];
      if (key != 0ull) warp_insert(list, len, k, key, lane);
    }
    for (int i = len + lane; i < k; i += 32) list[i] = 0ull;
    __syncwarp();
  }
  for (int i = lane; i < k; i += 32) {
    const uint64_t key = list[i];
    ids_out[row * k + i] = key ? key_id(key) : -1;
    if (scores_out) scores_out[row * k + i] = key ? key_score(key) : -INFINITY;
  }
  __syncwarp();
  }
}

// Large-k merge, one CTA per row: warp 0 selects the k-th key T over the row's n_splits zero-padded lists of k keys
// (the row has at least k keys: every split keeps min(k, its targets)), the block gathers the k keys >= T, sorts
// them and decodes.  Up to SORT_SM keys the sort runs in shared memory; above, it runs in the row's own workspace
// (buf_cap >= P keys), with the ids_out row as the staging area of the gather.
constexpr int64_t SORT_SM = 8192;

__global__ void __launch_bounds__(256) topk_merge_large_kernel(uint64_t* __restrict__ part_keys, int n_splits, int k,
                                                               int64_t buf_cap, int64_t P, int64_t* __restrict__ ids_out,
                                                               float* __restrict__ scores_out) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ uint64_t s_T;
  __shared__ int s_n;
  const int64_t row = blockIdx.x;
  uint64_t* region = part_keys + row * n_splits * buf_cap;
  if (threadIdx.x < 32) {
    const uint64_t T = warp_kth_largest_mem(region, n_splits, k, buf_cap, k);
    if (threadIdx.x == 0) {
      s_T = T;
      s_n = 0;
    }
  }
  __syncthreads();
  const uint64_t T = s_T;
  const bool in_sm = P <= SORT_SM;
  uint64_t* stage = in_sm ? reinterpret_cast<uint64_t*>(smem_raw) : reinterpret_cast<uint64_t*>(ids_out + row * k);
  for (int s = 0; s < n_splits; ++s)
    for (int i = threadIdx.x; i < k; i += blockDim.x) {
      const uint64_t x = region[s * buf_cap + i];
      if (x != 0ull && x >= T) {
        const int slot = atomicAdd(&s_n, 1);
        if (slot < k) stage[slot] = x;
      }
    }
  __syncthreads();
  const int64_t m = min(s_n, k);
  uint64_t* buf = in_sm ? stage : region;
  if (!in_sm)
    for (int64_t i = threadIdx.x; i < m; i += blockDim.x) buf[i] = stage[i];
  for (int64_t i = m + threadIdx.x; i < P; i += blockDim.x) buf[i] = 0ull;
  __syncthreads();
  block_bitonic_sort_desc(buf, P);
  for (int64_t i = threadIdx.x; i < k; i += blockDim.x) {
    const uint64_t key = buf[i];
    ids_out[row * k + i] = key ? key_id(key) : -1;
    if (scores_out) scores_out[row * k + i] = key ? key_score(key) : -INFINITY;
  }
}

// ---- collector.py:178-183 without the [n, I] matrix ---------------------------------------------
__global__ void __launch_bounds__(256) topk_hits_kernel(const int64_t* __restrict__ ids, int64_t n, int k,
                                                        const int64_t* __restrict__ pos_off,
                                                        const int64_t* __restrict__ pos_items,
                                                        int32_t* __restrict__ out) {
  const int64_t total = n * (int64_t)(k + 1);
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (int64_t)gridDim.x * blockDim.x) {
    const int64_t u = idx / (k + 1);
    const int i = (int)(idx - u * (k + 1));
    int64_t lo = pos_off[u], hi = pos_off[u + 1];
    if (i == k) {
      out[idx] = (int32_t)(hi - lo);
      continue;
    }
    const int64_t id = ids[u * k + i];
    int hit = 0;
    while (lo < hi) {
      const int64_t mid = (lo + hi) >> 1;
      const int64_t v = pos_items[mid];
      if (v == id) { hit = 1; break; }
      if (v < id) lo = mid + 1; else hi = mid;
    }
    out[idx] = hit;
  }
}

// ---- metrics.py summed over users ---------------------------------------------------------------
// sums[5][k]: recall, mrr, ndcg, hit, precision (the order of overall.yaml's default metrics).
__device__ __forceinline__ double warp_sum_f64(double x) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
  return x;
}

__global__ void __launch_bounds__(256) topk_metric_sums_kernel(const int32_t* __restrict__ rec, int64_t n, int k,
                                                               double* __restrict__ sums) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double* acc = reinterpret_cast<double*>(smem_raw);  // [warps][5*k]
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, warps = blockDim.x >> 5;
  for (int i = threadIdx.x; i < warps * 5 * k; i += blockDim.x) acc[i] = 0.0;
  __syncthreads();
  double* mine = acc + warp * 5 * k;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t base = (int64_t)blockIdx.x * blockDim.x + warp * 32; base < n; base += stride) {
    const int64_t u = base + lane;
    const bool valid = u < n;
    const int32_t* row = rec + (valid ? u : 0) * (int64_t)(k + 1);
    const int pos_len = row[k];
    const int ilen = pos_len < k ? pos_len : k;
    int cum = 0, first = -1;
    double dcg = 0.0, idcg = 0.0;
    for (int j = 0; j < k; ++j) {
      const int hit = row[j] != 0;
      const double disc = 1.0 / log2((double)(j + 2));
      if (hit) {
        if (first < 0) first = j;
        dcg += disc;
      }
      cum += hit;
      if (j < ilen) idcg += disc;  // idcg freezes after min(pos_len, k) terms (metrics.py:191-207)
      double v0 = (double)cum / (double)pos_len;
      double v1 = first >= 0 ? 1.0 / (double)(first + 1) : 0.0;
      double v2 = dcg / idcg;
      double v3 = cum > 0 ? 1.0 : 0.0;
      double v4 = (double)cum / (double)(j + 1);
      if (!valid) v0 = v1 = v2 = v3 = v4 = 0.0;
      v0 = warp_sum_f64(v0);
      v1 = warp_sum_f64(v1);
      v2 = warp_sum_f64(v2);
      v3 = warp_sum_f64(v3);
      v4 = warp_sum_f64(v4);
      if (lane == 0) {
        mine[0 * k + j] += v0;
        mine[1 * k + j] += v1;
        mine[2 * k + j] += v2;
        mine[3 * k + j] += v3;
        mine[4 * k + j] += v4;
      }
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 5 * k; i += blockDim.x) {
    double t = 0.0;
    for (int w = 0; w < warps; ++w) t += acc[w * 5 * k + i];
    atomicAdd(&sums[i], t);
  }
}

// The same sums for k > KMAX, whose per-warp [5][k] accumulators would not fit shared memory: blockIdx.y strides over
// windows of MW cutoffs.  A lane first rebuilds its user's running state (hits, first hit, dcg, idcg) over the columns
// before the window, adding in the same order as the loop above, then accumulates the window as above.
constexpr int MW = 128;

__global__ void __launch_bounds__(256) topk_metric_sums_window_kernel(const int32_t* __restrict__ rec, int64_t n, int k,
                                                                      double* __restrict__ sums) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double* acc = reinterpret_cast<double*>(smem_raw);  // [warps][5*MW]
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, warps = blockDim.x >> 5;
  double* mine = acc + warp * 5 * MW;
  const int n_win = (k + MW - 1) / MW;
  for (int win = blockIdx.y; win < n_win; win += gridDim.y) {
    const int j0 = win * MW, j1 = min(k, j0 + MW);
    __syncthreads();   // (the previous window's flush is done)
    for (int i = threadIdx.x; i < warps * 5 * MW; i += blockDim.x) acc[i] = 0.0;
    __syncthreads();
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t base = (int64_t)blockIdx.x * blockDim.x + warp * 32; base < n; base += stride) {
      const int64_t u = base + lane;
      const bool valid = u < n;
      const int32_t* row = rec + (valid ? u : 0) * (int64_t)(k + 1);
      const int pos_len = row[k];
      const int ilen = pos_len < k ? pos_len : k;
      int cum = 0, first = -1;
      double dcg = 0.0, idcg = 0.0;
      for (int j = 0; j < j0; ++j) {
        if (row[j] != 0) {
          if (first < 0) first = j;
          dcg += 1.0 / log2((double)(j + 2));
          ++cum;
        }
      }
      for (int j = 0; j < min(ilen, j0); ++j) idcg += 1.0 / log2((double)(j + 2));
      for (int j = j0; j < j1; ++j) {
        const int hit = row[j] != 0;
        const double disc = 1.0 / log2((double)(j + 2));
        if (hit) {
          if (first < 0) first = j;
          dcg += disc;
        }
        cum += hit;
        if (j < ilen) idcg += disc;
        double v0 = (double)cum / (double)pos_len;
        double v1 = first >= 0 ? 1.0 / (double)(first + 1) : 0.0;
        double v2 = dcg / idcg;
        double v3 = cum > 0 ? 1.0 : 0.0;
        double v4 = (double)cum / (double)(j + 1);
        if (!valid) v0 = v1 = v2 = v3 = v4 = 0.0;
        v0 = warp_sum_f64(v0);
        v1 = warp_sum_f64(v1);
        v2 = warp_sum_f64(v2);
        v3 = warp_sum_f64(v3);
        v4 = warp_sum_f64(v4);
        if (lane == 0) {
          const int jj = j - j0;
          mine[0 * MW + jj] += v0;
          mine[1 * MW + jj] += v1;
          mine[2 * MW + jj] += v2;
          mine[3 * MW + jj] += v3;
          mine[4 * MW + jj] += v4;
        }
      }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < 5 * MW; i += blockDim.x) {
      const int c = i / MW, jj = i - c * MW;
      if (j0 + jj >= j1) continue;
      double t = 0.0;
      for (int w = 0; w < warps; ++w) t += acc[w * 5 * MW + i];
      atomicAdd(&sums[(int64_t)c * k + j0 + jj], t);
    }
  }
}

// ---- rank counts of listed targets (collector.py's rec.meanrank without the sorted [n, I] matrix) -------------------
// Three launches: rank_thresholds_kernel scores every (row, positive) pair and sorts those scores per row, the tile
// kernel's rank epilogue counts the targets against them during the sweep, rank_finalize_kernel turns the counts into
// (greater, equal) per positive.
struct RankPrep {
  ScoreArgs s;
  int64_t n_targets;
  const int64_t* hist_off;
  const int64_t* hist_items;
  int mask_first;
  const int64_t* pos_off;
  const int64_t* pos_items;
  int64_t cap;      // entries the workspace holds
  float* score;     // [n_pos] the positive's masked score
  float* sorted;    // [n_pos] the row's scores, ascending
  int64_t* first;   // [n_pos] #{entries of the row scoring below this one} = first sorted position of its value
  float* lo;        // [n] lowest finite score among the row's positives (+inf: none)
};

// One warp per row.  The positives are scored with exact_chain, the tile kernel's own sequence of fp32 operations, so
// that every unmasked positive ties with itself in the sweep.  A masked positive (column 0 with mask_first, an id in
// the row's history, or an id outside [0, n_targets), which is not a target) scores -inf.  The row's scores are then
// placed by counting: position = #{smaller} + #{equal and listed earlier}.  That is quadratic in the row's positives,
// which is cheap for evaluation's few positives per user and stays correct for any number.
template <int MODE>
__global__ void __launch_bounds__(TILE_THREADS) rank_thresholds_kernel(const RankPrep a) {
  constexpr bool DIST = MODE == MODE_DIST;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int parts = (a.s.m.model == KGE_ROTATE || a.s.m.model == KGE_COMPLEX) ? 2 : 1;
  const int d = a.s.m.d;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, warps = TILE_THREADS / 32;
  float* q = reinterpret_cast<float*>(smem_raw) + warp * parts * d;   // [parts * d] this warp's query row
  if (a.pos_off[a.s.n] > a.cap) return;                                // (the workspace was sized for fewer positives)
  const float margin = (a.s.m.model == KGE_ROTATE) ? a.s.m.margin : 0.f;
  for (int64_t row = (int64_t)blockIdx.x * warps + warp; row < a.s.n; row += (int64_t)gridDim.x * warps) {
    for (int c = lane; c < d; c += 32) {
      float q0, q1;
      query_value(a.s, row, c, q0, q1);
      q[c] = q0;
      if (parts == 2) q[d + c] = q1;
    }
    __syncwarp();
    const int64_t p0 = a.pos_off[row], p1 = a.pos_off[row + 1];
    const int64_t h0 = a.hist_off ? a.hist_off[row] : 0, h1 = a.hist_off ? a.hist_off[row + 1] : 0;
    float lo = INFINITY;
    for (int64_t i = p0 + lane; i < p1; i += 32) {
      const int64_t j = a.pos_items[i];
      bool masked = j < 0 || j >= a.n_targets || (a.mask_first && j == 0);
      if (!masked && h1 > h0) {
        int64_t l = h0, h = h1;
        while (l < h) {
          const int64_t mid = (l + h) >> 1;
          if (a.hist_items[mid] < j) l = mid + 1; else h = mid;
        }
        masked = l < h1 && a.hist_items[l] == j;
      }
      float sc = -INFINITY;
      if (!masked) {
        float acc = 0.f;
        for (int p = 0; p < parts; ++p) acc = exact_chain<MODE>(q + p * d, a.s.m.entity.w[p] + j * d, d, acc);
        sc = DIST ? (margin - sqrtf(acc)) : (MODE == MODE_TORUS ? -(4.f * acc) : acc);
        lo = fminf(lo, sc);
      }
      a.score[i] = sc;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) lo = fminf(lo, __shfl_xor_sync(0xffffffffu, lo, o));
    __syncwarp();   // the row's scores are visible to the whole warp
    for (int64_t i = p0 + lane; i < p1; i += 32) {
      const float s = a.score[i];
      int64_t less = 0, before = 0;
      for (int64_t x = p0; x < p1; ++x) {
        const float v = a.score[x];
        less += v < s;
        before += (v == s) && (x < i);
      }
      a.sorted[p0 + less + before] = s;
      a.first[i] = less;
    }
    if (lane == 0) a.lo[row] = lo;
    __syncwarp();   // q is rewritten for the next row
  }
}

// One warp per row: suffix sums over the row's 2m bins (in place), then per positive
//   greater = #{targets scoring above} = the bins above its value's equal bin, equal = that bin;
// a positive scoring -inf ties with every target scoring -inf (masked ones included) and trails all the others.
__global__ void __launch_bounds__(256) rank_finalize_kernel(int64_t n, int64_t n_targets, int64_t cap,
                                                            const int64_t* __restrict__ pos_off,
                                                            const float* __restrict__ score,
                                                            const int64_t* __restrict__ first, uint64_t* bins,
                                                            const uint64_t* __restrict__ ninf,
                                                            int64_t* __restrict__ greater_out,
                                                            int64_t* __restrict__ equal_out,
                                                            int64_t* __restrict__ n_unmasked_out) {
  const int lane = threadIdx.x & 31, warps = blockDim.x >> 5;
  const bool overflow = pos_off[n] > cap;
  for (int64_t row = (int64_t)blockIdx.x * warps + (threadIdx.x >> 5); row < n; row += (int64_t)gridDim.x * warps) {
    if (overflow) {   // nothing was counted: say so in every row instead of returning counts of nothing
      if (lane == 0) n_unmasked_out[row] = -1;
      continue;
    }
    const int64_t p0 = pos_off[row], p1 = pos_off[row + 1];
    const int64_t slots = 2 * (p1 - p0);
    uint64_t* b = bins + 2 * p0;
    uint64_t carry = 0;
    for (int64_t top = slots; top > 0; top -= 32) {   // lane 0 takes the highest slot of each round
      const int64_t s = top - 1 - lane;
      uint64_t v = s >= 0 ? b[s] : 0ull;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const uint64_t y = __shfl_up_sync(0xffffffffu, v, o);
        if (lane >= o) v += y;
      }
      v += carry;
      if (s >= 0) b[s] = v;
      carry = __shfl_sync(0xffffffffu, v, 31);
    }
    __syncwarp();
    const int64_t nf = (int64_t)ninf[row];
    for (int64_t i = p0 + lane; i < p1; i += 32) {
      int64_t gt, eq;
      if (score[i] == -INFINITY) {
        eq = nf;
        gt = n_targets - nf;
      } else {
        const int64_t e = 2 * first[i];
        const uint64_t above = e + 1 < slots ? b[e + 1] : 0ull;
        gt = (int64_t)above;
        eq = (int64_t)(b[e] - above);
      }
      greater_out[i] = gt;
      equal_out[i] = eq;
    }
    __syncwarp();
  }
}

struct RankLayout {
  size_t lo, ninf, score, sorted, first, bins, total;
};

RankLayout rank_layout(int64_t n, int64_t n_pos) {
  auto a16 = [](size_t x) { return (x + 15) / 16 * 16; };
  RankLayout l;
  size_t o = 0;
  l.lo = o;
  o += a16((size_t)n * 4);
  l.ninf = o;
  o += a16((size_t)n * 8);
  l.score = o;
  o += a16((size_t)n_pos * 4);
  l.sorted = o;
  o += a16((size_t)n_pos * 4);
  l.first = o;
  o += a16((size_t)n_pos * 8);
  l.bins = o;
  o += a16((size_t)n_pos * 16);
  l.total = o;
  return l;
}

int check_score_model(const kge_model_t* m) {
  KGE_REQUIRE(m, KGE_E_ARG, "model is NULL");
  KGE_REQUIRE(m->model != KGE_TRANSH, KGE_E_UNSUPPORTED,
              "TransH scores through kge_transh_project and the KGE_TRANSE scoring entry points");
  KGE_REQUIRE(m->model != KGE_TRANSD, KGE_E_UNSUPPORTED,
              "TransD scores through kge_transd_project and the KGE_TRANSE scoring entry points");
  KGE_REQUIRE(m->model >= KGE_TRANSE && m->model <= KGE_TORUSE, KGE_E_ARG, "unknown model kind %d", m->model);
  const int ph = (m->model == KGE_ROTATE || m->model == KGE_COMPLEX) ? 2 : 1;
  const int pr = m->model == KGE_COMPLEX ? 2 : 1;
  for (int p = 0; p < ph; ++p) KGE_REQUIRE(m->user.w[p] && m->entity.w[p], KGE_E_ARG, "NULL weight table");
  for (int p = 0; p < pr; ++p) KGE_REQUIRE(m->relation.w[p], KGE_E_ARG, "NULL relation table");
  KGE_REQUIRE(m->d >= 1 && m->d <= KGE_MAX_D, KGE_E_UNSUPPORTED, "embedding_size %d unsupported (1 to %d)", m->d,
              KGE_MAX_D);
  return 0;
}

struct TilePlan {
  int kpad, bu, n_splits, tiles_per_split;
  size_t smem;
  int64_t n_blocks;
};

// Shared memory of the tile kernel with a query block of BU rows.
size_t tile_smem(int BU, int parts, int kpad, int k, int epi) {
  size_t smem = (size_t)BU * parts * kpad * 4 + (size_t)BT * TS * 4;
  if (epi == EPI_TOPK) smem += (size_t)BU * k * 8 + (size_t)BU * BT * 8 + BU * 8 + BU * (BT / 32) * 4 + BU * 4 * 2 + BU * 8;
  if (epi == EPI_TOPK_LARGE)   // the same without the lists: cand, thr, maskbits, cnt, llen, cursor
    smem += (size_t)BU * BT * 8 + BU * 8 + BU * (BT / 32) * 4 + BU * 4 * 2 + BU * 8;
  if (epi == EPI_RANK)   // maskbits, cursor | rbase, rthr, rcnt, rlo, rm
    smem += BU * (BT / 32) * 4 + BU * 8 + BU * 8 + (size_t)BU * RANK_SM * 4 * 3 + BU * 4 * 2;
  smem += BU * 8;   // rowid
  return smem;
}

int plan_tiles(const kge_model_t* m, int64_t n, int64_t n_targets, int k, int epi, TilePlan& pl) {
  KGE_REQUIRE(m->d >= 1 && m->d <= KGE_MAX_D, KGE_E_UNSUPPORTED, "embedding_size %d unsupported (1 to %d)", m->d,
              KGE_MAX_D);
  const int parts = (m->model == KGE_ROTATE || m->model == KGE_COMPLEX) ? 2 : 1;
  pl.kpad = (m->d + KC - 1) / KC * KC;
  // 32 query rows where they fit; 16 above (the two-part models from d = 545 to 801 on, by epilogue and k).  Sixteen
  // rows need at most 183 KB (parts * kpad = 2,048, k = 128), so no smaller block is needed up to KGE_MAX_D.
  pl.bu = 32;
  if (tile_smem(32, parts, pl.kpad, k, epi) > 220 * 1024) pl.bu = 16;
  const size_t smem = tile_smem(pl.bu, parts, pl.kpad, k, epi);
  pl.smem = smem;
  KGE_REQUIRE(smem <= 220 * 1024, KGE_E_UNSUPPORTED, "embedding_size %d needs %zu bytes of shared memory", m->d, smem);
  pl.n_blocks = (n + pl.bu - 1) / pl.bu;
  const int64_t n_tiles = (n_targets + BT - 1) / BT;
  int splits = 1;
  if (epi != EPI_DENSE) {
    // enough CTAs for two waves at 2 CTAs/SM, but at least 8 tiles per split (large k: and at least k targets, so
    // that the merge does not read many nearly empty lists)
    const int64_t want = (int64_t)kge_num_sms() * 4;
    int64_t s = (want + pl.n_blocks - 1) / pl.n_blocks;
    const int64_t k_tiles = ((int64_t)k + BT - 1) / BT;
    const int64_t min_tiles = (epi == EPI_TOPK_LARGE && k_tiles > 8) ? k_tiles : 8;
    const int64_t max_s = (n_tiles + min_tiles - 1) / min_tiles;
    if (s > max_s) s = max_s;
    if (s < 1) s = 1;
    if (s > 65535) s = 65535;
    splits = (int)s;
  }
  pl.tiles_per_split = (int)((n_tiles + splits - 1) / splits);
  pl.n_splits = (int)((n_tiles + pl.tiles_per_split - 1) / pl.tiles_per_split);
  if (pl.n_splits < 1) pl.n_splits = 1;
  return 0;
}

int tile_mode(int model) {
  if (model == KGE_TORUSE) return MODE_TORUS;
  return (model == KGE_TRANSE || model == KGE_ROTATE) ? MODE_DIST : MODE_DOT;
}

}  // namespace

extern "C" int kge_predict(const kge_model_t* model, const int64_t* heads, const int64_t* rels, const int64_t* tails,
                           int64_t n, int head_is_user, float* out, kge_stream_t stream) {
  if (int e = check_score_model(model)) return e;
  KGE_REQUIRE(n >= 0, KGE_E_ARG, "negative n");
  if (n == 0) return 0;
  KGE_REQUIRE(heads && tails && out, KGE_E_ARG, "NULL heads / tails / out");
  RowCfg c = {};
  KGE_REQUIRE(kge_pick_rowcfg(model->d, c), KGE_E_UNSUPPORTED, "embedding_size %d unsupported (1 to %d)", model->d,
              KGE_MAX_D);
  ScoreArgs a;
  a.m = *model;
  a.heads = heads;
  a.rels = rels;
  a.tails = tails;
  a.n = n;
  a.head_is_user = head_is_user;
  a.rel_row = model->ui_relation;
  const int threads = 256;
  int64_t g = (n + threads / c.g - 1) / (threads / c.g);
  const int64_t cap = (int64_t)kge_num_sms() * 8;
  const int grid = (int)(g < cap ? g : cap);
  cudaStream_t st = (cudaStream_t)stream;
#define CALL(V, G, N)                                                                          \
  switch (model->model) {                                                                      \
    case KGE_TRANSE: predict_kernel<KGE_TRANSE, V, G, N><<<grid, threads, 0, st>>>(a, out); break;     \
    case KGE_DISTMULT: predict_kernel<KGE_DISTMULT, V, G, N><<<grid, threads, 0, st>>>(a, out); break; \
    case KGE_ROTATE: predict_kernel<KGE_ROTATE, V, G, N><<<grid, threads, 0, st>>>(a, out); break;     \
    case KGE_TORUSE: predict_kernel<KGE_TORUSE, V, G, N><<<grid, threads, 0, st>>>(a, out); break;     \
    default: predict_kernel<KGE_COMPLEX, V, G, N><<<grid, threads, 0, st>>>(a, out); break;            \
  }
  KGE_DISPATCH_ROWCFG(c, CALL);
#undef CALL
  KGE_LAUNCH_CHECK();
  return 0;
}

extern "C" int kge_transd_project(const float* emb, const float* vec, const int64_t* ids, int64_t n, int32_t d,
                                  const float* rel_vec, const int64_t* rel_ids, int64_t rel_row, float* out,
                                  kge_stream_t stream) {
  KGE_REQUIRE(n >= 0 && d >= 1, KGE_E_ARG, "bad n / d");
  if (n == 0) return 0;
  KGE_REQUIRE(emb && vec && rel_vec && out && (rel_ids || rel_row >= 0), KGE_E_ARG, "NULL argument");
  RowCfg c = {};
  KGE_REQUIRE(kge_pick_rowcfg(d, c), KGE_E_UNSUPPORTED, "embedding_size %d unsupported (1 to %d)", d, KGE_MAX_D);
  const int threads = 256;
  int64_t g = (n + threads / c.g - 1) / (threads / c.g);
  const int64_t cap = (int64_t)kge_num_sms() * 8;
  const int grid = (int)(g < cap ? g : cap);
  cudaStream_t st = (cudaStream_t)stream;
#define CALL(V, G, N) \
  transd_project_kernel<V, G, N><<<grid, threads, 0, st>>>(emb, vec, ids, n, d, rel_vec, rel_ids, rel_row, out)
  KGE_DISPATCH_ROWCFG(c, CALL);
#undef CALL
  KGE_LAUNCH_CHECK();
  return 0;
}

extern "C" int kge_transh_project(const float* emb, const int64_t* ids, int64_t n, int32_t d, const float* norm_vec,
                                  const int64_t* rel_ids, int64_t rel_row, float* out, kge_stream_t stream) {
  KGE_REQUIRE(n >= 0 && d >= 1, KGE_E_ARG, "bad n / d");
  if (n == 0) return 0;
  KGE_REQUIRE(emb && norm_vec && out && (rel_ids || rel_row >= 0), KGE_E_ARG, "NULL argument");
  RowCfg c = {};
  KGE_REQUIRE(kge_pick_rowcfg(d, c), KGE_E_UNSUPPORTED, "embedding_size %d unsupported (1 to %d)", d, KGE_MAX_D);
  const int threads = 256;
  int64_t g = (n + threads / c.g - 1) / (threads / c.g);
  const int64_t cap = (int64_t)kge_num_sms() * 8;
  const int grid = (int)(g < cap ? g : cap);
  cudaStream_t st = (cudaStream_t)stream;
#define CALL(V, G, N) transh_project_kernel<V, G, N><<<grid, threads, 0, st>>>(emb, ids, n, d, norm_vec, rel_ids, rel_row, out)
  KGE_DISPATCH_ROWCFG(c, CALL);
#undef CALL
  KGE_LAUNCH_CHECK();
  return 0;
}

template <int MODE, int EPI>
static int launch_tile(const TileArgs& a, const TilePlan& pl, cudaStream_t st) {
  auto kern = pl.bu == 32 ? fullsort_tile_kernel<MODE, EPI, 32> : fullsort_tile_kernel<MODE, EPI, 16>;
  KGE_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.smem));
  // blockIdx.x is limited to 2^31-1 rows/pl.bu: fine for any table that fits the device
  dim3 grid((unsigned)pl.n_blocks, (unsigned)pl.n_splits);
  kern<<<grid, TILE_THREADS, pl.smem, st>>>(a);
  KGE_LAUNCH_CHECK();
  return 0;
}

extern "C" int kge_full_sort_scores(const kge_model_t* model, const int64_t* heads, const int64_t* rels, int64_t n,
                                    int head_is_user, int64_t n_targets, float* out, kge_stream_t stream) {
  if (int e = check_score_model(model)) return e;
  KGE_REQUIRE(n >= 0 && n_targets >= 1 && n_targets <= model->entity.rows, KGE_E_ARG, "bad n / n_targets");
  if (n == 0) return 0;
  KGE_REQUIRE(heads && out, KGE_E_ARG, "NULL heads / out");
  TilePlan pl = {};
  if (int e = plan_tiles(model, n, n_targets, 0, EPI_DENSE, pl)) return e;
  TileArgs a = {};
  a.s.m = *model;
  a.s.heads = heads;
  a.s.rels = rels;
  a.s.tails = nullptr;
  a.s.n = n;
  a.s.head_is_user = head_is_user;
  a.s.rel_row = model->ui_relation_fullsort;
  a.n_targets = n_targets;
  a.kpad = pl.kpad;
  a.tiles_per_split = pl.tiles_per_split;
  a.out = out;
  a.n_splits = 1;
  switch (tile_mode(model->model)) {
    case MODE_DIST: return launch_tile<MODE_DIST, EPI_DENSE>(a, pl, (cudaStream_t)stream);
    case MODE_TORUS: return launch_tile<MODE_TORUS, EPI_DENSE>(a, pl, (cudaStream_t)stream);
    default: return launch_tile<MODE_DOT, EPI_DENSE>(a, pl, (cudaStream_t)stream);
  }
}

extern "C" int64_t kge_full_sort_topk_workspace_bytes(const kge_model_t* model, int64_t n, int64_t n_targets,
                                                      int32_t k) {
  if (!model || n < 0 || n_targets < 1 || k < 1) return -1;
  TilePlan pl = {};
  if (k > KMAX) {
    if (large_k_cap(k) > 0x7fffffff || plan_tiles(model, n > 0 ? n : 1, n_targets, k, EPI_TOPK_LARGE, pl)) return -1;
    return (int64_t)n * pl.n_splits * large_k_cap(k) * 8;
  }
  if (plan_tiles(model, n > 0 ? n : 1, n_targets, k, EPI_TOPK, pl)) return -1;
  return (int64_t)n * pl.n_splits * k * 8;
}

extern "C" int kge_full_sort_topk(const kge_model_t* model, const int64_t* heads, const int64_t* rels, int64_t n,
                                  int head_is_user, int64_t n_targets, const int64_t* hist_off,
                                  const int64_t* hist_items, int mask_first, int32_t k, int64_t* ids_out,
                                  float* scores_out, void* workspace, int64_t workspace_bytes, kge_stream_t stream) {
  if (int e = check_score_model(model)) return e;
  KGE_REQUIRE(n >= 0 && n_targets >= 1 && n_targets <= model->entity.rows, KGE_E_ARG, "bad n / n_targets");
  KGE_REQUIRE(k >= 1, KGE_E_UNSUPPORTED, "k=%d below 1", k);
  KGE_REQUIRE(k <= n_targets, KGE_E_ARG, "k=%d larger than the number of targets", k);
  KGE_REQUIRE(n_targets < 0xFFFFFFFFll, KGE_E_UNSUPPORTED, "more than 2^32-2 targets");
  if (n == 0) return 0;
  KGE_REQUIRE(heads && ids_out, KGE_E_ARG, "NULL heads / ids_out");
  KGE_REQUIRE((hist_off == nullptr) == (hist_items == nullptr) || hist_off, KGE_E_ARG, "hist_items without hist_off");
  const bool large = k > KMAX;
  KGE_REQUIRE(!large || large_k_cap(k) <= 0x7fffffff, KGE_E_UNSUPPORTED, "k=%d: buffers above 2^31 keys", k);
  TilePlan pl = {};
  if (int e = plan_tiles(model, n, n_targets, k, large ? EPI_TOPK_LARGE : EPI_TOPK, pl)) return e;
  const int64_t need = n * pl.n_splits * (large ? large_k_cap(k) : k) * 8;
  KGE_REQUIRE(workspace && workspace_bytes >= need, KGE_E_ARG, "workspace too small: need %lld bytes", (long long)need);
  TileArgs a = {};
  a.s.m = *model;
  a.s.heads = heads;
  a.s.rels = rels;
  a.s.tails = nullptr;
  a.s.n = n;
  a.s.head_is_user = head_is_user;
  a.s.rel_row = model->ui_relation_fullsort;
  a.n_targets = n_targets;
  a.kpad = pl.kpad;
  a.tiles_per_split = pl.tiles_per_split;
  a.hist_off = hist_off;
  a.hist_items = hist_items;
  a.mask_first = mask_first;
  a.k = k;
  a.part_keys = reinterpret_cast<uint64_t*>(workspace);
  a.n_splits = pl.n_splits;
  cudaStream_t st = (cudaStream_t)stream;
  const int mode = tile_mode(model->model);
  if (large) {
    a.buf_cap = large_k_cap(k);
    if (int e = mode == MODE_DIST ? launch_tile<MODE_DIST, EPI_TOPK_LARGE>(a, pl, st)
                                  : (mode == MODE_TORUS ? launch_tile<MODE_TORUS, EPI_TOPK_LARGE>(a, pl, st)
                                                        : launch_tile<MODE_DOT, EPI_TOPK_LARGE>(a, pl, st)))
      return e;
    int64_t P = 1;
    while (P < k) P <<= 1;
    const size_t smem = P <= SORT_SM ? (size_t)P * 8 : 0;
    KGE_CUDA(cudaFuncSetAttribute(topk_merge_large_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)(SORT_SM * 8)));
    topk_merge_large_kernel<<<(unsigned)n, 256, smem, st>>>(a.part_keys, pl.n_splits, k, a.buf_cap, P, ids_out,
                                                            scores_out);
    KGE_LAUNCH_CHECK();
    return 0;
  }
  if (int e = mode == MODE_DIST ? launch_tile<MODE_DIST, EPI_TOPK>(a, pl, st)
                                : (mode == MODE_TORUS ? launch_tile<MODE_TORUS, EPI_TOPK>(a, pl, st)
                                                      : launch_tile<MODE_DOT, EPI_TOPK>(a, pl, st)))
    return e;
  const int warps = 8;
  const int64_t mg = (n + warps - 1) / warps;
  topk_merge_kernel<<<(unsigned)mg, warps * 32, (size_t)warps * k * 8, st>>>(a.part_keys, n, pl.n_splits, k, ids_out,
                                                                            scores_out, nullptr, nullptr, 0, 0);
  KGE_LAUNCH_CHECK();
  return 0;
}

extern "C" int64_t kge_full_sort_rank_workspace_bytes(const kge_model_t* model, int64_t n, int64_t n_targets,
                                                      int64_t n_pos) {
  if (!model || n < 0 || n_targets < 1 || n_pos < 0) return -1;
  TilePlan pl = {};
  if (plan_tiles(model, n > 0 ? n : 1, n_targets, 0, EPI_RANK, pl)) return -1;
  return (int64_t)rank_layout(n, n_pos).total;
}

template <int MODE>
static int launch_rank(const RankPrep& rp, const TileArgs& a, const TilePlan& pl, int64_t* greater_out,
                       int64_t* equal_out, int64_t* n_unmasked_out, cudaStream_t st) {
  const int parts = (rp.s.m.model == KGE_ROTATE || rp.s.m.model == KGE_COMPLEX) ? 2 : 1;
  const size_t smem = (size_t)(TILE_THREADS / 32) * parts * rp.s.m.d * 4;
  KGE_CUDA(cudaFuncSetAttribute(rank_thresholds_kernel<MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int64_t rows_per_cta = TILE_THREADS / 32;
  int64_t g = (rp.s.n + rows_per_cta - 1) / rows_per_cta;
  const int64_t cap = (int64_t)kge_num_sms() * 8;
  rank_thresholds_kernel<MODE><<<(unsigned)(g < cap ? g : cap), TILE_THREADS, smem, st>>>(rp);
  KGE_LAUNCH_CHECK();
  if (int e = launch_tile<MODE, EPI_RANK>(a, pl, st)) return e;
  rank_finalize_kernel<<<(unsigned)(g < cap ? g : cap), 256, 0, st>>>(rp.s.n, rp.n_targets, rp.cap, rp.pos_off,
                                                                     rp.score, rp.first, a.rank_bins, a.rank_ninf,
                                                                     greater_out, equal_out, n_unmasked_out);
  KGE_LAUNCH_CHECK();
  return 0;
}

extern "C" int kge_full_sort_rank_counts(const kge_model_t* model, const int64_t* heads, const int64_t* rels, int64_t n,
                                         int head_is_user, int64_t n_targets, const int64_t* hist_off,
                                         const int64_t* hist_items, int mask_first, const int64_t* pos_off,
                                         const int64_t* pos_items, int64_t* greater_out, int64_t* equal_out,
                                         int64_t* n_unmasked_out, void* workspace, int64_t workspace_bytes,
                                         kge_stream_t stream) {
  if (int e = check_score_model(model)) return e;
  KGE_REQUIRE(n >= 0 && n_targets >= 1 && n_targets <= model->entity.rows, KGE_E_ARG, "bad n / n_targets");
  if (n == 0) return 0;
  KGE_REQUIRE(heads && pos_off && n_unmasked_out, KGE_E_ARG, "NULL heads / pos_off / n_unmasked_out");
  KGE_REQUIRE((hist_off == nullptr) == (hist_items == nullptr) || hist_off, KGE_E_ARG, "hist_items without hist_off");
  TilePlan pl = {};
  if (int e = plan_tiles(model, n, n_targets, 0, EPI_RANK, pl)) return e;
  const RankLayout l0 = rank_layout(n, 0);
  KGE_REQUIRE(workspace && workspace_bytes >= (int64_t)l0.total, KGE_E_ARG, "workspace too small: need %lld bytes",
              (long long)l0.total);
  // the number of positives lives on the device: the workspace size says how many it holds (the kernels check it)
  int64_t cap = (workspace_bytes - (int64_t)l0.total) / 32;
  while (cap > 0 && (int64_t)rank_layout(n, cap).total > workspace_bytes) --cap;
  const RankLayout l = rank_layout(n, cap);
  unsigned char* ws = reinterpret_cast<unsigned char*>(workspace);
  cudaStream_t st = (cudaStream_t)stream;
  KGE_CUDA(cudaMemsetAsync(ws + l.ninf, 0, (size_t)n * 8, st));
  KGE_CUDA(cudaMemsetAsync(ws + l.bins, 0, (size_t)cap * 16, st));
  KGE_CUDA(cudaMemsetAsync(n_unmasked_out, 0, (size_t)n * 8, st));
  RankPrep rp = {};
  rp.s.m = *model;
  rp.s.heads = heads;
  rp.s.rels = rels;
  rp.s.n = n;
  rp.s.head_is_user = head_is_user;
  rp.s.rel_row = model->ui_relation_fullsort;
  rp.n_targets = n_targets;
  rp.hist_off = hist_off;
  rp.hist_items = hist_items;
  rp.mask_first = mask_first;
  rp.pos_off = pos_off;
  rp.pos_items = pos_items;
  rp.cap = cap;
  rp.score = reinterpret_cast<float*>(ws + l.score);
  rp.sorted = reinterpret_cast<float*>(ws + l.sorted);
  rp.first = reinterpret_cast<int64_t*>(ws + l.first);
  rp.lo = reinterpret_cast<float*>(ws + l.lo);
  TileArgs a = {};
  a.s = rp.s;
  a.n_targets = n_targets;
  a.kpad = pl.kpad;
  a.tiles_per_split = pl.tiles_per_split;
  a.hist_off = hist_off;
  a.hist_items = hist_items;
  a.mask_first = mask_first;
  a.n_splits = pl.n_splits;
  a.pos_off = pos_off;
  a.rank_thr = rp.sorted;
  a.rank_lo = rp.lo;
  a.rank_bins = reinterpret_cast<uint64_t*>(ws + l.bins);
  a.rank_unmasked = reinterpret_cast<uint64_t*>(n_unmasked_out);
  a.rank_ninf = reinterpret_cast<uint64_t*>(ws + l.ninf);
  a.rank_cap = cap;
  switch (tile_mode(model->model)) {
    case MODE_DIST: return launch_rank<MODE_DIST>(rp, a, pl, greater_out, equal_out, n_unmasked_out, st);
    case MODE_TORUS: return launch_rank<MODE_TORUS>(rp, a, pl, greater_out, equal_out, n_unmasked_out, st);
    default: return launch_rank<MODE_DOT>(rp, a, pl, greater_out, equal_out, n_unmasked_out, st);
  }
}

// ---- device-gated exact top-k for a row list that only exists on the device ------------------------------
// Used by the tensor-core path (mma_topk.cu) for the rows its filter hands back: `row_map[0 .. *row_count)` are
// their indices.  No host round trip: two fixed-size launches cover every possible count --
//   entries [0, FB_SPLIT_ROWS)      row blocks x target splits, so that a handful of rows still fills the GPU
//   entries [FB_SPLIT_ROWS, n)      one CTA per row block (plenty of rows: no splits needed), CTAs stride
// -- and CTAs beyond the count leave at once (~10 us per call when nothing was flagged).
namespace {
constexpr int64_t FB_SPLIT_ROWS = 1024;
constexpr int FB_SPLITS = 48;
struct FallbackPlan {
  TilePlan tp;
  int splits, tiles_per_split;
  int64_t keys_a, keys_b;   // part_keys elements of the two regions
};
int plan_fallback(const kge_model_t* m, int64_t n, int64_t n_targets, int k, FallbackPlan& fp) {
  if (int e = plan_tiles(m, n > 0 ? n : 1, n_targets, k, EPI_TOPK, fp.tp)) return e;
  const int64_t n_tiles = (n_targets + BT - 1) / BT;
  int64_t s = FB_SPLITS;
  if (s > (n_tiles + 7) / 8) s = (n_tiles + 7) / 8;
  if (s < 1) s = 1;
  fp.tiles_per_split = (int)((n_tiles + s - 1) / s);
  fp.splits = (int)((n_tiles + fp.tiles_per_split - 1) / fp.tiles_per_split);
  const int64_t ra = n < FB_SPLIT_ROWS ? n : FB_SPLIT_ROWS;
  fp.keys_a = ra * fp.splits * k;
  fp.keys_b = (n - ra) * k;
  return 0;
}
}  // namespace

int64_t kge_topk_rows_indirect_workspace_bytes(const kge_model_t* model, int64_t n, int64_t n_targets, int32_t k) {
  FallbackPlan fp = {};
  if (!model || k < 1 || k > KMAX || plan_fallback(model, n, n_targets, k, fp)) return -1;
  return (fp.keys_a + fp.keys_b) * 8;
}

int kge_topk_rows_indirect(const kge_model_t* model, const int64_t* heads, const int64_t* rels, int64_t n,
                           int head_is_user, int64_t n_targets, const int64_t* hist_off, const int64_t* hist_items,
                           int mask_first, int32_t k, const int32_t* row_map, const int32_t* row_count,
                           int64_t* ids_out, float* scores_out, void* workspace, cudaStream_t st) {
  if (int e = check_score_model(model)) return e;
  FallbackPlan fp = {};
  if (int e = plan_fallback(model, n, n_targets, k, fp)) return e;
  TileArgs a = {};
  a.s.m = *model;
  a.s.heads = heads;
  a.s.rels = rels;
  a.s.n = n;
  a.s.head_is_user = head_is_user;
  a.s.rel_row = model->ui_relation_fullsort;
  a.n_targets = n_targets;
  a.kpad = fp.tp.kpad;
  a.hist_off = hist_off;
  a.hist_items = hist_items;
  a.mask_first = mask_first;
  a.k = k;
  a.row_map = row_map;
  a.row_count = row_count;
  const int mode = tile_mode(model->model);
  const int bu = fp.tp.bu;
  auto kern = bu == 32 ? (mode == MODE_DIST ? fullsort_tile_kernel<MODE_DIST, EPI_TOPK, 32>
                                            : (mode == MODE_TORUS ? fullsort_tile_kernel<MODE_TORUS, EPI_TOPK, 32>
                                                                  : fullsort_tile_kernel<MODE_DOT, EPI_TOPK, 32>))
                       : (mode == MODE_DIST ? fullsort_tile_kernel<MODE_DIST, EPI_TOPK, 16>
                                            : (mode == MODE_TORUS ? fullsort_tile_kernel<MODE_TORUS, EPI_TOPK, 16>
                                                                  : fullsort_tile_kernel<MODE_DOT, EPI_TOPK, 16>));
  KGE_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fp.tp.smem));
  const int warps = 8;
  const int64_t ra = n < FB_SPLIT_ROWS ? n : FB_SPLIT_ROWS;
  uint64_t* keys = reinterpret_cast<uint64_t*>(workspace);
  // region A: few rows, many splits
  a.part_keys = keys;
  a.n_splits = fp.splits;
  a.tiles_per_split = fp.tiles_per_split;
  a.row_begin = 0;
  a.row_end = ra;
  kern<<<dim3((unsigned)((ra + bu - 1) / bu), (unsigned)fp.splits), TILE_THREADS, fp.tp.smem, st>>>(a);
  KGE_LAUNCH_CHECK();
  topk_merge_kernel<<<(unsigned)((ra + warps - 1) / warps), warps * 32, (size_t)warps * k * 8, st>>>(
      a.part_keys, n, a.n_splits, k, ids_out, scores_out, row_map, row_count, 0, ra);
  KGE_LAUNCH_CHECK();
  if (n > ra) {   // region B: one CTA per row block, striding
    a.part_keys = keys + fp.keys_a;
    a.n_splits = 1;
    a.tiles_per_split = (int)((n_targets + BT - 1) / BT);
    a.row_begin = ra;
    a.row_end = n;
    int64_t g = (n - ra + bu - 1) / bu;
    const int64_t cap = (int64_t)kge_num_sms() * 2;
    if (g > cap) g = cap;
    kern<<<dim3((unsigned)g, 1), TILE_THREADS, fp.tp.smem, st>>>(a);
    KGE_LAUNCH_CHECK();
    topk_merge_kernel<<<(unsigned)g, warps * 32, (size_t)warps * k * 8, st>>>(a.part_keys, n, 1, k, ids_out, scores_out,
                                                                             row_map, row_count, ra, n);
    KGE_LAUNCH_CHECK();
  }
  return 0;
}

extern "C" int kge_topk_hits(const int64_t* ids, int64_t n, int32_t k, const int64_t* pos_off, const int64_t* pos_items,
                             int32_t* out, kge_stream_t stream) {
  KGE_REQUIRE(n >= 0 && k >= 1, KGE_E_ARG, "bad n / k");
  if (n == 0) return 0;
  KGE_REQUIRE(ids && pos_off && pos_items && out, KGE_E_ARG, "NULL argument");
  const int64_t total = n * (int64_t)(k + 1);
  int64_t g = (total + 255) / 256;
  const int64_t cap = (int64_t)kge_num_sms() * 8;
  topk_hits_kernel<<<(unsigned)(g < cap ? g : cap), 256, 0, (cudaStream_t)stream>>>(ids, n, k, pos_off, pos_items, out);
  KGE_LAUNCH_CHECK();
  return 0;
}

extern "C" int kge_topk_metric_sums(const int32_t* rec_topk, int64_t n, int32_t k, double* sums, kge_stream_t stream) {
  KGE_REQUIRE(n >= 0 && k >= 1, KGE_E_ARG, "bad n / k");
  if (n == 0) return 0;
  KGE_REQUIRE(rec_topk && sums, KGE_E_ARG, "NULL argument");
  int64_t g = (n + 255) / 256;
  const int64_t cap = (int64_t)kge_num_sms() * 4;
  if (k > KMAX) {
    const int64_t n_win = (k + MW - 1) / MW;
    // about as many CTAs in all as the k <= KMAX launch (each one takes a window)
    int64_t gx = (g < cap ? g : cap) / n_win;
    if (gx < 1) gx = 1;
    const dim3 grid((unsigned)gx, (unsigned)(n_win < 65535 ? n_win : 65535));
    topk_metric_sums_window_kernel<<<grid, 256, (size_t)8 * 5 * MW * 8, (cudaStream_t)stream>>>(rec_topk, n, k, sums);
    KGE_LAUNCH_CHECK();
    return 0;
  }
  topk_metric_sums_kernel<<<(unsigned)(g < cap ? g : cap), 256, (size_t)8 * 5 * k * 8, (cudaStream_t)stream>>>(rec_topk, n, k,
                                                                                                         sums);
  KGE_LAUNCH_CHECK();
  return 0;
}

// ---- sampled evaluation: per-row selection over a candidate list (uni-N / pop-N) ----------------------------------
// The dense route scatters each row's candidate scores into a -inf row of n_targets columns, then runs torch.topk and
// (for GAUC) a full sort over it.  Here a row is its candidate list only: keys are sorted in on-chip or workspace
// memory, twice -- by id (duplicates collapse, positives find their scores, the padding finds the smallest
// non-candidate ids) and then by (score desc, id asc) for the top k and the rank counts.  Rows pick their regime on
// the device: up to CAND_WARP_MAX keys a warp sorts them in shared memory, up to CAND_CTA_MAX a CTA does, longer rows
// sort in the workspace at their own candidate offset.
namespace {
constexpr int CAND_WARP_MAX = 512;
constexpr int CAND_CTA_MAX = 8192;
constexpr int CAND_THREADS = 256;

struct CandArgs {
  const float* scores;
  const int64_t* items;
  int64_t n_cand;
  const int64_t* off;
  int64_t n, n_targets;
  const int64_t* pos_off;
  const int64_t* pos_items;
  int k;
  int64_t* ids_out;
  float* scores_out;
  int64_t* greater_out;
  int64_t* equal_out;
  int64_t* n_unmasked_out;
  uint64_t* ws;   // [n_cand] keys: rows above CAND_CTA_MAX sort at their candidate offset
};

__device__ __forceinline__ uint64_t rot32(uint64_t x) { return (x << 32) | (x >> 32); }

template <bool BLOCK>
__device__ __forceinline__ void group_sync() {
  if (BLOCK) __syncthreads(); else __syncwarp();
}

// Sort buf[0, len) descending with a group of nt threads (a warp or the block).  Bitonic network over the next power
// of two P >= len in the form whose every compare-exchange moves the larger key to the lower index (each merge starts
// with the mirrored comparison): the keys past len are virtual zeros, the smallest key, which never move, so they
// need no storage.
template <bool BLOCK>
__device__ void group_sort_desc(uint64_t* buf, int64_t len, int tid, int nt) {
  int64_t P = 1;
  while (P < len) P <<= 1;
  for (int64_t size = 2; size <= P; size <<= 1) {
    const int64_t half = size >> 1;
    for (int64_t i = tid; i < P / 2; i += nt) {
      const int64_t blk = i / half, j = i - blk * half;
      const int64_t lo = blk * size + j, hi = blk * size + size - 1 - j;
      if (hi < len) {
        const uint64_t x = buf[lo], y = buf[hi];
        if (x < y) {
          buf[lo] = y;
          buf[hi] = x;
        }
      }
    }
    group_sync<BLOCK>();
    for (int64_t stride = size >> 2; stride > 0; stride >>= 1) {
      for (int64_t i = tid; i < P / 2; i += nt) {
        const int64_t lo = 2 * i - (i & (stride - 1)), hi = lo + stride;
        if (hi < len) {
          const uint64_t x = buf[lo], y = buf[hi];
          if (x < y) {
            buf[lo] = y;
            buf[hi] = x;
          }
        }
      }
      group_sync<BLOCK>();
    }
  }
}

// Drop the repeats of the sorted buf[0, len) in place; returns the number of distinct keys (group-uniform).  A round
// reads all its keys before it writes, and writes land at or below the positions read, so later rounds read
// untouched keys; the last key of a round is carried into the next (s_carry / s_cnt: block only).
template <bool BLOCK>
__device__ int64_t group_unique(uint64_t* buf, int64_t len, int tid, int nt, uint32_t* s_cnt, uint64_t* s_carry) {
  const int lane = tid & 31, warp = tid >> 5;
  int64_t w = 0;
  uint64_t carry = 0ull;   // no key is 0
  if (BLOCK) {
    if (tid == 0) *s_carry = 0ull;
    __syncthreads();
  }
  for (int64_t base = 0; base < len; base += nt) {
    const int64_t i = base + tid;
    const uint64_t x = i < len ? buf[i] : 0ull;
    uint64_t prev;
    if (BLOCK) {
      prev = (tid == 0) ? *s_carry : (i < len ? buf[i - 1] : 0ull);
    } else {
      prev = __shfl_up_sync(0xffffffffu, x, 1);
      if (lane == 0) prev = carry;
    }
    const bool keep = i < len && x != prev;
    const unsigned b = __ballot_sync(0xffffffffu, keep);
    const int below = __popc(b & ((1u << lane) - 1u));
    if (BLOCK) {
      if (lane == 0) s_cnt[warp] = __popc(b);
      __syncthreads();   // every read of the round is done and the counts are in
      int before = 0, total = 0;
      for (int q = 0; q < (nt >> 5); ++q) {
        const int c = (int)s_cnt[q];
        before += q < warp ? c : 0;
        total += c;
      }
      if (keep) buf[w + before + below] = x;
      if (tid == nt - 1) *s_carry = x;
      w += total;
      __syncthreads();
    } else {
      if (keep) buf[w + below] = x;
      w += __popc(b);
      carry = __shfl_sync(0xffffffffu, x, 31);
      __syncwarp();
    }
  }
  return w;
}

// Number of keys of the descending buf[0, D) whose upper 32 bits are >= h (h <= 2^32).
__device__ __forceinline__ int64_t count_hi_ge(const uint64_t* buf, int64_t D, uint64_t h) {
  int64_t lo = 0, hi = D;
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    if ((buf[mid] >> 32) >= h) lo = mid + 1; else hi = mid;
  }
  return lo;
}

template <bool BLOCK>
__device__ void cand_row(const CandArgs& a, int64_t row, int64_t c0, int64_t len, uint64_t* buf, int tid, int nt,
                         uint32_t* s_cnt, uint64_t* s_carry) {
  // 1. by id: key (~id << 32 | score bits), sorted descending = id ascending; equal ids carry equal scores
  for (int64_t i = tid; i < len; i += nt)
    buf[i] = rot32(make_key(__ldg(a.scores + c0 + i), (uint32_t)__ldg(a.items + c0 + i)));
  group_sync<BLOCK>();
  group_sort_desc<BLOCK>(buf, len, tid, nt);
  const int64_t D = group_unique<BLOCK>(buf, len, tid, nt, s_cnt, s_carry);
  if (a.n_unmasked_out && tid == 0) a.n_unmasked_out[row] = D;
  const int64_t k = a.k;
  // the padding of a row with fewer than k candidates: the smallest non-candidate ids, ascending, score -inf.  Id x
  // that is not a candidate is non-candidate number x - #(candidates < x).
  if (D < k && (a.ids_out || a.scores_out))
    for (int64_t x = tid; x < k + D && x < a.n_targets; x += nt) {
      const int64_t c = count_hi_ge(buf, D, 0x100000000ull - (uint64_t)x);   // candidates with id < x
      const bool member = c < D && (buf[c] >> 32) == 0xFFFFFFFFull - (uint64_t)x;
      const int64_t j = x - c;
      if (!member && j < k - D) {
        if (a.ids_out) a.ids_out[row * k + D + j] = x;
        if (a.scores_out) a.scores_out[row * k + D + j] = -INFINITY;
      }
    }
  // each positive's score bits, or -1 when it is not a candidate, parked in its own greater_out slot
  const int64_t p0 = a.greater_out ? a.pos_off[row] : 0, p1 = a.greater_out ? a.pos_off[row + 1] : 0;
  for (int64_t i = p0 + tid; i < p1; i += nt) {
    const uint64_t h = 0xFFFFFFFFull - (uint64_t)(uint32_t)a.pos_items[i];
    const int64_t c = count_hi_ge(buf, D, h + 1);
    a.greater_out[i] = (c < D && (buf[c] >> 32) == h) ? (int64_t)(uint32_t)buf[c] : -1;
  }
  group_sync<BLOCK>();
  // 2. by (score desc, id asc): make_key's layout
  for (int64_t i = tid; i < D; i += nt) buf[i] = rot32(buf[i]);
  group_sync<BLOCK>();
  group_sort_desc<BLOCK>(buf, D, tid, nt);
  const int64_t top = D < k ? D : k;
  for (int64_t i = tid; i < top; i += nt) {
    const uint64_t key = buf[i];
    if (a.ids_out) a.ids_out[row * k + i] = key_id(key);
    if (a.scores_out) a.scores_out[row * k + i] = key_score(key);
  }
  // the counts of kge_full_sort_rank_counts over the row's distinct candidates; the rest of the row is -inf
  for (int64_t i = p0 + tid; i < p1; i += nt) {
    const int64_t t = a.greater_out[i];
    int64_t g = D, e = a.n_targets - D;
    if (t >= 0) {
      g = count_hi_ge(buf, D, (uint64_t)t + 1);
      e = count_hi_ge(buf, D, (uint64_t)t) - g;
    }
    a.greater_out[i] = g;
    a.equal_out[i] = e;
  }
  group_sync<BLOCK>();
}

__device__ __forceinline__ void cand_range(const CandArgs& a, int64_t row, int64_t& c0, int64_t& len) {
  // (clamped to [0, n_cand]: a malformed offset list cannot send a row outside the candidates)
  int64_t s = __ldg(a.off + row), e = __ldg(a.off + row + 1);
  s = s < 0 ? 0 : (s > a.n_cand ? a.n_cand : s);
  e = e < s ? s : (e > a.n_cand ? a.n_cand : e);
  c0 = s;
  len = e - s;
}

// One warp per row, rows of at most CAND_WARP_MAX candidates.
__global__ void __launch_bounds__(CAND_THREADS) cand_select_warp_kernel(const CandArgs a) {
  __shared__ uint64_t bufs[CAND_THREADS / 32][CAND_WARP_MAX];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t row = (int64_t)blockIdx.x * (CAND_THREADS / 32) + warp;
  if (row >= a.n) return;
  int64_t c0, len;
  cand_range(a, row, c0, len);
  if (len > CAND_WARP_MAX) return;
  cand_row<false>(a, row, c0, len, bufs[warp], lane, 32, nullptr, nullptr);
}

// One CTA per row, rows above CAND_WARP_MAX candidates: in shared memory up to CAND_CTA_MAX, else in the workspace.
// The CTAs stride over the rows (how many are long is only known on the device).
__global__ void __launch_bounds__(CAND_THREADS) cand_select_cta_kernel(const CandArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ uint32_t s_cnt[CAND_THREADS / 32];
  __shared__ uint64_t s_carry;
  for (int64_t row = blockIdx.x; row < a.n; row += gridDim.x) {
    int64_t c0, len;
    cand_range(a, row, c0, len);
    if (len <= CAND_WARP_MAX) continue;
    uint64_t* buf = len <= CAND_CTA_MAX ? reinterpret_cast<uint64_t*>(smem_raw) : a.ws + c0;
    cand_row<true>(a, row, c0, len, buf, threadIdx.x, blockDim.x, s_cnt, &s_carry);
  }
}
}  // namespace

extern "C" int64_t kge_candidate_select_workspace_bytes(int64_t n, int64_t n_cand) {
  if (n < 0 || n_cand < 0) return -1;
  return n_cand * 8;
}

extern "C" int kge_candidate_select(const float* scores, const int64_t* cand_items, int64_t n_cand,
                                    const int64_t* cand_off, int64_t n, int64_t n_targets, const int64_t* pos_off,
                                    const int64_t* pos_items, int32_t k, int64_t* ids_out, float* scores_out,
                                    int64_t* greater_out, int64_t* equal_out, int64_t* n_unmasked_out,
                                    void* workspace, int64_t workspace_bytes, kge_stream_t stream) {
  KGE_REQUIRE(n >= 0 && n_cand >= 0, KGE_E_ARG, "negative n / n_cand");
  KGE_REQUIRE(k >= 1, KGE_E_ARG, "k=%d below 1", k);
  KGE_REQUIRE(n_targets >= 1 && n_targets < 0xFFFFFFFFll, KGE_E_ARG, "n_targets outside [1, 2^32-2]");
  KGE_REQUIRE(k <= n_targets, KGE_E_ARG, "k=%d larger than the number of targets", k);
  KGE_REQUIRE((greater_out == nullptr) == (equal_out == nullptr), KGE_E_ARG, "greater_out and equal_out go together");
  if (n == 0) return 0;
  KGE_REQUIRE(cand_off, KGE_E_ARG, "NULL cand_off");
  KGE_REQUIRE(n_cand == 0 || (scores && cand_items), KGE_E_ARG, "NULL scores / cand_items");
  KGE_REQUIRE(!greater_out || (pos_off && pos_items), KGE_E_ARG, "NULL pos_off / pos_items");
  KGE_REQUIRE(workspace_bytes >= n_cand * 8 && (n_cand == 0 || workspace), KGE_E_ARG,
              "workspace too small: need %lld bytes", (long long)(n_cand * 8));
  CandArgs a;
  a.scores = scores;
  a.items = cand_items;
  a.n_cand = n_cand;
  a.off = cand_off;
  a.n = n;
  a.n_targets = n_targets;
  a.pos_off = pos_off;
  a.pos_items = pos_items;
  a.k = k;
  a.ids_out = ids_out;
  a.scores_out = scores_out;
  a.greater_out = greater_out;
  a.equal_out = equal_out;
  a.n_unmasked_out = n_unmasked_out;
  a.ws = reinterpret_cast<uint64_t*>(workspace);
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t rows_per_cta = CAND_THREADS / 32;
  cand_select_warp_kernel<<<(unsigned)((n + rows_per_cta - 1) / rows_per_cta), CAND_THREADS, 0, st>>>(a);
  KGE_LAUNCH_CHECK();
  // rows above CAND_WARP_MAX need at least that many candidates each
  int64_t g = n_cand / (CAND_WARP_MAX + 1);
  const int64_t cap = (int64_t)kge_num_sms() * 3;
  if (g > cap) g = cap;
  if (g > n) g = n;
  if (g >= 1) {
    const size_t smem = (size_t)CAND_CTA_MAX * 8;
    KGE_CUDA(cudaFuncSetAttribute(cand_select_cta_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    cand_select_cta_kernel<<<(unsigned)g, CAND_THREADS, smem, st>>>(a);
    KGE_LAUNCH_CHECK();
  }
  return 0;
}
