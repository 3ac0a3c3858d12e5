// Full-sort top-k on the 5th-generation tensor cores (tcgen05 + TMEM) of sm_100a, exact in fp32.
//
// Replaces the same reference code as score.cu's fused top-k
// (model/knowledge_graph_embedding_recommender/{distmult.py:119-133, complex.py:162-190,
// transe.py:112-126, rotate.py:161-190}, trainer/trainer.py:716-735, evaluator/collector.py:176-177)
// for the scorers that are dense contractions: DistMult / ComplEx directly (score = q . t) and
// the L2 models through  -||q - t||^2 = 2 (q . t - ||t||^2 / 2) - ||q||^2  (the per-row constant
// does not change the order; -||t||^2/2 rides in three extra K columns as an fp16 hi/mid/lo split).
//
// The tensor cores only FILTER; the answer is exact:
//   1. fp16 GEMM  a^_ij ~ S_i (q_i . t_j)  with fp32 accumulation in TMEM.  Operands are scaled by powers of two
//      (exact): the target image by 2^e_t so that max |t_c| lands in [2^7, 2^8), every query row by its own 2^e_i
//      the same way, S_i = 2^(e_i + e_t).  fp16 keeps 11 significant bits: fl(x) = x (1 + d), |d| <= 2^-11 (or an
//      absolute error below 2^-14 in the subnormal range, flushed or not), so with Cauchy-Schwarz
//        |a^ - S a| <= eps_i = (2^-10 + 2^-20) |q^| |t^|max + 2^-14 sqrt(K) (|q^| + |t^|max) + K 2^-22 (...)
//      (two roundings per product, the subnormal floor, fp32 accumulation; see row_eps()).  Round 1 used bf16
//      with 1.02 * 2^-8: too small by 2x (two roundings of 2^-8 each) -- fp16 is 8x tighter than the valid bf16
//      bound at the same tensor-core rate.
//   2. sweep epilogue, one thread per query row: the maximum of each chunk of 32 adjacent targets is compared
//      with a running threshold thr_i = tau_i - 2 eps_i, where tau_i is the k-th largest chunk maximum
//      among chunks without masked targets seen so far (a lower bound of the k-th largest unmasked
//      approximate score).  Every member of the exact top-k has a^ >= tau_final - 2 eps, so its chunk
//      survives.  A surviving chunk is appended, with the mask of its groups of GRP targets that clear the
//      threshold, to a list of CAND entries per (row, split, column slice) in global memory (L2); when a list
//      fills, its warp compacts it (radix select of tau, keep the entries >= tau - 2 eps); a list that cannot
//      be compacted flags the row.
//   3. rescore kernel (one warp per row): final tau over the row's lists, then only the targets of
//      the groups >= tau - 2 eps are scored in fp32 with the same sequential FMA chain as the
//      CUDA-core kernel (bit-identical scores), masked, pre-filtered by score >= tau - eps (the k
//      targets behind tau have exact scores above that) and selected under (score desc, id asc).
//      Flagged rows and rows with fewer than k valid candidates are reported to the caller, which
//      runs them through kge_full_sort_topk.
//
// Sweep kernel (fullsort_mma_kernel): a CTA keeps NH row halves of 128 query rows in shared memory and sweeps
// target tiles of TN rows; every B tile feeds one M = 128 MMA per half.  Each half has NBUF accumulators in TMEM:
// one in shape (a) (256 columns, so that two CTAs share an SM), two in shapes (f), (c) and (k), where the MMAs of
// tile i+1 run under the epilogue of tile i.  plan_mma picks the shape (DESIGN 3.4(b) item 2).  Warp roles, in warp
// order (sweep_threads): the epilogue warps, one thread per query row; one producer warp that streams the pre-tiled
// fp16 target image with cp.async.bulk into a ring of shared-memory stages (mbarrier expect_tx); NMMA issuer warps
// whose elected lane issues tcgen05.mma.  A grid of (row blocks) x (target splits) fills the GPU when few users are
// evaluated; every (row, split, column slice) owns a list.  Operands use the no-swizzle K-major canonical layout
// [K/8][rows][8 fp16]: 8x16-byte core matrices, SBO = 128 B, LBO = rows * 16 B.
#include <cuda_fp16.h>
#include <math.h>

#include "common.cuh"
#include "score_common.cuh"

namespace {

constexpr int MH = 128;    // query rows per row half (one M = 128 accumulator); a CTA sweeps NH = 1 or 2 halves
constexpr int GRP = 4;     // targets per candidate group (what the rescore kernel reads per mask bit)
constexpr int CAND = 128;  // candidate chunks kept per (row, split)
constexpr int MAX_SPLITS = 4;
// Warps of a sweep CTA, in this order: 4 * NH * NCOL epilogue warps (warp % 4 = TMEM lane quadrant, (warp / 4) % NH =
// row half, warp / (4 * NH) = column slice of the tile), one producer warp, NMMA issuer warps.  The issuers come last:
// the issue arbiter favours high warp ids, and an MMA issuer must never starve.  (A CTA that has the SM to itself
// takes one issuer per row half: a free-running issuer needs ~125 cycles per tcgen05.mma.)
constexpr int PRODUCER_WARPS = 1;
__host__ __device__ constexpr int sweep_threads(int nh, int ncol, int nmma) {
  return (4 * nh * ncol + PRODUCER_WARPS + nmma) * 32;
}
constexpr int IMG_HEADER = 128;  // bytes before the first tile image: {max |t|, max |t_c|, max |t|^2} (floats)
constexpr uint32_t SPIN_LIMIT = 1u << 26;

// ---- PTX wrappers -------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;   // (a suspend-time hint or a pure test_wait spin made no difference: measured, scripts/gpu_exp_sweep.sh)
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
// A wait that cannot hang the GPU: a protocol bug traps instead of spinning forever.  The loop is written in PTX:
// the C form let the compiler re-derive the barrier address (S2R + shifts) inside the spin, eight instructions
// per poll that compete with the working warps for issue slots.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred p, q;\n\t.reg .u32 n;\n\t"
      "mov.u32 n, 0;\n"
      "KGE_WAIT:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra KGE_DONE;\n\t"
      "add.u32 n, n, 1;\n\t"
      "setp.lt.u32 q, n, %2;\n\t"
      "@q bra KGE_WAIT;\n\t"
      "trap;\n"
      "KGE_DONE:\n\t}"
      :
      : "r"(bar), "r"(parity), "n"(SPIN_LIMIT)
      : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
               "l"(src), "r"(bytes), "r"(bar)
               : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_alloc(uint32_t dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t addr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                         uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      :
      : "r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
#define KGE_TMEM_LD32_ASM(R, ADDR)                                                                                  \
  asm volatile(                                                                                                    \
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "                                                                    \
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "                                     \
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"                     \
      : "=r"(R[0]), "=r"(R[1]), "=r"(R[2]), "=r"(R[3]), "=r"(R[4]), "=r"(R[5]), "=r"(R[6]), "=r"(R[7]), "=r"(R[8]),  \
        "=r"(R[9]), "=r"(R[10]), "=r"(R[11]), "=r"(R[12]), "=r"(R[13]), "=r"(R[14]), "=r"(R[15]), "=r"(R[16]),      \
        "=r"(R[17]), "=r"(R[18]), "=r"(R[19]), "=r"(R[20]), "=r"(R[21]), "=r"(R[22]), "=r"(R[23]), "=r"(R[24]),     \
        "=r"(R[25]), "=r"(R[26]), "=r"(R[27]), "=r"(R[28]), "=r"(R[29]), "=r"(R[30]), "=r"(R[31])                   \
      : "r"(ADDR)                                                                                                  \
      : "memory")
// 32 consecutive accumulator columns of this thread's TMEM lane, issued without waiting ...
__device__ __forceinline__ void tmem_ld32_issue(uint32_t taddr, uint32_t (&r)[32]) {
  KGE_TMEM_LD32_ASM(r, taddr);
}
// ... and the wait; naming the registers keeps every use of them behind it.
__device__ __forceinline__ void tmem_ld_wait(uint32_t (&r)[32]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]),
                 "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15]),
                 "+r"(r[16]), "+r"(r[17]), "+r"(r[18]), "+r"(r[19]), "+r"(r[20]), "+r"(r[21]), "+r"(r[22]), "+r"(r[23]),
                 "+r"(r[24]), "+r"(r[25]), "+r"(r[26]), "+r"(r[27]), "+r"(r[28]), "+r"(r[29]), "+r"(r[30]), "+r"(r[31])
               :
               : "memory");
}
// The same wait for two register sets in flight (tcgen05.wait::ld covers every load the thread has issued).
__device__ __forceinline__ void tmem_ld_wait2(uint32_t (&r)[32], uint32_t (&q)[32]) {
  tmem_ld_wait(r);
  asm volatile(""
               : "+r"(q[0]), "+r"(q[1]), "+r"(q[2]), "+r"(q[3]), "+r"(q[4]), "+r"(q[5]), "+r"(q[6]), "+r"(q[7]),
                 "+r"(q[8]), "+r"(q[9]), "+r"(q[10]), "+r"(q[11]), "+r"(q[12]), "+r"(q[13]), "+r"(q[14]), "+r"(q[15]),
                 "+r"(q[16]), "+r"(q[17]), "+r"(q[18]), "+r"(q[19]), "+r"(q[20]), "+r"(q[21]), "+r"(q[22]), "+r"(q[23]),
                 "+r"(q[24]), "+r"(q[25]), "+r"(q[26]), "+r"(q[27]), "+r"(q[28]), "+r"(q[29]), "+r"(q[30]), "+r"(q[31])
               :
               : "memory");
}
__device__ __forceinline__ float max3f(float a, float b, float c) {
  float r;
  asm("max.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c));
  return r;
}

// One lane of the (converged) warp; the choice is stable across calls.
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

// Shared-memory matrix descriptors (no-swizzle, K-major) are assembled in the MMA issuer: bits start>>4 [0,14),
// LBO>>4 [16,30), SBO>>4 [32,46), version = 1 [46,48), layout type 0 = SWIZZLE_NONE [61,64).
// kind::f16 instruction descriptor: D fp32 (bit 4), A/B fp16 (format 0), both K-major, N = tn, M = 128.
__host__ __device__ constexpr uint32_t make_idesc(int tn) {
  return (1u << 4) | ((uint32_t)(tn >> 3) << 17) | ((128u >> 4) << 24);
}

__device__ __forceinline__ uint16_t f16_bits(float x) { return __half_as_ushort(__float2half_rn(x)); }
__device__ __forceinline__ float f16_back(uint16_t b) { return __half2float(__ushort_as_half(b)); }

// ---- operand scaling ------------------------------------------------------------------------------
// Powers of two, so exact.  The image header holds {tmax = max_j |t_j| (x 1.0001), max |t_jc|, max |t_j|^2}:
//   e_t: targets are stored as fp16(t * 2^e_t), the largest element in [2^7, 2^8)
//   e_w: the L2 models' extra K columns hold W_j = -|t_j|^2 / 2 * 2^e_w (|W| < 2^8) as an fp16 hi/mid/lo split; a
//        query row carries the constant c_i = 2^(e_i + e_t - e_w) there, so c_i W_j = -S_i |t_j|^2 / 2.
// Exponents are clamped to +-60 so that S_i and 1 / S_i stay finite fp32 numbers.
constexpr int E_CLAMP = 60;
struct ImgScale {
  float tmax;
  int e_t, e_w;
};
__device__ __forceinline__ int clamp_exp(int e) { return e > E_CLAMP ? E_CLAMP : (e < -E_CLAMP ? -E_CLAMP : e); }
__device__ __forceinline__ ImgScale img_scale(const float* header) {
  ImgScale s;
  s.tmax = header[0];
  const float ma = header[1], w = 0.5f * header[2];
  s.e_t = ma > 0.f ? clamp_exp(7 - ilogbf(ma)) : 0;
  s.e_w = w > 0.f ? clamp_exp(7 - ilogbf(w)) : 0;
  return s;
}

// Error bound of one row, in the row's scaled units.  nqs = |q| 2^e_i, tms = tmax 2^e_t, K = padded depth,
// c = the A-side constant of the L2 columns (0 for the bilinear models).  Terms:
//   (2^-10 + 2^-20) nqs tms            two fp16 roundings per product: (1 + u)^2 - 1 with u = 2^-11, Cauchy-Schwarz
//   2^-14 sqrt(K) (nqs + tms) 1.001    elements in the fp16 subnormal range: absolute error < 2^-14 each whether the
//                                      tensor core flushes them or rounds them (sum |x_c| <= sqrt(K) |x|)
//   K 2^-28                            products of two such elements
//   K 2^-22 (nqs tms 1.001 + 2^8 c)    fp32 accumulation of K products (one truncated ulp each, partial sums bounded by
//                                      the sum of magnitudes)
//   3 * 2^-14 c                        the hi/mid/lo split of W (exact up to the subnormal floor of each piece)
//   (K + 2) 2^-24 chain                the rescore's own fp32 chain: the top-k is decided by its scores, not by the real
//                                      ones, and one sequential chain over <= K - 2 columns is off by at most (K + 2)
//                                      2^-24 times the sum of its terms' magnitudes -- chain = S |q| tmax (q . t), or
//                                      S (|q| + tmax)^2 / 2 (a = (|q|^2 - |q - t|^2) / 2).  Without it a row whose |q|
//                                      dwarfs every |t| (L2 models) ranks targets the fp32 chain cannot tell apart, and
//                                      the id order among those ties picks members the filter dropped.  (K >= P + 3
//                                      columns for the L2 models: the spare covers the rounding of sqrtf(acc) as well.)
//   2^-23 last                         RotatE's reported score margin - sqrtf(acc) is rounded once more, to ulps of
//                                      the margin: targets whose |q - t| differ by less than that tie, which is
//                                      |margin| (|q| + tmax) 2^-24 in the units of a; last = S |margin| (|q| + tmax).
// and 1 % on top for the fp32 evaluation of the bound itself.
__device__ __forceinline__ float row_eps(float nqs, float tms, int kp, float c, float chain, float last) {
  const float K = (float)kp;
  float e = (9.765625e-4f + 9.5367431640625e-7f) * nqs * tms;
  e += 6.103515625e-5f * sqrtf(K) * (nqs + tms) * 1.001f;
  e += K * 3.725290298461914e-9f;
  e += K * 2.384185791015625e-7f * (nqs * tms * 1.001f + 256.f * c);
  e += 3.f * 6.103515625e-5f * c;
  e += (K + 2.f) * 5.9604644775390625e-8f * chain;
  e += 1.1920928955078125e-7f * last;
  return e * 1.01f;
}

// ---- target image ---------------------------------------------------------------------------------
struct PrepArgs {
  kge_model_t m;
  int64_t n_targets;
  int parts, kp, dist, tn;
  float* tn2;        // [n_targets] squared norms (scratch inside the image buffer's tail)
  float* header;     // {tmax, max |t_c|, max |t|^2}
  uint16_t* tiles;   // [n_tiles][kp/8][tn][8] fp16
};

__global__ void __launch_bounds__(256) target_norm_kernel(const PrepArgs a) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  const int d = a.m.d;
  float wmax = 0.f, amax = 0.f;
  for (int64_t j = warp; j < a.n_targets; j += n_warps) {
    float s = 0.f;
    for (int p = 0; p < a.parts; ++p)
      for (int c = lane; c < d; c += 32) {
        const float x = __ldg(a.m.entity.w[p] + j * d + c);
        s = fmaf(x, x, s);
        amax = fmaxf(amax, fabsf(x));
      }
    s = warp_sum(s);
    if (lane == 0) a.tn2[j] = s;
    wmax = fmaxf(wmax, s);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, o));
  // non-negative floats order like their bit patterns (the header is zeroed by the caller)
  if (lane == 0 && wmax > 0.f) {
    atomicMax(reinterpret_cast<int*>(a.header), __float_as_int(sqrtf(wmax) * 1.0001f));
    atomicMax(reinterpret_cast<int*>(a.header) + 1, __float_as_int(amax));
    atomicMax(reinterpret_cast<int*>(a.header) + 2, __float_as_int(wmax));
  }
}

__global__ void __launch_bounds__(256) target_image_kernel(const PrepArgs a) {
  const int d = a.m.d;
  const int tn = a.tn;
  const int kchunks = a.kp / 8;
  const int64_t n_tiles = (a.n_targets + tn - 1) / tn;
  const int64_t total = n_tiles * kchunks * tn;
  const int kd = a.parts * d;
  const ImgScale sc = img_scale(a.header);
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (int64_t)gridDim.x * blockDim.x) {
    const int r = (int)(idx % tn);
    const int kc = (int)((idx / tn) % kchunks);
    const int64_t tile = idx / ((int64_t)tn * kchunks);
    const int64_t j = tile * tn + r;
    uint16_t out[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const int k = kc * 8 + e;
      float x = 0.f;
      if (j < a.n_targets) {
        if (k < kd) {
          const int p = k / d, c = k - p * d;
          x = __ldg(a.m.entity.w[p] + j * d + c);
          out[e] = f16_bits(scalbnf(x, sc.e_t));
          continue;
        }
        if (a.dist && k < kd + 3) {  // fp16 hi / mid / lo of W = -||t||^2 / 2 * 2^e_w
          const float s = scalbnf(-0.5f * a.tn2[j], sc.e_w);
          const float hi = f16_back(f16_bits(s));
          const float mid = f16_back(f16_bits(s - hi));
          x = (k == kd) ? hi : (k == kd + 1 ? mid : (s - hi - mid));
        }
      }
      out[e] = f16_bits(x);
    }
    uint4 v;
    v.x = out[0] | ((uint32_t)out[1] << 16);
    v.y = out[2] | ((uint32_t)out[3] << 16);
    v.z = out[4] | ((uint32_t)out[5] << 16);
    v.w = out[6] | ((uint32_t)out[7] << 16);
    reinterpret_cast<uint4*>(a.tiles)[idx] = v;
  }
}

// ---- sweep kernel ------------------------------------------------------------------------------------
struct MmaArgs {
  ScoreArgs s;
  int64_t n_targets;
  int64_t n_tiles;
  int64_t rows_pad;       // n rounded up to MM: stride of the per-split arrays
  int tiles_per_split;
  int parts, kp, dist, stages;
  int kc, nkc;            // K columns per ring stage (a multiple of 16) and stages per tile: kc = kp, nkc = 1 unless K is
                          // too large for whole tiles in shared memory
  const float* header;
  const uint16_t* tiles;
  const int64_t* hist_off;
  const int64_t* hist_items;
  int mask_first;
  int k;
  uint2* cand;        // [splits][rows_pad][CAND]: {group maximum bits, group id | flags}
  int32_t* cand_cnt;  // [splits][rows_pad]: entries, or -1 when the list could not be compacted
  float* cand_thr;    // [splits][rows_pad]: threshold the list was last compacted with (-inf: never)
  float* eps_out;     // [rows_pad] error bound of the row, in the row's scaled units
  float* inv_scale_out;  // [rows_pad] 1 / S_i (a power of two): scaled approximate score -> score
  const uint32_t* unsafe_bits;  // [rows_pad][unsafe_wpr]: bit c = chunk c holds a masked / out-of-range target
  int64_t unsafe_wpr;
  float* dbg_out;     // optional dense approximate scores [n, dbg_stride]
  int64_t dbg_stride;
};

// Entry of a row's candidate list = one 32-target chunk of the sweep: x = maximum of the chunk's
// groups that cleared the threshold (fp32 bits) = the chunk maximum; y = mask of those groups (bits
// 0..7), chunk id (bits 8..28), bit 30 = "safety known", bit 31 = "unsafe" (the chunk holds a masked
// or out-of-range target, so its maximum must not feed the threshold).  Safety is resolved lazily, at
// compaction time, by the whole warp (one binary search per lane instead of one per push).
constexpr int CH = 32;  // targets per chunk = one tcgen05.ld.x32 = 8 groups
constexpr uint32_t CID_SHIFT = 8, CID_MASK = 0x1FFFFFu, F_KNOWN = 0x40000000u, F_UNSAFE = 0x80000000u;

__device__ __forceinline__ uint32_t orderable(float x) {
  const uint32_t b = __float_as_uint(x);
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float from_orderable(uint32_t b) {
  return __uint_as_float((b & 0x80000000u) ? (b & 0x7FFFFFFFu) : ~b);
}

struct MaskInfo {
  const int64_t* hist_items;
  int64_t h_lo, h_hi;
  int64_t n_targets;
  int mask_first;
};

// k-th largest of the warp's keys (NQ per lane, 0 = absent; all present keys are > 0), or 0 when fewer
// than k are present.  Radix descent on the order-preserving bit pattern that stops as soon as
// exactly k keys remain above the prefix (their minimum is the answer).
template <int NQ>
__device__ __forceinline__ uint32_t warp_kth_largest(const uint32_t (&key)[NQ], int k) {
  int n_t = 0;
  uint32_t k_or = 0u, k_and = 0xFFFFFFFFu;
#pragma unroll
  for (int q = 0; q < NQ; ++q) {
    n_t += __popc(__ballot_sync(0xffffffffu, key[q] != 0u));
    k_or |= key[q];
    if (key[q] != 0u) k_and &= key[q];
  }
  if (n_t < k) return 0u;
  // the keys of a list sit in a narrow band: the descent starts at the highest bit in which they differ
  k_or = __reduce_or_sync(0xffffffffu, k_or);
  k_and = __reduce_and_sync(0xffffffffu, k_and);
  const uint32_t diff = k_or ^ k_and;
  if (diff == 0u) return k_or;   // all present keys are equal
  const int top = 31 - __clz(diff);
  uint32_t P = top == 31 ? 0u : (k_and & ~((2u << top) - 1u));  // invariant: #(key >= max(P, 1)) = n_t >= k
  for (int bit = top; bit >= 0 && n_t > k; --bit) {
    const uint32_t c = P | (1u << bit);
    int n = 0;
#pragma unroll
    for (int q = 0; q < NQ; ++q) n += __popc(__ballot_sync(0xffffffffu, key[q] >= c));
    if (n >= k) {
      P = c;
      n_t = n;
    }
  }
  const uint32_t T = P ? P : 1u;
  uint32_t mn = 0xFFFFFFFFu;
#pragma unroll
  for (int q = 0; q < NQ; ++q)
    if (key[q] >= T) mn = min(mn, key[q]);
  return __reduce_min_sync(0xffffffffu, mn);
}

// Warp-cooperative compaction of one row's candidate list: tau = k-th largest maximum among the
// safe chunks, keep every entry >= tau - 2 eps.  Returns the new count (lane-uniform), -1 when the
// list cannot be shrunk enough to take `room` more entries; thr_out = new threshold.
__device__ __noinline__ int compact_row(uint2* buf, int cnt, int k, float eps, const uint32_t* unsafe_row, int room,
                                        float* thr_out) {
  const int lane = threadIdx.x & 31;
  uint2 e[CAND / 32];
  bool valid[CAND / 32];
  uint32_t key[CAND / 32];
  uint32_t word[CAND / 32];
#pragma unroll
  for (int q = 0; q < CAND / 32; ++q) {   // all loads first: one memory latency per compaction
    const int i = q * 32 + lane;
    valid[q] = i < cnt;
    e[q] = valid[q] ? buf[i] : make_uint2(0u, 0u);
  }
#pragma unroll
  for (int q = 0; q < CAND / 32; ++q) {
    const uint32_t cid = (e[q].y >> CID_SHIFT) & CID_MASK;
    word[q] = (valid[q] && !(e[q].y & F_KNOWN)) ? __ldg(unsafe_row + (cid >> 5)) : 0u;
  }
#pragma unroll
  for (int q = 0; q < CAND / 32; ++q) {
    const uint32_t cid = (e[q].y >> CID_SHIFT) & CID_MASK;
    if (valid[q] && !(e[q].y & F_KNOWN)) e[q].y |= F_KNOWN | (((word[q] >> (cid & 31u)) & 1u) ? F_UNSAFE : 0u);
    key[q] = (valid[q] && !(e[q].y & F_UNSAFE)) ? orderable(__uint_as_float(e[q].x)) : 0u;  // orderable() > 0
  }
  const uint32_t T = warp_kth_largest<CAND / 32>(key, k);
  const float tau = T ? from_orderable(T) : -INFINITY;
  const float thr = tau - 2.f * eps;
  __syncwarp();
  int base = 0;
#pragma unroll
  for (int q = 0; q < CAND / 32; ++q) {
    const bool keep = valid[q] && __uint_as_float(e[q].x) >= thr;
    const unsigned b = __ballot_sync(0xffffffffu, keep);
    if (keep) buf[base + __popc(b & ((1u << lane) - 1u))] = e[q];
    base += __popc(b);
  }
  __syncwarp();
  *thr_out = thr;
  return (base > CAND - room) ? -1 : base;
}

// Bitmap of the chunks a row must not trust for its threshold: chunks with a history item, the
// [PAD] chunk, the partial last chunk and the padding chunks behind it (their entries are dropped by the
// rescore kernel, which never scores a target id >= n_targets).  One warp per row; the buffer is zeroed by the caller.
__global__ void __launch_bounds__(256) unsafe_bitmap_kernel(uint32_t* bits, int64_t wpr, int64_t n, int64_t n_targets,
                                                            int64_t n_chunks, const int64_t* hist_off,
                                                            const int64_t* hist_items, int mask_first) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t row = warp; row < n; row += n_warps) {
    uint32_t* b = bits + row * wpr;
    if (hist_off) {
      const int64_t lo = hist_off[row], hi = hist_off[row + 1];
      for (int64_t i = lo + lane; i < hi; i += 32) {
        const int64_t c = hist_items[i] / CH;
        if (c >= 0 && (c >> 5) < wpr) atomicOr(b + (c >> 5), 1u << (c & 31));
      }
    }
    if (lane == 0 && mask_first) atomicOr(b, 1u);
    // the partial last chunk and the chunks of zero rows that pad the last tile of the image
    for (int64_t c = n_targets / CH + lane; c < n_chunks; c += 32) atomicOr(b + (c >> 5), 1u << (c & 31));
  }
}

// Filter state of one (row, split, slice) list.  widx = index of the next free entry in the global `cand` array
// (list base + count: lists are CAND entries long and CAND-aligned, and a count never reaches CAND).
struct EpiState {
  float thr;       // +inf: the row collects nothing (inactive, not representable, or its list overflowed)
  uint32_t widx;
};
constexpr int TRIG = CAND - 5;   // a list is compacted when it holds more than TRIG entries at the end of a tile

// One chunk (32 columns = 8 groups of 4) of one row, in two steps so that the registers of the chunk are free for
// the next tcgen05.ld as early as possible: the group maxima and the chunk maximum ...
__device__ __forceinline__ float chunk_reduce(const uint32_t (&r)[32], float (&gm)[8]) {
#pragma unroll
  for (int g = 0; g < 8; ++g)
    gm[g] = fmaxf(max3f(__uint_as_float(r[4 * g]), __uint_as_float(r[4 * g + 1]), __uint_as_float(r[4 * g + 2])),
                  __uint_as_float(r[4 * g + 3]));
  return fmaxf(max3f(gm[0], gm[1], gm[2]), max3f(max3f(gm[3], gm[4], gm[5]), gm[6], gm[7]));
}
// ... and (rarely) one list entry.
// The entry is born without its safety flag (F_KNOWN clear): whoever needs it -- the next compaction of the list, or
// the rescore kernel -- reads one word of the row's "unsafe chunk" bitmap.  Carrying the bitmap through the sweep
// (round 1) cost three live registers and ~13 ALU-pipe instructions per tile in a loop that is bound by exactly
// that pipe (FMNMX / FSETP / IADD / LOP3 issue every other cycle per scheduler: B300_MICROARCH "pipe rates").
__device__ __forceinline__ void chunk_push(const float (&gm)[8], float tm, EpiState& st, uint32_t cid8,
                                           uint2* __restrict__ cand) {
  if (tm >= st.thr) {  // rare per row after the first tiles (but most warps have one such row per chunk)
    // Group mask from sign bits: gm - thr on the FMA pipe, one funnel shift per group on the ALU pipe (a compare
    // plus a predicated add per group costs twice the ALU slots).  acc collects "below the threshold" bits, first
    // group in the highest position: mask bit (7 - g) <=> group g cleared the threshold.
    uint32_t acc = 0u;
#pragma unroll
    for (int g = 0; g < 8; ++g) {
      const uint32_t d = __float_as_uint(__fsub_rn(gm[g], st.thr));   // sign bit set <=> gm < thr (gm == thr: +0)
      asm("shf.l.wrap.b32 %0, %1, %0, 1;" : "+r"(acc) : "r"(d));
    }
    const uint32_t y = cid8 | (~acc & 0xFFu);
    cand[st.widx] = make_uint2(__float_as_uint(tm), y);
    ++st.widx;
  }
}

// TN targets per tile (one MMA instruction covers 128 rows x TN targets x 16 of K), NBUF accumulator buffers per
// half.  TMEM columns = NH * TN * NBUF: (2, 128, 1), (2, 64, 2) and (1, 128, 2) take 256, (2, 128, 2) all 512.
// NCOL column slices per tile: the 128 rows of a half are covered by NCOL warps per quadrant, each filtering
// TN / NCOL columns into its own list (a row then owns splits * NCOL lists, merged by the rescore kernel).
// NMMA issuer warps: 2 = one per row half (needed when the CTA has the SM to itself), 1 = one warp for both.
// NH row halves per CTA (MM = 128 * NH query rows).  NH = 1 is the large-K shape: the queries of 256 rows no longer fit
// shared memory next to a tile ring, so a CTA keeps 128 rows and the tiles stream through the ring in K chunks.
template <int NH, int TN, int NBUF, int NCOL, int NMMA, bool DBG>
__global__ void __launch_bounds__(sweep_threads(NH, NCOL, NMMA), (NBUF == 1 && NH == 2) ? 2 : 1)
    fullsort_mma_kernel(const MmaArgs a) {
  constexpr int MM = MH * NH;
  constexpr int ROOM = 16;              // list room demanded after a compaction
  constexpr int NCH = TN / CH / NCOL;   // chunks of 32 columns per tile and epilogue thread
  constexpr int EPI_WARPS = 4 * NH * NCOL, PRODUCER_WARP = EPI_WARPS, MMA_WARP0 = EPI_WARPS + PRODUCER_WARPS;
  constexpr int N_WARPS = EPI_WARPS + PRODUCER_WARPS + NMMA;
  constexpr uint32_t TMEM_COLS = NH * TN * NBUF;
  static_assert(NMMA <= NH, "one issuer warp per row half at most");
  static_assert(NCH % 2 == 0 && (NBUF == 1 || NBUF == 2), "the chunk pipeline alternates two register sets");
  static_assert(TRIG + NCH < CAND, "a list below the trigger takes one more tile's appends without reaching CAND");
  constexpr uint32_t IDESC = make_idesc(TN);
  extern __shared__ __align__(128) unsigned char smem[];
  const int kp = a.kp;
  const uint32_t a_bytes = (uint32_t)MM * kp * 2;
  const uint32_t b_bytes = (uint32_t)TN * kp * 2;          // one tile of the image
  const uint32_t s_bytes = (uint32_t)TN * a.kc * 2;        // one ring stage: kc K columns of a tile
  uint16_t* As = reinterpret_cast<uint16_t*>(smem);
  unsigned char* Bs = smem + a_bytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(Bs + (size_t)a.stages * s_bytes);
  // bars: full[stages], empty[stages], tfull[buf][half] (4), tempty[buf][half] (4)
  float* eps_row = reinterpret_cast<float*>(bars + 2 * a.stages + 8);  // [MM]
  float* inv_row = eps_row + MM;                                        // [MM] 1 / S_i
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(inv_row + MM);

  // (the shuffle tells the compiler that the warp index is warp-uniform: TMEM addresses, barrier addresses and the
  // role tests then live in uniform registers instead of the 96 vector registers the epilogue is short of)
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
  const int64_t row0 = (int64_t)blockIdx.x * MM;
  const int nrows = (int)min((int64_t)MM, a.s.n - row0);
  const int split = blockIdx.y;
  const int64_t t0 = (int64_t)split * a.tiles_per_split;
  const int64_t t1 = min(a.n_tiles, t0 + a.tiles_per_split);
  const int64_t nt = t1 - t0;
  const int d = a.s.m.d;
  const int kd = a.parts * d;

  // ---- setup: zero A, build the scaled fp16 queries, barriers, TMEM ---------------------------------
  for (uint32_t i = threadIdx.x; i < a_bytes / 16; i += blockDim.x) reinterpret_cast<uint4*>(As)[i] = make_uint4(0, 0, 0, 0);
  __syncthreads();
  const ImgScale isc = img_scale(a.header);
  // one fp32 query row per warp, staged in the (still idle) tile ring: the row's scale needs its largest element
  float* scratch = reinterpret_cast<float*>(Bs) + warp * kp;
  for (int u = warp; u < MM; u += N_WARPS) {
    float nq = 0.f, amax = 0.f;
    if (u < nrows) {
      for (int c = lane; c < d; c += 32) {
        float q0, q1;
        query_value(a.s, row0 + u, c, q0, q1);
        nq = fmaf(q0, q0, nq);
        amax = fmaxf(amax, fabsf(q0));
        scratch[c] = q0;
        if (a.parts == 2) {
          nq = fmaf(q1, q1, nq);
          amax = fmaxf(amax, fabsf(q1));
          scratch[d + c] = q1;
        }
      }
    }
    nq = warp_sum(nq);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, o));
    int e_i = amax > 0.f ? clamp_exp(7 - ilogbf(amax)) : 0;   // largest |q_c| 2^e_i in [2^7, 2^8)
    int e_c = 0;
    bool bad = !(nq < INFINITY);                              // inf / nan in the query: exact path
    if (a.dist) {
      e_c = e_i + isc.e_t - isc.e_w;                          // c_i = 2^e_c must be a normal fp16 number
      if (e_c > 15) {
        e_i -= e_c - 15;                                      // lower the row's scale (never raise it: no overflow)
        e_c = 15;
      }
      if (e_c < -14 || e_i < -E_CLAMP) bad = true;
    }
    __syncwarp();
    if (u < nrows && !bad) {
      for (int k1 = lane; k1 < kd; k1 += 32)
        As[((size_t)(k1 >> 3) * MM + u) * 8 + (k1 & 7)] = f16_bits(scalbnf(scratch[k1], e_i));
      if (a.dist && lane < 3) {
        const int k1 = kd + lane;
        As[((size_t)(k1 >> 3) * MM + u) * 8 + (k1 & 7)] = f16_bits(scalbnf(1.0f, e_c));
      }
    }
    if (lane == 0) {
      const float nqs = scalbnf(sqrtf(nq) * 1.0001f, e_i), tms = scalbnf(isc.tmax, isc.e_t);
      // S (|q| + tmax)^2 = ((|q| + tmax) 2^e_i) ((|q| + tmax) 2^e_t)
      const float qt_i = nqs + scalbnf(isc.tmax, e_i);   // (|q| + tmax) 2^e_i
      const float chain = a.dist ? 0.5f * qt_i * (scalbnf(sqrtf(nq) * 1.0001f, isc.e_t) + tms) : nqs * tms;
      const float last = a.s.m.model == KGE_ROTATE ? fabsf(a.s.m.margin) * scalbnf(qt_i, isc.e_t) : 0.f;
      const float eps = bad ? INFINITY : row_eps(nqs, tms, kp, a.dist ? scalbnf(1.0f, e_c) : 0.f, chain, last);
      const float inv = scalbnf(1.0f, -(e_i + isc.e_t));
      eps_row[u] = eps;
      inv_row[u] = inv;
      a.eps_out[row0 + u] = eps;        // (every split writes the same values)
      a.inv_scale_out[row0 + u] = inv;
    }
    __syncwarp();   // the scratch row is reused by the warp's next query
  }
  if (threadIdx.x == 0) {
    for (int s = 0; s < a.stages; ++s) {
      mbar_init(smem_u32(&bars[s]), 1);              // full: producer's expect_tx arrive
      mbar_init(smem_u32(&bars[a.stages + s]), NMMA);   // empty: one tcgen05.commit per MMA warp
    }
    for (int x = 0; x < 4; ++x) {
      mbar_init(smem_u32(&bars[2 * a.stages + x]), 1);      // tfull[buf][half]: one commit
      mbar_init(smem_u32(&bars[2 * a.stages + 4 + x]), 4 * NCOL);  // tempty[buf][half]: the epilogue warps of the half
    }
    fence_mbar_init();
  }
  if (warp == MMA_WARP0) {
    tmem_alloc(smem_u32(tmem_slot), TMEM_COLS);
    tmem_relinquish();
  }
  fence_proxy_async();  // the generic-proxy writes of A must be visible to the tensor core (async proxy)
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t full0 = smem_u32(&bars[0]), empty0 = smem_u32(&bars[a.stages]);
  const uint32_t tfull0 = smem_u32(&bars[2 * a.stages]), tempty0 = smem_u32(&bars[2 * a.stages + 4]);

  if (warp == PRODUCER_WARP) {
    // ===== producer: stream target tiles into the ring, one K chunk per stage (uniform control flow, one elected
    // lane issues).  A chunk [kc K columns][TN rows] of a tile is contiguous in the image.
    const bool leader = elect_one();
    int s = 0;
    uint32_t ph = 0;
    const unsigned char* src = reinterpret_cast<const unsigned char*>(a.tiles) + (size_t)t0 * b_bytes;
    const uint32_t bs0 = smem_u32(Bs);
    for (int64_t i = 0; i < nt; ++i) {
      for (int j = 0; j < a.nkc; ++j) {
        const int kcols = min(a.kc, kp - j * a.kc);
        const uint32_t bytes = (uint32_t)TN * kcols * 2;
        mbar_wait(empty0 + 8 * s, ph ^ 1u);
        if (leader) {
          mbar_arrive_expect_tx(full0 + 8 * s, bytes);
          bulk_g2s(bs0 + (uint32_t)s * s_bytes, src + (size_t)i * b_bytes + (size_t)j * s_bytes, bytes, full0 + 8 * s);
        }
        __syncwarp();
        if (++s == a.stages) {
          s = 0;
          ph ^= 1u;
        }
      }
    }
  } else if (warp >= MMA_WARP0) {
    // ===== MMA issuers, one warp per row half (or one for both): the warp runs the loop with uniform control flow
    // (descriptors live in uniform registers), one elected lane issues.  Only the 14-bit start-address field of a
    // descriptor changes.
    const bool leader = elect_one();
    const uint32_t a_lbo = MM * 16, b_lbo = TN * 16;
    const uint32_t desc_hi = (128u >> 4) | (1u << 14);   // SBO = 128 B, descriptor version 1
    const uint32_t a_lo0 = ((smem_u32(As) >> 4) & 0x3FFFu) | ((a_lbo >> 4) << 16);
    const uint32_t b_lo0 = ((smem_u32(Bs) >> 4) & 0x3FFFu) | ((b_lbo >> 4) << 16);
    const uint32_t a_kstep = (2 * a_lbo) >> 4, b_kstep = (2 * b_lbo) >> 4, a_hstep = (128 * 16) >> 4;
    const uint32_t b_sstep = s_bytes >> 4;
    const int h_lo = NMMA == NH ? warp - MMA_WARP0 : 0, h_hi = NMMA == NH ? h_lo + 1 : NH;
    int s = 0;
    uint32_t ph = 0;
    for (int64_t i = 0; i < nt; ++i) {
      const uint32_t buf = NBUF == 1 ? 0u : (uint32_t)(i & 1);
      const uint32_t tph = (uint32_t)((i / NBUF) & 1);
      for (int j = 0; j < a.nkc; ++j) {
        const int ksteps = min(a.kc, kp - j * a.kc) / 16;
        const int ks0 = j * (a.kc / 16);                    // K step of the tile this chunk starts at
        mbar_wait(full0 + 8 * s, ph);                       // chunk landed
        const uint32_t b_lo = b_lo0 + (uint32_t)s * b_sstep;
        for (int h = h_lo; h < h_hi; ++h) {
          if (j == 0) mbar_wait(tempty0 + 8 * (buf * 2 + h), tph ^ 1u);  // the half's epilogue warps have drained this accumulator
          tc_fence_after();
          if (leader) {
            const uint32_t dcol = tmem_base + (buf * NH + h) * TN;
            const uint32_t a_lo = a_lo0 + (uint32_t)h * a_hstep + (uint32_t)ks0 * a_kstep;
            for (int ks = 0; ks < ksteps; ++ks) {
              const uint64_t adesc = ((uint64_t)desc_hi << 32) | (a_lo + (uint32_t)ks * a_kstep);
              const uint64_t bdesc = ((uint64_t)desc_hi << 32) | (b_lo + (uint32_t)ks * b_kstep);
              umma_f16(dcol, adesc, bdesc, IDESC, (ks0 + ks) > 0 ? 1u : 0u);
            }
            if (j == a.nkc - 1) umma_commit(tfull0 + 8 * (buf * 2 + h));   // this half's accumulator is ready
            if (h == h_hi - 1) umma_commit(empty0 + 8 * s);                // stage reusable once its MMAs have read it
          }
        }
        __syncwarp();
        if (++s == a.stages) {
          s = 0;
          ph ^= 1u;
        }
      }
    }
  } else {
    // ===== epilogue =====
    const int quad = warp & 3;   // == warp % 4: the TMEM lane quadrant this warp may read
    // Compaction of the lists of this warp's rows that are (nearly) full; `st` is the lane's list of row `u`.
    auto compact_full = [&](EpiState& st, int u, int64_t lsplit, int trig) {
      const uint32_t wbase = (uint32_t)((lsplit * a.rows_pad + row0 + u) * CAND);
      unsigned full = __ballot_sync(0xffffffffu, (int)(st.widx & (CAND - 1)) > trig);
      while (full) {
        const int r = __ffs(full) - 1;
        full &= full - 1;
        const int cnt_r = __shfl_sync(0xffffffffu, (int)(st.widx & (CAND - 1)), r);
        const int u_r = u - lane + r;
        const float eps_r = eps_row[u_r];
        const int64_t qrow_r = row0 + u_r;
        uint2* buf_r = a.cand + (lsplit * a.rows_pad + qrow_r) * CAND;
        __syncwarp();
        float thr_new;
        const int n_new = compact_row(buf_r, cnt_r, a.k, eps_r, a.unsafe_bits + qrow_r * a.unsafe_wpr, ROOM, &thr_new);
        if (lane == r) {
          if (n_new < 0) {
            st.thr = INFINITY;  // stop collecting: the row goes to the exact path
            st.widx = wbase;
          } else {
            st.widx = wbase + (uint32_t)n_new;
            st.thr = thr_new;
          }
        }
      }
    };
    auto init_state = [&](EpiState& st, int u, int64_t lsplit) {
      const bool usable = u < nrows && eps_row[u] < INFINITY;   // rows the fp16 scaling cannot hold: exact path
      st.thr = usable ? -INFINITY : INFINITY;
      st.widx = (uint32_t)((lsplit * a.rows_pad + row0 + u) * CAND);
    };
    auto store_state = [&](const EpiState& st, int u, int64_t lsplit) {
      if (u < nrows) {   // (a list's threshold starts at -inf and only ever rises to finite values)
        const int64_t lrow = lsplit * a.rows_pad + row0 + u;
        a.cand_cnt[lrow] = st.thr == INFINITY ? -1 : (int)(st.widx - (uint32_t)(lrow * CAND));
        a.cand_thr[lrow] = st.thr;
      }
    };
    auto dump = [&](const uint32_t (&r)[32], int u, uint32_t cid) {   // debug: unscaled approximate scores
      if (DBG && u < nrows) {
        const float inv = inv_row[u];
        float* o = a.dbg_out + (row0 + u) * a.dbg_stride + (int64_t)cid * CH;
#pragma unroll
        for (int j = 0; j < CH; ++j) o[j] = __uint_as_float(r[j]) * inv;
      }
    };
    const int nti = (int)nt;
    uint32_t va[32], vb[32];
    float gm[8], gm2[8];

    {
      // ---- one warp = (row half, lane quadrant, column slice) -------------------------------------------------
      const int h = NH == 2 ? (warp >> 2) & 1 : 0;
      const int cs = warp / (4 * NH);                   // column slice of the tile
      const int64_t lsplit = (int64_t)split * NCOL + cs;   // list index of this (target split, column slice)
      const int u = h * 128 + quad * 32 + lane;
      EpiState st;
      init_state(st, u, lsplit);
      // (warp-uniform: these live in uniform registers)
      const uint32_t tlane = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(h * TN + cs * NCH * CH);
      const uint32_t my_tfull = tfull0 + 8 * h, my_tempty = tempty0 + 8 * h;   // + 16 * buf
      auto process = [&](const uint32_t (&r)[32], uint32_t cid) {
        dump(r, u, cid);
        const float tm = chunk_reduce(r, gm);
        chunk_push(gm, tm, st, cid << CID_SHIFT, a.cand);   // (targets beyond the table: zero rows, chunks marked unsafe)
      };
      uint32_t cid = (uint32_t)(t0 * (TN / CH) + cs * NCH);
      if constexpr (NBUF == 1) {
        static_assert(NCH == 4, "one accumulator per half: a tile is read as two batches of two chunks");
        // One accumulator per half: what bounds the sweep is how long an accumulator stays away from the tensor
        // core, i.e. the number of TMEM round trips between "tile ready" and "tile in registers".  Chunk by chunk
        // that is four latencies per tile (measured: MMAs alone 1.21 ms, filter alone 0.98 ms, together 2.23 ms --
        // the two never overlapped); here the tile is read as two batches of two chunks (both register sets in
        // flight), the second batch requested as soon as the max trees have consumed the first: two round trips,
        // and the MMAs of the next tile run under the filter of the second batch.
        mbar_wait(my_tfull, 0u);
        tc_fence_after();
        tmem_ld32_issue(tlane, va);
        tmem_ld32_issue(tlane + CH, vb);
        for (int i = 0; i < nti; ++i, cid += TN / CH) {
          // While the accumulator is held only what frees the registers runs (the two max trees: 40 ALU-pipe
          // instructions); the appends of the first batch wait until the accumulator is back with the tensor core.
          tmem_ld_wait2(va, vb);
          dump(va, u, cid);
          const float tma = chunk_reduce(va, gm);
          tmem_ld32_issue(tlane + 2 * CH, va);
          dump(vb, u, cid + 1);
          const float tmb = chunk_reduce(vb, gm2);
          tmem_ld32_issue(tlane + 3 * CH, vb);
          tmem_ld_wait2(va, vb);
          tc_fence_before();   // every chunk of the tile is in registers: release the accumulator
          __syncwarp();
          if (lane == 0) mbar_arrive(my_tempty);
          chunk_push(gm, tma, st, cid << CID_SHIFT, a.cand);
          chunk_push(gm2, tmb, st, (cid + 1) << CID_SHIFT, a.cand);
          process(va, cid + 2);
          process(vb, cid + 3);
          compact_full(st, u, lsplit, TRIG);
          if (i + 1 < nti) {   // computed while the second batch was filtered
            mbar_wait(my_tfull, (uint32_t)((i + 1) & 1));
            tc_fence_after();
            tmem_ld32_issue(tlane, va);
            tmem_ld32_issue(tlane + CH, vb);
          }
        }
      } else {
        static_assert(NBUF == 2, "the chunk pipeline alternates two accumulators");
        // Two accumulators per half, software pipeline over chunks: the load of the next chunk is in flight while the
        // current one is filtered, and an accumulator goes back to the tensor core as soon as its last chunk sits in
        // registers (the MMAs of the next tile already run in the other buffer).
        mbar_wait(my_tfull, 0u);
        tc_fence_after();
        tmem_ld32_issue(tlane, va);
        tmem_ld_wait(va);
        for (int i = 0; i < nti; ++i, cid += TN / CH) {
          const uint32_t buf = (uint32_t)(i & 1);
          const uint32_t tbase = tlane + buf * NH * TN;
#pragma unroll
          for (int c = 0; c < NCH; ++c) {
            uint32_t(&cur)[32] = (c & 1) ? vb : va;
            uint32_t(&nxt)[32] = (c & 1) ? va : vb;
            if (c + 1 < NCH) {
              tmem_ld32_issue(tbase + (uint32_t)((c + 1) * CH), nxt);
              process(cur, cid + c);
              tmem_ld_wait(nxt);
              if (c + 1 == NCH - 1) {   // every chunk of the tile is in registers: release the accumulator
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(my_tempty + 16 * buf);
              }
            } else {
              if (i + 1 < nti) {
                const uint32_t nbuf = buf ^ 1u;
                mbar_wait(my_tfull + 16 * nbuf, (uint32_t)(((i + 1) / 2) & 1));
                tc_fence_after();
                tmem_ld32_issue(tlane + nbuf * NH * TN, nxt);
              }
              process(cur, cid + c);
              if (i + 1 < nti) tmem_ld_wait(nxt);
            }
          }
          compact_full(st, u, lsplit, TRIG);
        }
      }
      store_state(st, u, lsplit);
    }
  }

  // ---- teardown ------------------------------------------------------------------------------------
  tc_fence_before();
  __syncthreads();
  if (warp == MMA_WARP0) tmem_dealloc(tmem_base, TMEM_COLS);
}

// ---- exact re-score + top-k ------------------------------------------------------------------------------
struct RescoreArgs {
  ScoreArgs s;
  int64_t n_targets;
  int64_t rows_pad;
  int splits, nent;
  int parts;
  const int64_t* hist_off;
  const int64_t* hist_items;
  int mask_first;
  int k;
  const uint2* cand;
  const int32_t* cand_cnt;
  const float* cand_thr;
  const float* eps;         // scaled units of the row
  const float* inv_scale;   // 1 / S_i
  int64_t* ids_out;
  float* scores_out;
  int32_t* row_flags;
  const uint32_t* unsafe_bits;   // [rows_pad][unsafe_wpr] the sweep's bitmap (entries may come without their flag)
  int64_t unsafe_wpr;
  int32_t* row_map;      // rows handed to the exact kernel, in arrival order ...
  int32_t* exact_rows;   // ... and their count (zeroed by the caller)
};

constexpr int RS_WARPS = 8;
constexpr int RS_GIDS = 256;               // group ids expanded per batch of 32 entries
constexpr int RS_HIST = 256;               // history items staged in shared memory (longer ones stay in global)
constexpr int RS_KEYS = 64;                // exact keys staged before they are ordered

// nent = entries a row can bring (splits * CAND, at least RS_GIDS so that kbuf also holds a batch of group ids)
__host__ __device__ inline size_t rescore_smem_per_warp(int kd, int nent) {
  return ((size_t)kd * 4 + 15) / 16 * 16 + (size_t)nent * 8 + (size_t)nent * 4 + (size_t)RS_HIST * 4 +
         (size_t)RS_KEYS * 8 + (size_t)32 * 8;
}

// 32 keys, one per lane, sorted descending across the warp (bitonic network).
__device__ __forceinline__ uint64_t warp_sort_desc(uint64_t key, int lane) {
#pragma unroll
  for (int k2 = 2; k2 <= 32; k2 <<= 1) {
#pragma unroll
    for (int j = k2 >> 1; j > 0; j >>= 1) {
      const uint64_t other = __shfl_xor_sync(0xffffffffu, key, j);
      const bool desc_block = (lane & k2) == 0;
      const bool lower = (lane & j) == 0;
      const bool take_max = lower == desc_block;
      key = take_max ? (key > other ? key : other) : (key < other ? key : other);
    }
  }
  return key;
}

template <bool DIST>
__global__ void __launch_bounds__(RS_WARPS * 32, 2) rescore_topk_kernel(const RescoreArgs a) {
  extern __shared__ __align__(128) unsigned char smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int d = a.s.m.d;
  const int kd = a.parts * d;
  const int k = a.k;
  // per warp: q[kd] | ent[nent] {value, chunk|mask|flags} | kbuf[nent] keys / group ids | hist | keys | list
  unsigned char* base = smem + warp * rescore_smem_per_warp(kd, a.nent);
  float* q = reinterpret_cast<float*>(base);
  uint2* ent = reinterpret_cast<uint2*>(base + ((size_t)kd * 4 + 15) / 16 * 16);
  uint32_t* kbuf = reinterpret_cast<uint32_t*>(ent + a.nent);
  uint32_t* hist = kbuf + a.nent;
  uint64_t* keys = reinterpret_cast<uint64_t*>(hist + RS_HIST);
  uint64_t* list = keys + RS_KEYS;
  const float margin = (a.s.m.model == KGE_ROTATE) ? a.s.m.margin : 0.f;

  for (int64_t row = (int64_t)blockIdx.x * RS_WARPS + warp; row < a.s.n; row += (int64_t)gridDim.x * RS_WARPS) {
    // ---- gather the row's lists ------------------------------------------------------------------------
    // The kernel is a chain of dependent L2 round trips per row (one warp per row): everything that only depends
    // on the row index is requested first, in one go -- lane s takes the count and threshold of list s.
    int my_cnt = 0;
    float my_thr = -INFINITY;
    if (lane < a.splits) {
      const int64_t lrow = (int64_t)lane * a.rows_pad + row;
      my_cnt = __ldg(a.cand_cnt + lrow);
      my_thr = __ldg(a.cand_thr + lrow);
    }
    int64_t h_lo = 0, h_hi = 0;
    if (a.hist_off) {
      h_lo = __ldg(a.hist_off + row);
      h_hi = __ldg(a.hist_off + row + 1);
    }
    const float eps = __ldg(a.eps + row);
    const float inv_scale = __ldg(a.inv_scale + row);
    const bool bad = __any_sync(0xffffffffu, my_cnt < 0);
    float thr0 = my_thr;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) thr0 = fmaxf(thr0, __shfl_xor_sync(0xffffffffu, thr0, o));
    int E = 0;
    if (!bad) {
      for (int s = 0; s < a.splits; ++s) {
        const int c = __shfl_sync(0xffffffffu, my_cnt, s);
        const uint2* src = a.cand + ((int64_t)s * a.rows_pad + row) * CAND;
        for (int i = lane; i < c; i += 32) ent[E + i] = src[i];
        E += c;
      }
    }
    if (bad) {
      if (lane == 0) {
        a.row_flags[row] = 1;
        a.row_map[atomicAdd(a.exact_rows, 1)] = (int32_t)row;
      }
      continue;
    }
    float nq2 = 0.f;
    for (int c = lane; c < d; c += 32) {
      float q0, q1;
      query_value(a.s, row, c, q0, q1);
      q[c] = q0;
      nq2 = fmaf(q0, q0, nq2);
      if (a.parts == 2) {
        q[d + c] = q1;
        nq2 = fmaf(q1, q1, nq2);
      }
    }
    nq2 = warp_sum(nq2);
    MaskInfo mi;
    mi.hist_items = a.hist_items;
    mi.h_lo = h_lo;
    mi.h_hi = h_hi;
    mi.n_targets = a.n_targets;
    mi.mask_first = a.mask_first;
    const int hlen = (int)(mi.h_hi - mi.h_lo);
    const bool hist_sm = hlen <= RS_HIST;
    if (hist_sm)
      for (int i = lane; i < hlen; i += 32) hist[i] = (uint32_t)a.hist_items[mi.h_lo + i];
    __syncwarp();
    // ---- final tau: k-th largest maximum among the safe chunks that clear every split's threshold ------
    for (int i = lane; i < E; i += 32) {
      const uint2 e = ent[i];
      uint32_t key = 0u;
      if (__uint_as_float(e.x) >= thr0) {
        bool unsafe = (e.y & F_UNSAFE) != 0;
        if (!(e.y & F_KNOWN)) {   // appended since the list's last compaction: one word of the row's bitmap
          const uint32_t cid = (e.y >> CID_SHIFT) & CID_MASK;
          unsafe = (__ldg(a.unsafe_bits + row * a.unsafe_wpr + (cid >> 5)) >> (cid & 31u)) & 1u;
        }
        if (!unsafe) key = orderable(__uint_as_float(e.x));
      }
      kbuf[i] = key;
    }
    __syncwarp();
    uint32_t T = 0u;
    if (E <= 256) {
      // the usual case (one or two lists): the keys fit eight registers per lane, and the radix descent of the sweep's
      // compaction (starts at the highest bit in which the keys differ, stops when exactly k remain) selects tau in
      // ~20 ballots instead of 32 passes over shared memory
      uint32_t key8[8];
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        const int i = q * 32 + lane;
        key8[q] = i < E ? kbuf[i] : 0u;
      }
      if (E <= 128) {
        const uint32_t key4[4] = {key8[0], key8[1], key8[2], key8[3]};
        T = warp_kth_largest<4>(key4, k);
      } else {
        T = warp_kth_largest<8>(key8, k);
      }
    } else {
      int n_t = 0;
      for (int i = lane; i < E; i += 32) n_t += kbuf[i] != 0u;
      n_t = __reduce_add_sync(0xffffffffu, n_t);
      if (n_t >= k) {
        uint32_t P = 0u;
        for (int bit = 31; bit >= 0 && n_t > k; --bit) {
          const uint32_t c = P | (1u << bit);
          int n = 0;
          for (int i = lane; i < E; i += 32) n += kbuf[i] >= c;
          n = __reduce_add_sync(0xffffffffu, n);
          if (n >= k) {
            P = c;
            n_t = n;
          }
        }
        const uint32_t Tm = P ? P : 1u;
        uint32_t mn = 0xFFFFFFFFu;
        for (int i = lane; i < E; i += 32)
          if (kbuf[i] >= Tm) mn = min(mn, kbuf[i]);
        T = __reduce_min_sync(0xffffffffu, mn);
      }
    }
    const float tau = T ? from_orderable(T) : -INFINITY;
    const float thr = fmaxf(thr0, tau - 2.f * eps);
    // The k targets behind tau have exact S a >= tau - eps (a = q.t, or q.t - |t|^2/2 for the L2 models, where
    // the squared distance is |q|^2 - 2a): nothing that scores below them can enter the top-k.  The list lives in
    // the row's scaled units, the exact chain does not: 1 / S is a power of two, the conversion is exact.
    const float lo_a = (tau - 1.25f * eps) * inv_scale;
    const float hi_acc = (nq2 - 2.f * lo_a) * 1.00001f + 4e-6f * nq2;   // only used when tau is finite
    const bool have_tau = T != 0u;
    __syncwarp();
    // ---- survivors: the masked groups of the chunks >= thr ----------------------------------------------------
    // Group ids of all surviving entries are expanded first (kbuf, reused) and scored in full rounds of 32 targets;
    // a row whose groups outgrow the buffer is scored in several fills.
    int n_pass = 0, nk = 0, len = 0;
    auto score_groups = [&](int ng) {
      // exact scores of the members
      const int total = ng * GRP;
      for (int m0 = 0; m0 < total; m0 += 32) {
        const int idx = m0 + lane;
        uint64_t key = 0ull;
        if (idx < total) {
          const int64_t j = (int64_t)kbuf[idx / GRP] * GRP + (idx % GRP);
          bool ok = j < a.n_targets && !(a.mask_first && j == 0);
          if (ok && hlen > 0) {
            if (hist_sm) {
              int lo = 0, hi = hlen;
              while (lo < hi) {
                const int mid = (lo + hi) >> 1;
                if ((int64_t)hist[mid] < j) lo = mid + 1; else hi = mid;
              }
              ok = !(lo < hlen && (int64_t)hist[lo] == j);
            } else {
              int64_t lo = mi.h_lo, hi = mi.h_hi;
              while (lo < hi) {
                const int64_t mid = (lo + hi) >> 1;
                if (a.hist_items[mid] < j) lo = mid + 1; else hi = mid;
              }
              ok = !(lo < mi.h_hi && a.hist_items[lo] == j);
            }
          }
          if (ok) {
            // the CUDA-core kernel's chain: parts in order, columns ascending, one fmaf per column
            float acc = 0.f;
            for (int p = 0; p < a.parts; ++p)
              acc = exact_chain<DIST ? MODE_DIST : MODE_DOT>(q + p * d, a.s.m.entity.w[p] + j * d, d, acc);
            const bool in = !have_tau || (DIST ? (acc <= hi_acc) : (acc >= lo_a));
            if (in) key = make_key(DIST ? (margin - sqrtf(acc)) : acc, (uint32_t)j);
          }
        }
        // stage the keys that can still matter (warp-uniform order: lane ascending)
        const unsigned bal = __ballot_sync(0xffffffffu, key != 0ull);
        const int nb = __popc(bal);
        if (nb) {
          if (nk + nb > RS_KEYS) {   // rare: fold the staged keys into the sorted list first
            for (int x = 0; x < nk; ++x) warp_insert(list, len, k, keys[x], lane);
            nk = 0;
          }
          if (key != 0ull) keys[nk + __popc(bal & ((1u << lane) - 1u))] = key;
          nk += nb;
          n_pass += nb;
          __syncwarp();
        }
      }
          };
    for (int b0 = 0; b0 < E || b0 == 0;) {   // (one fill per pass; a single call site keeps the scoring code un-duplicated)
      int ngt = 0;
      for (; b0 < E; b0 += 32) {
        const int i = b0 + lane;
        uint32_t gmask = 0u, cid = 0u;
        if (i < E && __uint_as_float(ent[i].x) >= thr) {
          gmask = ent[i].y & 0xFFu;
          cid = (ent[i].y >> CID_SHIFT) & CID_MASK;
        }
        int pos = __popc(gmask);   // exclusive prefix over the lanes -> slot of this lane's first group
        int incl = pos;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const int y = __shfl_up_sync(0xffffffffu, incl, o);
          if (lane >= o) incl += y;
        }
        const int ng = __shfl_sync(0xffffffffu, incl, 31);
        if (ngt + ng > a.nent) break;   // (a batch holds at most 256 groups and the buffer at least 256 slots)
        pos = ngt + incl - pos;
        while (gmask) {
          const int b = __ffs(gmask) - 1;   // mask bit b = group 7 - b of the chunk (see chunk_push)
          gmask &= gmask - 1;
          kbuf[pos++] = cid * 8u + (uint32_t)(7 - b);
        }
        ngt += ng;
      }
      __syncwarp();
      score_groups(ngt);
      __syncwarp();   // kbuf is refilled by the next pass
      if (b0 >= E) break;
    }
    // ---- order the keys: (score desc, id asc) ------------------------------------------------------------------
    if (n_pass < k) {
      if (lane == 0) {
        a.row_flags[row] = 1;
        a.row_map[atomicAdd(a.exact_rows, 1)] = (int32_t)row;
      }
    } else {
      uint64_t out;
      if (len == 0 && nk <= 32) {
        out = warp_sort_desc(lane < nk ? keys[lane] : 0ull, lane);
      } else {
        for (int x = 0; x < nk; ++x) warp_insert(list, len, k, keys[x], lane);
        out = lane < k ? list[lane] : 0ull;
      }
      if (lane == 0) a.row_flags[row] = 0;
      if (lane < k) {
        a.ids_out[row * k + lane] = key_id(out);
        if (a.scores_out) a.scores_out[row * k + lane] = key_score(out);
      }
    }
    __syncwarp();
  }
}

struct MmaPlan {
  int parts, dist, kp, stages, tn, nbuf, ncol, nh, kc, nkc, ctas_per_sm, splits, tiles_per_split;
  char cfg;
  size_t smem;
  int64_t n_tiles, rows_pad, unsafe_wpr;
};
constexpr int KP_MAX = 640;   // largest padded K of the tensor-core path (shape k: 128 query rows x 640 x 2 B = 160 KB)

int plan_mma(const kge_model_t* m, int64_t n, int64_t n_targets, int k, int shape, MmaPlan& pl) {
  KGE_REQUIRE(m && m->model >= KGE_TRANSE && m->model <= KGE_COMPLEX, KGE_E_ARG, "bad model");
  pl.parts = (m->model == KGE_ROTATE || m->model == KGE_COMPLEX) ? 2 : 1;
  pl.dist = (m->model == KGE_TRANSE || m->model == KGE_ROTATE) ? 1 : 0;
  const int kd = pl.parts * m->d + (pl.dist ? 3 : 0);
  pl.kp = (kd + 15) / 16 * 16;
  KGE_REQUIRE(pl.kp <= KP_MAX, KGE_E_UNSUPPORTED, "K = %d too large for the tensor-core path (max %d)", pl.kp, KP_MAX);
  KGE_REQUIRE(k >= 1 && k <= 32, KGE_E_UNSUPPORTED, "k = %d too large for the tensor-core path (max 32)", k);
  KGE_REQUIRE(n_targets >= 1 && n_targets < (int64_t)CID_MASK * CH, KGE_E_UNSUPPORTED, "bad n_targets");
  // Sweep shape (NH row halves of 128 queries per CTA, TN targets per tile, NBUF accumulators per row half, NCOL
  // column slices per tile).  SS-mode tcgen05.mma with N = 64 runs at well under half rate (operand fetch + a
  // per-instruction cost), so TN = 128 wherever it fits:
  //   (a) NH 2, TN 128, NBUF 1, NCOL 1: 256 TMEM columns, two CTAs per SM = four accumulator streams per SM
  //                                                                                          -- K <= 80
  //   (f) NH 2, TN 128, NBUF 2, NCOL 2: all 512 columns, one CTA of 16 epilogue warps and two MMA issuer warps per
  //       SM                                                                                 -- K <= ~190
  //   (c) NH 2, TN 64,  NBUF 2, NCOL 1: one CTA per SM: (f) has no room for two whole tiles  -- K <= 256
  //   (k) NH 1, TN 128, NBUF 2, NCOL 2: the queries of 256 rows no longer fit next to a ring, so a CTA keeps 128 rows
  //       and the tiles stream through the ring in chunks of 64 K columns (RotatE d = 128 / 256: K = 272 / 528).
  //       Every B element now serves 128 rows instead of 256: the sweep reads the image twice as often from L2
  //       (~42 B/clk/SM at full tensor rate, about the chip's L2 limit), which bounds this shape   -- K <= 640
  // `shape` = 'a' | 'f' | 'c' | 'k' forces one (tests, experiments; 0 = pick); the target image depends on TN only.
  KGE_REQUIRE(shape == 0 || shape == 'a' || shape == 'f' || shape == 'c' || shape == 'k', KGE_E_ARG,
              "unknown sweep shape %d", shape);
  const size_t two_per_sm = 112 * 1024, one_per_sm = 200 * 1024, one_per_sm_max = 225 * 1024;   // 227 KB per SM
  auto fixed_for = [&](int nh) { return (size_t)MH * nh * pl.kp * 2 + 32 * 8 + 2 * (size_t)MH * nh * 4 + 64; };
  const size_t fixed2 = fixed_for(2);
  char cfg = (char)shape;
  if (cfg == 'a' && fixed2 + 2 * (size_t)128 * pl.kp * 2 > two_per_sm) cfg = 0;
  if (cfg == 'f' && fixed2 + 2 * (size_t)128 * pl.kp * 2 > one_per_sm) cfg = 0;
  if (cfg == 'c' && fixed2 + 2 * (size_t)64 * pl.kp * 2 > one_per_sm) cfg = 0;
  if (!cfg) {
    if (fixed2 + 3 * (size_t)128 * pl.kp * 2 <= two_per_sm) cfg = 'a';
    else if (fixed2 + 2 * (size_t)128 * pl.kp * 2 <= one_per_sm) cfg = 'f';
    else cfg = (fixed2 + 2 * (size_t)64 * pl.kp * 2 <= one_per_sm) ? 'c' : 'k';
  }
  pl.cfg = cfg;
  pl.nh = cfg == 'k' ? 1 : 2;
  pl.tn = cfg == 'c' ? 64 : 128;
  pl.nbuf = cfg == 'a' ? 1 : 2;
  pl.ncol = (cfg == 'f' || cfg == 'k') ? 2 : 1;
  pl.kc = cfg == 'k' ? (pl.kp < 64 ? pl.kp : 64) : pl.kp;   // 16 KB stages: several chunks in flight ahead of the MMAs
  pl.nkc = (pl.kp + pl.kc - 1) / pl.kc;
  const int mm = MH * pl.nh;
  const size_t fixed = fixed_for(pl.nh), a_bytes = (size_t)mm * pl.kp * 2;
  const size_t s_bytes = (size_t)pl.tn * pl.kc * 2;
  const size_t budget = cfg == 'a' ? two_per_sm : (cfg == 'k' ? one_per_sm_max : one_per_sm);
  KGE_REQUIRE(fixed + 2 * s_bytes <= budget, KGE_E_UNSUPPORTED, "K = %d leaves no room for a pipeline", pl.kp);
  pl.ctas_per_sm = cfg == 'a' ? 2 : 1;
  int stages = (int)((budget - fixed) / s_bytes);
  if (stages > 8) stages = 8;
  pl.stages = stages;
  pl.smem = a_bytes + (size_t)stages * s_bytes + (size_t)(2 * stages + 8) * 8 + 2 * (size_t)mm * 4 + 64;
  // the setup stages one fp32 query row per warp in the ring
  const int n_warps = 4 * pl.nh * pl.ncol + 3;
  KGE_REQUIRE((size_t)stages * s_bytes >= (size_t)n_warps * pl.kp * 4, KGE_E_UNSUPPORTED, "ring too small");
  pl.n_tiles = (n_targets + pl.tn - 1) / pl.tn;
  pl.rows_pad = (n + mm - 1) / mm * mm;
  pl.unsafe_wpr = (pl.n_tiles * (pl.tn / CH) + 31) / 32;
  // target splits: fill the resident CTA slots when there are few row blocks
  const int64_t row_blocks = pl.rows_pad / mm > 0 ? pl.rows_pad / mm : 1;
  const int64_t slots = (int64_t)kge_num_sms() * pl.ctas_per_sm;
  int64_t s = slots / row_blocks;
  if (s > MAX_SPLITS) s = MAX_SPLITS;
  if (s > pl.n_tiles / 16) s = pl.n_tiles / 16;
  if (s < 1) s = 1;
  pl.tiles_per_split = (int)((pl.n_tiles + s - 1) / s);
  pl.splits = (int)((pl.n_tiles + pl.tiles_per_split - 1) / pl.tiles_per_split);
  return 0;
}

}  // namespace

extern "C" int64_t kge_mma_image_bytes(const kge_model_t* model, int64_t n_targets, int32_t shape) {
  MmaPlan pl = {};
  if (!model || plan_mma(model, 1, n_targets, 1, shape, pl)) return -1;
  return IMG_HEADER + pl.n_tiles * pl.tn * (int64_t)pl.kp * 2 + ((n_targets * 4 + 127) / 128) * 128;
}

extern "C" int kge_mma_prepare_targets(const kge_model_t* model, int64_t n_targets, void* image, int64_t image_bytes,
                                       int32_t shape, kge_stream_t stream) {
  MmaPlan pl = {};
  if (int e = plan_mma(model, 1, n_targets, 1, shape, pl)) return e;
  KGE_REQUIRE(n_targets <= model->entity.rows, KGE_E_ARG, "n_targets beyond the entity table");
  const int64_t need = kge_mma_image_bytes(model, n_targets, shape);
  KGE_REQUIRE(image && image_bytes >= need, KGE_E_ARG, "image buffer too small: need %lld bytes", (long long)need);
  KGE_REQUIRE((reinterpret_cast<uintptr_t>(image) & 127) == 0, KGE_E_ARG, "image buffer must be 128-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  PrepArgs a;
  a.m = *model;
  a.n_targets = n_targets;
  a.parts = pl.parts;
  a.kp = pl.kp;
  a.dist = pl.dist;
  a.tn = pl.tn;
  a.header = reinterpret_cast<float*>(image);
  a.tiles = reinterpret_cast<uint16_t*>(reinterpret_cast<unsigned char*>(image) + IMG_HEADER);
  a.tn2 = reinterpret_cast<float*>(reinterpret_cast<unsigned char*>(image) + IMG_HEADER + pl.n_tiles * pl.tn * (int64_t)pl.kp * 2);
  KGE_CUDA(cudaMemsetAsync(image, 0, IMG_HEADER, st));
  const int sms = kge_num_sms();
  target_norm_kernel<<<sms * 4, 256, 0, st>>>(a);
  KGE_LAUNCH_CHECK();
  target_image_kernel<<<sms * 8, 256, 0, st>>>(a);
  KGE_LAUNCH_CHECK();
  return 0;
}

namespace {
// Workspace layout (all offsets 16-byte aligned): candidate lists | counts | thresholds | eps | 1/S | unsafe bitmap |
// row map of the rows handed to the exact kernel | that kernel's partial lists.
struct WsLayout {
  int64_t cand, cnt, thr, eps, inv, bits, rowmap, exact, total;
};
int64_t align16(int64_t x) { return (x + 15) / 16 * 16; }
int ws_layout(const kge_model_t* model, const MmaPlan& pl, int64_t n, int64_t n_targets, int k, WsLayout& w) {
  const int64_t lists = (int64_t)pl.splits * pl.ncol * pl.rows_pad;
  const int64_t exact = kge_topk_rows_indirect_workspace_bytes(model, n, n_targets, k);
  KGE_REQUIRE(exact >= 0, KGE_E_UNSUPPORTED, "the exact fallback kernel does not support this shape");
  int64_t o = 0;
  w.cand = o; o = align16(o + lists * CAND * 8);
  w.cnt = o; o = align16(o + lists * 4);
  w.thr = o; o = align16(o + lists * 4);
  w.eps = o; o = align16(o + pl.rows_pad * 4);
  w.inv = o; o = align16(o + pl.rows_pad * 4);
  w.bits = o; o = align16(o + pl.rows_pad * pl.unsafe_wpr * 4);
  w.rowmap = o; o = align16(o + pl.rows_pad * 4);
  w.exact = o; o = align16(o + exact);
  w.total = o;
  return 0;
}
}  // namespace

extern "C" int64_t kge_full_sort_topk_mma_workspace_bytes(const kge_model_t* model, int64_t n, int64_t n_targets,
                                                          int32_t k, int32_t shape) {
  MmaPlan pl = {};
  WsLayout w = {};
  if (!model || n < 0 || plan_mma(model, n, n_targets, k, shape, pl) || ws_layout(model, pl, n, n_targets, k, w)) return -1;
  return w.total;
}

extern "C" int kge_full_sort_topk_mma(const kge_model_t* model, const int64_t* heads, const int64_t* rels, int64_t n,
                                      int head_is_user, int64_t n_targets, const void* image, const int64_t* hist_off,
                                      const int64_t* hist_items, int mask_first, int32_t k, int64_t* ids_out,
                                      float* scores_out, int32_t* row_flags, int32_t* exact_rows, void* workspace,
                                      int64_t workspace_bytes, float* debug_scores, int32_t shape,
                                      kge_stream_t stream) {
  MmaPlan pl = {};
  if (int e = plan_mma(model, n, n_targets, k, shape, pl)) return e;
  KGE_REQUIRE(n >= 0 && n_targets <= model->entity.rows && k <= n_targets, KGE_E_ARG, "bad n / n_targets / k");
  KGE_REQUIRE(exact_rows, KGE_E_ARG, "NULL exact_rows");
  cudaStream_t st = (cudaStream_t)stream;
  KGE_CUDA(cudaMemsetAsync(exact_rows, 0, 4, st));
  if (n == 0) return 0;
  KGE_REQUIRE(heads && image && ids_out && row_flags && workspace, KGE_E_ARG, "NULL argument");
  KGE_REQUIRE((hist_off == nullptr) == (hist_items == nullptr), KGE_E_ARG, "hist_off / hist_items must come together");
  KGE_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 15) == 0, KGE_E_ARG, "workspace must be 16-byte aligned");
  WsLayout w = {};
  if (int e = ws_layout(model, pl, n, n_targets, k, w)) return e;
  KGE_REQUIRE(workspace_bytes >= w.total, KGE_E_ARG, "workspace too small: need %lld bytes", (long long)w.total);

  MmaArgs a = {};
  a.s.m = *model;
  a.s.heads = heads;
  a.s.rels = rels;
  a.s.tails = nullptr;
  a.s.n = n;
  a.s.head_is_user = head_is_user;
  a.s.rel_row = model->ui_relation_fullsort;
  a.n_targets = n_targets;
  a.n_tiles = pl.n_tiles;
  a.rows_pad = pl.rows_pad;
  a.tiles_per_split = pl.tiles_per_split;
  a.parts = pl.parts;
  a.kp = pl.kp;
  a.dist = pl.dist;
  a.stages = pl.stages;
  a.kc = pl.kc;
  a.nkc = pl.nkc;
  a.header = reinterpret_cast<const float*>(image);
  a.tiles = reinterpret_cast<const uint16_t*>(reinterpret_cast<const unsigned char*>(image) + IMG_HEADER);
  a.hist_off = hist_off;
  a.hist_items = hist_items;
  a.mask_first = mask_first;
  a.k = k;
  unsigned char* ws = reinterpret_cast<unsigned char*>(workspace);
  a.cand = reinterpret_cast<uint2*>(ws + w.cand);
  a.cand_cnt = reinterpret_cast<int32_t*>(ws + w.cnt);
  a.cand_thr = reinterpret_cast<float*>(ws + w.thr);
  a.eps_out = reinterpret_cast<float*>(ws + w.eps);
  a.inv_scale_out = reinterpret_cast<float*>(ws + w.inv);
  uint32_t* unsafe_bits = reinterpret_cast<uint32_t*>(ws + w.bits);
  a.unsafe_bits = unsafe_bits;
  a.unsafe_wpr = pl.unsafe_wpr;
  a.dbg_out = debug_scores;
  a.dbg_stride = (n_targets + 127) / 128 * 128;

  KGE_CUDA(cudaMemsetAsync(unsafe_bits, 0, (size_t)pl.rows_pad * pl.unsafe_wpr * 4, st));
  {
    int64_t g = (n + 7) / 8;
    const int64_t cap = (int64_t)kge_num_sms() * 8;
    unsafe_bitmap_kernel<<<(unsigned)(g < cap ? g : cap), 256, 0, st>>>(unsafe_bits, pl.unsafe_wpr, n, n_targets,
                                                                       pl.n_tiles * (pl.tn / CH), hist_off, hist_items,
                                                                       mask_first);
    KGE_LAUNCH_CHECK();
  }
  const dim3 grid((unsigned)(pl.rows_pad / (MH * pl.nh)), (unsigned)pl.splits);
#define KGE_SWEEP(NH_, TN_, NB_, NC_, NM_, DBG_)                                                                   \
  do {                                                                                                            \
    KGE_CUDA(cudaFuncSetAttribute(fullsort_mma_kernel<NH_, TN_, NB_, NC_, NM_, DBG_>,                             \
                                  cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.smem));                    \
    fullsort_mma_kernel<NH_, TN_, NB_, NC_, NM_, DBG_>                                                            \
        <<<grid, sweep_threads(NH_, NC_, NM_), pl.smem, st>>>(a);                                                 \
  } while (0)
  if (pl.cfg == 'a') {
    if (debug_scores) KGE_SWEEP(2, 128, 1, 1, 1, true); else KGE_SWEEP(2, 128, 1, 1, 1, false);
  } else if (pl.cfg == 'f') {
    if (debug_scores) KGE_SWEEP(2, 128, 2, 2, 2, true); else KGE_SWEEP(2, 128, 2, 2, 2, false);
  } else if (pl.cfg == 'c') {
    if (debug_scores) KGE_SWEEP(2, 64, 2, 1, 2, true); else KGE_SWEEP(2, 64, 2, 1, 2, false);
  } else {
    if (debug_scores) KGE_SWEEP(1, 128, 2, 2, 1, true); else KGE_SWEEP(1, 128, 2, 2, 1, false);
  }
#undef KGE_SWEEP
  KGE_LAUNCH_CHECK();

  RescoreArgs r = {};
  r.s = a.s;
  r.n_targets = n_targets;
  r.rows_pad = pl.rows_pad;
  r.splits = pl.splits * pl.ncol;
  r.parts = pl.parts;
  r.hist_off = hist_off;
  r.hist_items = hist_items;
  r.mask_first = mask_first;
  r.k = k;
  r.cand = a.cand;
  r.cand_cnt = a.cand_cnt;
  r.cand_thr = a.cand_thr;
  r.eps = a.eps_out;
  r.inv_scale = a.inv_scale_out;
  r.ids_out = ids_out;
  r.scores_out = scores_out;
  r.row_flags = row_flags;
  r.unsafe_bits = a.unsafe_bits;
  r.unsafe_wpr = a.unsafe_wpr;
  r.row_map = reinterpret_cast<int32_t*>(ws + w.rowmap);
  r.exact_rows = exact_rows;
  r.nent = r.splits * CAND > RS_GIDS ? r.splits * CAND : RS_GIDS;
  const size_t rs_smem = rescore_smem_per_warp(pl.parts * model->d, r.nent) * RS_WARPS;
  int64_t g = (n + RS_WARPS - 1) / RS_WARPS;
  const int64_t cap = (int64_t)kge_num_sms() * 8;
  const unsigned rs_grid = (unsigned)(g < cap ? g : cap);
  if (pl.dist) {
    KGE_CUDA(cudaFuncSetAttribute(rescore_topk_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rs_smem));
    rescore_topk_kernel<true><<<rs_grid, RS_WARPS * 32, rs_smem, st>>>(r);
  } else {
    KGE_CUDA(cudaFuncSetAttribute(rescore_topk_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rs_smem));
    rescore_topk_kernel<false><<<rs_grid, RS_WARPS * 32, rs_smem, st>>>(r);
  }
  KGE_LAUNCH_CHECK();
  // the rows the filter could not bound (row_map[0 .. *exact_rows)), through the exact fp32 kernel: sized and gated
  // on the device, no host round trip
  return kge_topk_rows_indirect(model, heads, rels, n, head_is_user, n_targets, hist_off, hist_items, mask_first, k,
                                r.row_map, exact_rows, ids_out, scores_out, ws + w.exact, st);
}
