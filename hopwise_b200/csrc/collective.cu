// In-switch all-reduce of the gradient accumulators over NVLink multicast (NVLS): the dense route of the
// data-parallel train step (hopwise_b200/distributed.py), replacing DDP's dense all-reduce of every embedding
// table (trainer/trainer.py:82-112) and, on this route, NCCL.
//
// Every rank maps the same symmetric buffer and holds a multicast address that names all N copies at once.
// Rank r owns the r-th slice of the buffer: one multimem.ld_reduce per 16 bytes makes the NVSwitch fetch the N
// copies and return their sum, one multimem.st writes the sum back into all N copies.  Each element is reduced
// exactly once, by one rank, and broadcast: the replicas receive bit-identical sums, and a GPU sends and
// receives ~one buffer per step instead of the 2(N-1)/N buffers a ring moves through its links.  The caller
// brackets the launch with a cross-rank barrier on each side (all gradients written before / all slices
// reduced after).
#include "common.cuh"

namespace {

__device__ __forceinline__ float4 multimem_ld_reduce_add(const float* mc) {
  float4 v;
  asm volatile("multimem.ld_reduce.relaxed.sys.global.add.v4.f32 {%0, %1, %2, %3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
               : "l"(mc)
               : "memory");
  return v;
}
__device__ __forceinline__ void multimem_st(float* mc, float4 v) {
  asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(mc), "f"(v.x), "f"(v.y), "f"(v.z),
               "f"(v.w)
               : "memory");
}

__global__ void __launch_bounds__(256) multimem_all_reduce_kernel(float* __restrict__ mc, int64_t q_lo, int64_t q_hi) {
  // q = index of a 16-byte quad; four quads in flight per thread
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  int64_t q = q_lo + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  for (; q + 3 * stride < q_hi; q += 4 * stride) {
    float4 v[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) v[u] = multimem_ld_reduce_add(mc + 4 * (q + u * stride));
#pragma unroll
    for (int u = 0; u < 4; ++u) multimem_st(mc + 4 * (q + u * stride), v[u]);
  }
  for (; q < q_hi; q += stride) multimem_st(mc + 4 * q, multimem_ld_reduce_add(mc + 4 * q));
  __threadfence_system();
}

// ---- the same reduction with both cross-rank barriers inside the kernel ------------------------------------------
// Around the plain kernel the caller needs two host-launched barriers (torch's symmetric-memory barrier: one more
// kernel launch and signal round each) plus a fill of the touch marks: ~90 us of an 8-GPU step whose reduction moves
// 14 MB in ~30 us.  Here block 0 performs barrier A (every rank's gradient kernel has finished: stream order on
// each rank, made visible by release / acquire at system scope) and releases the other blocks through a flag in
// local memory; every block reduces its part of this rank's slice; the touch marks of the dense tables are stored;
// and the LAST block to finish performs barrier B (every slice has been reduced and broadcast), so that the kernel's
// completion on this stream means the whole buffer is final on this GPU.  Barrier = the flag protocol of torch's own
// symmetric-memory barrier: rank r raises slot [r] in every peer's signal pad (CAS 0 -> 1, release) and consumes
// slot [p] in its own pad for every peer p (CAS 1 -> 0, acquire).  The grid must be co-resident (it is sized for
// half of the SMs' block slots, and the stream runs nothing else); every spin is bounded and traps.
constexpr uint32_t COLL_SPIN_LIMIT = 1u << 28;

__device__ __forceinline__ uint32_t cas_release_sys(uint32_t* p, uint32_t cmp, uint32_t val) {
  uint32_t old;
  asm volatile("atom.global.release.sys.cas.b32 %0, [%1], %2, %3;" : "=r"(old) : "l"(p), "r"(cmp), "r"(val) : "memory");
  return old;
}
__device__ __forceinline__ uint32_t cas_acquire_sys(uint32_t* p, uint32_t cmp, uint32_t val) {
  uint32_t old;
  asm volatile("atom.global.acquire.sys.cas.b32 %0, [%1], %2, %3;" : "=r"(old) : "l"(p), "r"(cmp), "r"(val) : "memory");
  return old;
}
// threads [0, world) of one block; `slots` = first slot of this barrier inside every signal pad
__device__ __forceinline__ void cross_rank_barrier(uint32_t* const* pads, int rank, int world, int slots) {
  const int p = threadIdx.x;
  if (p < world) {
    uint32_t spins = 0;
    while (cas_release_sys(pads[p] + slots + rank, 0u, 1u) != 0u)
      if (++spins > COLL_SPIN_LIMIT) __trap();
    spins = 0;
    while (cas_acquire_sys(pads[rank] + slots + p, 1u, 0u) != 1u)
      if (++spins > COLL_SPIN_LIMIT) __trap();
  }
}

__global__ void __launch_bounds__(256) multimem_all_reduce_fused_kernel(float* __restrict__ mc, int64_t q_lo,
                                                                        int64_t q_hi, uint32_t* const* pads, int rank,
                                                                        int world, int slot_base, uint32_t* local,
                                                                        uint32_t epoch, int32_t* row_state,
                                                                        int64_t n_mark, int32_t step) {
  __shared__ int s_last;
  // ---- barrier A, then release the grid
  if (blockIdx.x == 0) {
    cross_rank_barrier(pads, rank, world, slot_base);
    __syncthreads();
    if (threadIdx.x == 0) asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(local), "r"(epoch) : "memory");
  } else {
    if (threadIdx.x == 0) {
      uint32_t seen, spins = 0;
      do {
        asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(seen) : "l"(local) : "memory");
        if (++spins > COLL_SPIN_LIMIT) __trap();
      } while (seen != epoch);
    }
    __syncthreads();
  }
  // ---- this rank's slice: the switch fetches the N copies and returns their sum; one store writes all N copies
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  int64_t q = q_lo + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  for (; q + 3 * stride < q_hi; q += 4 * stride) {
    float4 v[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) v[u] = multimem_ld_reduce_add(mc + 4 * (q + u * stride));
#pragma unroll
    for (int u = 0; u < 4; ++u) multimem_st(mc + 4 * (q + u * stride), v[u]);
  }
  for (; q < q_hi; q += stride) multimem_st(mc + 4 * q, multimem_ld_reduce_add(mc + 4 * q));
  // every row of a dense table counts as touched in this step (a row nobody touched holds a zero gradient)
  for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n_mark; r += stride) row_state[2 * r + 1] = step;
  __threadfence_system();
  __syncthreads();
  // ---- barrier B by the last block to get here
  if (threadIdx.x == 0) {
    const uint32_t done = atomicAdd(local + 1, 1u);
    s_last = done == gridDim.x - 1;
    if (s_last) local[1] = 0u;   // (re-armed for the next call; nobody else touches it any more)
  }
  __syncthreads();
  if (s_last) cross_rank_barrier(pads, rank, world, slot_base + world);
}

// ---- owner-sharded dense Adam over the switch ---------------------------------------------------------------------
// One kernel per step instead of all-reduce + Adam: rank r owns the r-th slice of the flat parameter space.  It reads
// the SUM of the N gradient copies of its slice straight from the switch (multimem.ld_reduce), takes the Adam step for
// those elements with its (sharded) moments, and multicasts the new weights to every
// replica (multimem.st).  Every rank moves 1/N of the gradient in and 1/N of the weights out, and does 1/N of the
// optimiser arithmetic; torch.optim.Adam's (or AdamW's) dense semantics (every element, every step), which is what the
// reference trains with (trainer/trainer.py:131-170 builds optim.Adam over all parameters; DDP averages the gradients
// first).
struct OwnerAdam {
  float* g_mc;        // multicast address of the flat gradient buffer
  float* w_mc;        // multicast address of the flat weight buffer
  const float* w;     // this rank's replica of the weights (same layout)
  float* m;           // moments: only [q_lo, q_hi) is ever touched on this rank
  float* v;
  int64_t q_lo, q_hi; // float4 units
  float scale;        // 1 / world (DDP's mean) times the caller's loss scale
  float lr_c, rsq_c;  // lr / (1 - b1^t), 1 / sqrt(1 - b2^t)
  float b2, omb1, omb2, eps;
  int decays;         // AdamW: the weights are multiplied by `decay` = fp32(1 - lr * weight_decay) first
  float decay;
};

__device__ __forceinline__ void owner_adam_quad(const OwnerAdam& a, int64_t q, float4 g, float4 w4, float4 m4,
                                                float4 v4) {
  float wv[4] = {w4.x, w4.y, w4.z, w4.w}, mv[4] = {m4.x, m4.y, m4.z, m4.w}, vv[4] = {v4.x, v4.y, v4.z, v4.w};
  const float gv[4] = {g.x, g.y, g.z, g.w};
#pragma unroll
  for (int e = 0; e < 4; ++e) {   // the arithmetic of adam_row (train.cu), element for element
    const float ge = gv[e] * a.scale;
    if (a.decays) wv[e] *= a.decay;
    mv[e] += a.omb1 * (ge - mv[e]);
    vv[e] = vv[e] * a.b2 + a.omb2 * ge * ge;
    const float den = sqrt_nonneg(vv[e]) * a.rsq_c + a.eps;
    wv[e] -= a.lr_c * div_pos_den(mv[e], den);
  }
  *reinterpret_cast<float4*>(a.m + 4 * q) = make_float4(mv[0], mv[1], mv[2], mv[3]);
  *reinterpret_cast<float4*>(a.v + 4 * q) = make_float4(vv[0], vv[1], vv[2], vv[3]);
  multimem_st(a.w_mc + 4 * q, make_float4(wv[0], wv[1], wv[2], wv[3]));
}

// U quads of one thread: every load first (the switch round trip of the gradient and the three local reads of each
// quad are all in flight together), then the arithmetic and the stores.  The kernel is latency-bound on those round
// trips: at two quads in flight the step of a 3.6 M-float model took ~84 us on 2 GPUs, barriers included.
template <int U>
__device__ __forceinline__ void owner_adam_batch(const OwnerAdam& a, int64_t q, int64_t stride, int n) {
  float4 g[U], w4[U], m4[U], v4[U];
#pragma unroll
  for (int u = 0; u < U; ++u)
    if (u < n) {
      const int64_t qq = q + u * stride;
      g[u] = multimem_ld_reduce_add(a.g_mc + 4 * qq);
      w4[u] = *reinterpret_cast<const float4*>(a.w + 4 * qq);
      m4[u] = *reinterpret_cast<const float4*>(a.m + 4 * qq);
      v4[u] = *reinterpret_cast<const float4*>(a.v + 4 * qq);
    }
#pragma unroll
  for (int u = 0; u < U; ++u)
    if (u < n) owner_adam_quad(a, q + u * stride, g[u], w4[u], m4[u], v4[u]);
}

__global__ void __launch_bounds__(256, 2) owner_adam_kernel(const OwnerAdam a, uint32_t* const* pads, int rank, int world,
                                                         int slot_base, uint32_t* local, uint32_t epoch) {
  __shared__ int s_last;
  // ---- barrier A (every rank's forward kernel has written its gradients), then release the grid
  if (blockIdx.x == 0) {
    cross_rank_barrier(pads, rank, world, slot_base);
    __syncthreads();
    if (threadIdx.x == 0) asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(local), "r"(epoch) : "memory");
  } else {
    if (threadIdx.x == 0) {
      uint32_t seen, spins = 0;
      do {
        asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(seen) : "l"(local) : "memory");
        if (++spins > COLL_SPIN_LIMIT) __trap();
      } while (seen != epoch);
    }
    __syncthreads();
  }
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  constexpr int U = 4;
  for (int64_t q = a.q_lo + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < a.q_hi; q += U * stride) {
    const int64_t left = (a.q_hi - q + stride - 1) / stride;   // quads of this thread from q on
    owner_adam_batch<U>(a, q, stride, left < U ? (int)left : U);
  }
  __threadfence_system();
  __syncthreads();
  // ---- barrier B (every replica holds every slice's new weights and a zeroed gradient) by the last block
  if (threadIdx.x == 0) {
    const uint32_t done = atomicAdd(local + 1, 1u);
    s_last = done == gridDim.x - 1;
    if (s_last) local[1] = 0u;
  }
  __syncthreads();
  if (s_last) cross_rank_barrier(pads, rank, world, slot_base + world);
}

}  // namespace

extern "C" int kge_multimem_all_reduce_fused_f32(void* multicast_ptr, int64_t n_floats, int32_t rank, int32_t world,
                                                 void* const* signal_pads_dev, int32_t slot_base, uint32_t* local_flags,
                                                 uint32_t epoch, int32_t* row_state, int64_t n_mark_rows, int32_t step,
                                                 kge_stream_t stream) {
  KGE_REQUIRE(multicast_ptr && n_floats >= 0 && world >= 1 && world <= 32 && rank >= 0 && rank < world, KGE_E_ARG,
              "bad multimem all-reduce arguments");
  KGE_REQUIRE((reinterpret_cast<uintptr_t>(multicast_ptr) & 15) == 0 && (n_floats & 3) == 0, KGE_E_ARG,
              "multimem all-reduce needs a 16-byte aligned buffer of a multiple of 4 floats");
  KGE_REQUIRE(signal_pads_dev && local_flags && slot_base >= 0 && epoch != 0, KGE_E_ARG, "bad barrier arguments");
  KGE_REQUIRE(n_mark_rows == 0 || row_state, KGE_E_ARG, "row_state missing");
  const int64_t quads = n_floats / 4;
  const int64_t per = (quads + world - 1) / world;
  const int64_t lo = per * rank, hi = lo + per < quads ? lo + per : quads;   // (an empty slice still takes the barriers)
  const int threads = 256;
  int64_t grid = hi > lo ? (hi - lo + 4 * threads - 1) / (4 * threads) : 1;
  const int64_t cap = (int64_t)kge_num_sms() * 4;   // co-resident: 8 blocks of 256 threads fit an SM
  if (grid > cap) grid = cap;
  multimem_all_reduce_fused_kernel<<<(unsigned)grid, threads, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<float*>(multicast_ptr), lo, hi > lo ? hi : lo, reinterpret_cast<uint32_t* const*>(signal_pads_dev),
      rank, world, slot_base, local_flags, epoch, row_state, n_mark_rows, step);
  KGE_LAUNCH_CHECK();
  return 0;
}

extern "C" int kge_multimem_all_reduce_f32(void* multicast_ptr, int64_t n_floats, int32_t rank, int32_t world,
                                           kge_stream_t stream) {
  KGE_REQUIRE(multicast_ptr && n_floats >= 0 && world >= 1 && rank >= 0 && rank < world, KGE_E_ARG,
              "bad multimem all-reduce arguments");
  KGE_REQUIRE((reinterpret_cast<uintptr_t>(multicast_ptr) & 15) == 0 && (n_floats & 3) == 0, KGE_E_ARG,
              "multimem all-reduce needs a 16-byte aligned buffer of a multiple of 4 floats");
  const int64_t quads = n_floats / 4;
  const int64_t per = (quads + world - 1) / world;
  const int64_t lo = per * rank, hi = lo + per < quads ? lo + per : quads;
  if (hi <= lo) return 0;
  const int threads = 256;
  int64_t grid = (hi - lo + 4 * threads - 1) / (4 * threads);
  const int64_t cap = (int64_t)kge_num_sms() * 4;
  if (grid > cap) grid = cap;
  multimem_all_reduce_kernel<<<(unsigned)grid, threads, 0, (cudaStream_t)stream>>>(reinterpret_cast<float*>(multicast_ptr),
                                                                                 lo, hi);
  KGE_LAUNCH_CHECK();
  return 0;
}

extern "C" int kge_owner_adam_step(void* grad_multicast, float* grad_local, void* weight_multicast,
                                   const float* weight_local, float* m, float* v, int64_t n_floats, int32_t rank,
                                   int32_t world, const kge_adam_t* adam,
                                   float grad_scale, void* const* signal_pads_dev, int32_t slot_base,
                                   uint32_t* local_flags, uint32_t epoch, kge_stream_t stream) {
  KGE_REQUIRE(grad_multicast && grad_local && weight_multicast && weight_local && m && v && adam, KGE_E_ARG,
              "NULL argument");
  KGE_REQUIRE(n_floats >= 0 && (n_floats & 3) == 0 && world >= 1 && world <= 32 && rank >= 0 && rank < world, KGE_E_ARG,
              "bad owner-Adam arguments");
  KGE_REQUIRE(((reinterpret_cast<uintptr_t>(grad_multicast) | reinterpret_cast<uintptr_t>(weight_multicast) |
                reinterpret_cast<uintptr_t>(weight_local) | reinterpret_cast<uintptr_t>(m) |
                reinterpret_cast<uintptr_t>(v)) & 15) == 0, KGE_E_ARG, "buffers must be 16-byte aligned");
  KGE_REQUIRE(signal_pads_dev && local_flags && slot_base >= 0 && epoch != 0 && adam->step >= 1, KGE_E_ARG,
              "bad barrier / step arguments");
  if (int e = kge_check_optimizer(adam)) return e;
  KGE_REQUIRE(adam->optimizer == KGE_OPT_ADAM || adam->optimizer == KGE_OPT_ADAMW, KGE_E_UNSUPPORTED,
              "the owner-sharded step implements Adam and AdamW (optimizer %d)", adam->optimizer);
  const int64_t quads = n_floats / 4;
  const int64_t per = (quads + world - 1) / world;
  const int64_t lo = per * rank < quads ? per * rank : quads, hi = lo + per < quads ? lo + per : quads;
  OwnerAdam a;
  a.g_mc = reinterpret_cast<float*>(grad_multicast);
  a.w_mc = reinterpret_cast<float*>(weight_multicast);
  a.w = weight_local;
  a.m = m;
  a.v = v;
  a.q_lo = lo;
  a.q_hi = hi;
  a.scale = grad_scale;
  // the bias corrections of kge_adam_table_fill (train.cu), formed in double like torch.optim.Adam's
  const double bc1 = 1.0 - pow((double)adam->beta1, adam->step), bc2 = 1.0 - pow((double)adam->beta2, adam->step);
  a.lr_c = (float)((double)adam->lr / bc1);
  a.rsq_c = (float)(1.0 / sqrt(bc2));
  a.b2 = adam->beta2;
  a.omb1 = (float)(1.0 - (double)adam->beta1);
  a.omb2 = (float)(1.0 - (double)adam->beta2);
  a.eps = adam->eps;
  a.decays = adam->weight_decay != 0.f;   // (AdamW: kge_check_optimizer refuses decay under Adam)
  a.decay = (float)(1.0 - (double)adam->lr * (double)adam->weight_decay);
  const int threads = 256;
  int64_t grid = hi > lo ? (hi - lo + threads - 1) / threads : 1;   // (a thread per quad until the grid is full)
  const int64_t cap = (int64_t)kge_num_sms() * 2;   // co-resident at 128 registers (the grid spins on a flag block 0 raises)
  if (grid > cap) grid = cap;
  owner_adam_kernel<<<(unsigned)grid, threads, 0, (cudaStream_t)stream>>>(
      a, reinterpret_cast<uint32_t* const*>(signal_pads_dev), rank, world, slot_base, local_flags, epoch);
  KGE_LAUNCH_CHECK();
  // The kernel's barrier B means every rank has finished reading every copy of the gradient: this rank's copy is
  // zeroed locally for the next step (zeroing through the multicast address instead doubles what every GPU receives
  // over NVLink per step: N slices of weights AND N slices of zeros).
  KGE_CUDA(cudaMemsetAsync(grad_local, 0, (size_t)n_floats * sizeof(float), (cudaStream_t)stream));
  return 0;
}
