// Data-parallel gradient averaging FUSED into the optimiser update: one ordinary (non-cooperative) kernel per step.
// Every rank's flat gradient buffer lives in peer-mapped memory (torch symmetric memory / CUDA IPC), so the backward
// kernels write the gradients where the peers can read them -- there is no staging copy.  The kernel
//   (1) raises one flag per peer over NVLink (system-scope release store into every peer's flag array),
//   (2) has every CTA wait for all peers' flags of this exchange (acquire spin on its OWN flag array: local reads),
//   (3) reads every rank's gradient straight from peer memory (P2P loads through NVLink / NVSwitch), sums them in RANK
//       ORDER -- every rank computes bit-identical averages, the replicas never drift -- and applies the TF-1.x Adam
//       step (models_gcn.py:294) in the same pass.
// It replaces `ncclAllReduce` + `k_adam_tf`: the all-reduce of this path is 632 KB once per ~0.3 ms step, i.e. pure
// latency (+26 us per step measured for the NCCL call inside the CUDA graph at 2 GPUs).  The reference has no
// distributed code at all (SURVEY.md 2.4); the collective exists only because SURVEY.md 8(e) shards the batch.
//
// Reuse of the gradient buffer: the caller alternates between TWO gradient buffers (even / odd steps; train.py keeps
// one CUDA graph per parity).  A buffer a peer may still be reading is only rewritten two steps later, and by then that
// peer has raised its flag for the step in between, which it does after finishing its reads: no second handshake.
// Flags carry an exchange counter of their own (slot 63 of the rank's flag array) that only grows -- the optimiser
// state may be rewound (warm-up steps before a graph capture), the flags may not.
#include <algorithm>

#include "common.cuh"

namespace gcnb {

constexpr int kMaxRanks = 16;

struct AdamArParams {
  float* p;
  float *m, *v;
  const uint8_t* decay;
  const float* state;            // {b1^t, b2^t, lr_t, t}, already advanced for this step
  long long n;
  float b1, b2, eps, reg;
  const float* grad[kMaxRanks];  // grad[q] = rank q's flat gradient of this step (peer-mapped); grad[rank] is local
  uint32_t* flags[kMaxRanks];    // flags[q] = rank q's flag array: [0, world) one per source rank, 62 CTA counter, 63 exchange
  int rank, world;
};

__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ float4 ld_cv4(const float* p) {
  float4 v;
  asm volatile("ld.global.cv.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
  return v;
}

// kNesterov: TF's NadamOptimizer (ApplyAdam with use_nesterov), the step takes b1 m + (1-b1) g_total in place of m --
// the same rule as k_adam_tf<true> (head.cu).
template <bool kNesterov>
__device__ __forceinline__ void adam_one(const AdamArParams& P, long long i, float gsum, float gscale, float lr_t) {
  const float pi = P.p[i];
  float gi = gsum * gscale;
  if (P.decay != nullptr && P.decay[i]) gi = fmaf(P.reg, pi, gi);
  const float mi = fmaf(1.f - P.b1, gi - P.m[i], P.m[i]);
  const float vi = fmaf(1.f - P.b2, gi * gi - P.v[i], P.v[i]);
  P.m[i] = mi;
  P.v[i] = vi;
  P.p[i] = pi - lr_t * (kNesterov ? fmaf(P.b1, mi, (1.f - P.b1) * gi) : mi) / (sqrtf(vi) + P.eps);
}

template <bool kNesterov>
__global__ void __launch_bounds__(256) k_adam_tf_allreduce(const AdamArParams P) {
  uint32_t* myflags = P.flags[P.rank];
  __shared__ uint32_t s_seq;
  if (threadIdx.x == 0) s_seq = *reinterpret_cast<volatile uint32_t*>(myflags + 63) + 1u;  // bumped by the LAST CTA only
  __syncthreads();
  const uint32_t seq = s_seq;
  // (1) the gradients of this rank were written by earlier kernels of this stream: publish them system-wide, raise flags
  if (blockIdx.x == 0 && (int)threadIdx.x < P.world) {
    __threadfence_system();
    st_release_sys(P.flags[threadIdx.x] + P.rank, seq);
  }
  // (2) every CTA waits for every peer (local acquire loads; the flags arrive over NVLink)
  if ((int)threadIdx.x < P.world) {
    const uint32_t* f = myflags + threadIdx.x;
    const long long t0 = clock64();
    while ((int32_t)(ld_acquire_sys(f) - seq) < 0) {
      if (clock64() - t0 > 20000000000ll) __trap();  // a missing peer must not hang the GPU forever
    }
  }
  __syncthreads();
  // (3) sum the ranks in rank order straight from peer memory (all peer loads of an element group in flight before the
  // first add), then Adam (Nadam)
  const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x, nth = (long long)gridDim.x * blockDim.x;
  const long long n4 = P.n >> 2;
  const float lr_t = P.state[2];
  const float gscale = 1.f / (float)P.world;
  for (long long i = tid; i < n4; i += nth) {
    float4 gs = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int q0 = 0; q0 < P.world; q0 += 8) {
      float4 v[8];
#pragma unroll
      for (int u = 0; u < 8; ++u)
        if (q0 + u < P.world) v[u] = ld_cv4(P.grad[q0 + u] + (i << 2));  // .cv: never a stale cached line
#pragma unroll
      for (int u = 0; u < 8; ++u)
        if (q0 + u < P.world) { gs.x += v[u].x; gs.y += v[u].y; gs.z += v[u].z; gs.w += v[u].w; }
    }
    adam_one<kNesterov>(P, (i << 2) + 0, gs.x, gscale, lr_t);
    adam_one<kNesterov>(P, (i << 2) + 1, gs.y, gscale, lr_t);
    adam_one<kNesterov>(P, (i << 2) + 2, gs.z, gscale, lr_t);
    adam_one<kNesterov>(P, (i << 2) + 3, gs.w, gscale, lr_t);
  }
  for (long long i = (n4 << 2) + tid; i < P.n; i += nth) {
    float gs = 0.f;
    for (int q = 0; q < P.world; ++q) gs += __ldcv(P.grad[q] + i);
    adam_one<kNesterov>(P, i, gs, gscale, lr_t);
  }
  // the last CTA to finish closes the exchange: only then may the next launch see the new counter
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    if (atomicAdd(myflags + 62, 1u) == gridDim.x - 1) {
      myflags[62] = 0;
      __threadfence();
      *reinterpret_cast<volatile uint32_t*>(myflags + 63) = seq;
    }
  }
}

}  // namespace gcnb

using namespace gcnb;

namespace {

int launch_allreduce(bool nesterov, const char* what, float* p, float* m, float* v, const uint8_t* decay,
                     const float* state, long long n, float beta1, float beta2, float eps, float reg,
                     const void* const* peer_grad, void* const* peer_flags, int rank, int world, gcnb_stream_t stream) {
  GCNB_REQUIRE(p && m && v && state && n >= 1 && peer_grad && peer_flags, "%s: bad arguments", what);
  GCNB_REQUIRE(world >= 1 && world <= kMaxRanks && rank >= 0 && rank < world,
               "%s: rank %d / world %d out of range (at most %d ranks)", what, rank, world, kMaxRanks);
  AdamArParams P{};
  P.p = p; P.m = m; P.v = v; P.decay = decay; P.state = state; P.n = n;
  P.b1 = beta1; P.b2 = beta2; P.eps = eps; P.reg = reg; P.rank = rank; P.world = world;
  for (int q = 0; q < world; ++q) {
    GCNB_REQUIRE(peer_grad[q] != nullptr && peer_flags[q] != nullptr, "%s: peer pointer %d is NULL", what, q);
    GCNB_REQUIRE((reinterpret_cast<uintptr_t>(peer_grad[q]) & 15) == 0, "%s: gradient buffers must be 16-byte aligned",
                 what);
    P.grad[q] = static_cast<const float*>(peer_grad[q]);
    P.flags[q] = static_cast<uint32_t*>(peer_flags[q]);
  }
  DeviceInfo di;
  int rc = device_info(&di);
  if (rc) return rc;
  // at most one CTA per SM: every CTA spins on the flags, so all of them must be resident together with CTA 0
  const int grid = (int)std::max<long long>(1, std::min<long long>(ceil_div_ll(n, 256 * 4), di.sm_count));
  if (nesterov) {
    k_adam_tf_allreduce<true><<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(P);
    GCNB_LAUNCH_CHECK("k_adam_tf_allreduce<true>");
  } else {
    k_adam_tf_allreduce<false><<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(P);
    GCNB_LAUNCH_CHECK("k_adam_tf_allreduce");
  }
  return GCNB_OK;
}

}  // namespace

extern "C" {

size_t gcnb_adam_allreduce_flag_bytes(void) { return 64 * sizeof(uint32_t); }

int gcnb_adam_tf_allreduce_f32(float* p, float* m, float* v, const uint8_t* decay, const float* state, long long n,
                               float beta1, float beta2, float eps, float reg, const void* const* peer_grad,
                               void* const* peer_flags, int rank, int world, gcnb_stream_t stream) {
  return launch_allreduce(false, "gcnb_adam_tf_allreduce_f32", p, m, v, decay, state, n, beta1, beta2, eps, reg,
                          peer_grad, peer_flags, rank, world, stream);
}

int gcnb_nadam_tf_allreduce_f32(float* p, float* m, float* v, const uint8_t* decay, const float* state, long long n,
                                float beta1, float beta2, float eps, float reg, const void* const* peer_grad,
                                void* const* peer_flags, int rank, int world, gcnb_stream_t stream) {
  return launch_allreduce(true, "gcnb_nadam_tf_allreduce_f32", p, m, v, decay, state, n, beta1, beta2, eps, reg,
                          peer_grad, peer_flags, rank, world, stream);
}

}  // extern "C"
