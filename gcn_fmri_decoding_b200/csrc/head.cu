// Training-step pieces around the conv stack ("next" rows of the scope table, SURVEY.md 8f):
//   * sparse softmax cross-entropy, forward and backward in one pass (models_gcn.py:253-259),
//   * TensorFlow-1.x Adam over one flat parameter buffer, L2 term folded in (models_gcn.py:260-262, :294), and its
//     Nesterov variant (tf.contrib.opt.NadamOptimizer) for fine-tuning a new classifier head.
// They exist so that a whole training step is a handful of launches inside one CUDA graph.
#include <algorithm>

#include "common.cuh"

namespace gcnb {

// One warp per row: loss_row = logsumexp(z) - z[label]; dlogits = (softmax(z) - onehot) * scale.
// Row losses go to loss_rows[B]; a second tiny kernel averages them in a fixed order.
__global__ void k_softmax_xent(const float* __restrict__ logits, const long long* __restrict__ labels,
                               float* __restrict__ loss_rows, float* __restrict__ dlogits, int B, int C, float scale) {
  const int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (row >= B) return;
  const float* z = logits + (long long)row * C;
  float mx = -INFINITY;
  for (int c = lane; c < C; c += 32) mx = fmaxf(mx, z[c]);
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, d));
  float se = 0.f;
  for (int c = lane; c < C; c += 32) se += expf(z[c] - mx);
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) se += __shfl_xor_sync(0xffffffffu, se, d);
  const float lse = mx + logf(se);
  const long long lab64 = labels[row];
  const bool ok = lab64 >= 0 && lab64 < C;  // a label outside [0, C) contributes neither loss nor gradient
  const int lab = ok ? (int)lab64 : 0;
  if (dlogits != nullptr)
    for (int c = lane; c < C; c += 32)
      dlogits[(long long)row * C + c] = ok ? (expf(z[c] - lse) - (c == lab ? 1.f : 0.f)) * scale : 0.f;
  if (lane == 0) loss_rows[row] = ok ? lse - z[lab] : 0.f;
}

// state[0] = beta1^t, state[1] = beta2^t, state[2] = lr_t = lr * sqrt(1 - beta2^t) / (1 - beta1^t), state[3] = t
__device__ __forceinline__ void adam_tick(float* state, float lr, float b1, float b2) {
  const float p1 = state[0] * b1, p2 = state[1] * b2;
  state[0] = p1;
  state[1] = p2;
  state[2] = lr * sqrtf(1.f - p2) / (1.f - p1);
  state[3] += 1.f;
}


__global__ void k_mean_rows(const float* __restrict__ v, float* __restrict__ out, int n, float* adam_state, float lr,
                            float b1, float b2) {
  __shared__ float red[256];
  float s = 0.f;
  for (int i = threadIdx.x; i < n; i += 256) s += v[i];
  red[threadIdx.x] = s;
  __syncthreads();
  for (int d = 128; d > 0; d >>= 1) {
    if ((int)threadIdx.x < d) red[threadIdx.x] += red[threadIdx.x + d];
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    out[0] = red[0] / (float)n;
    if (adam_state != nullptr) adam_tick(adam_state, lr, b1, b2);
  }
}

__global__ void k_adam_tick(float* state, float lr, float b1, float b2) { adam_tick(state, lr, b1, b2); }

// Single-CTA variant of the cross-entropy (B up to a few thousand rows): rows strided over the warps, fixed-order
// block reduction of the mean, optional optimiser clock tick -- one launch for loss, dlogits and the clock.
__global__ void __launch_bounds__(1024) k_softmax_xent_1cta(const float* __restrict__ logits,
                                                            const long long* __restrict__ labels, float* __restrict__ loss,
                                                            float* __restrict__ dlogits, int B, int C, float scale,
                                                            float* adam_state, float lr, float b1, float b2) {
  __shared__ float red[32];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
  float mine = 0.f;
  for (int row = warp; row < B; row += nw) {
    const float* z = logits + (long long)row * C;
    float mx = -INFINITY;
    for (int c = lane; c < C; c += 32) mx = fmaxf(mx, z[c]);
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, d));
    float se = 0.f;
    for (int c = lane; c < C; c += 32) se += expf(z[c] - mx);
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) se += __shfl_xor_sync(0xffffffffu, se, d);
    const float lse = mx + logf(se);
    const long long lab64 = labels[row];
    const bool ok = lab64 >= 0 && lab64 < C;
    const int lab = ok ? (int)lab64 : 0;
    if (dlogits != nullptr)
      for (int c = lane; c < C; c += 32)
        dlogits[(long long)row * C + c] = ok ? (expf(z[c] - lse) - (c == lab ? 1.f : 0.f)) * scale : 0.f;
    if (ok) mine += lse - z[lab];
  }
  if (lane == 0) red[warp] = mine;
  __syncthreads();
  if (threadIdx.x == 0) {
    float s = 0.f;
    for (int w = 0; w < nw; ++w) s += red[w];
    loss[0] = s / (float)B;
    if (adam_state != nullptr) adam_tick(adam_state, lr, b1, b2);
  }
}

__global__ void k_relu_dropout_fwd(float* __restrict__ x, long long rows, int cols, int ld, float keep, float inv_keep,
                                   uint32_t seed, const float* __restrict__ step) {
  const long long total = rows * cols;
  const uint32_t key = dropout_key(seed, step);
  const uint32_t thresh = dropout_threshold(keep);
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / cols;
    const int c = (int)(i - r * cols);
    float v = fmaxf(x[r * ld + c], 0.f);
    if (keep < 1.f) v = dropout_keeps((uint32_t)i, key, thresh) ? v * inv_keep : 0.f;
    x[r * ld + c] = v;
  }
}

__global__ void k_relu_dropout_bwd(float* __restrict__ d, const float* __restrict__ act, long long rows, int cols, int ld_d,
                                   int ld_act, float inv_keep) {
  const long long total = rows * cols;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / cols;
    const int c = (int)(i - r * cols);
    d[r * ld_d + c] = act[r * ld_act + c] > 0.f ? d[r * ld_d + c] * inv_keep : 0.f;
  }
}

struct ColsumArgs {
  const float* m[4];
  float* out[4];
  int rows[4], cols[4];
  int block_begin[5];  // blocks of 32 columns, prefix over the matrices
};

// block = (matrix, 32-column chunk): 32 row groups x 32 lanes, four independent chains per thread, fixed-order combine
__global__ void __launch_bounds__(1024) k_colsum_multi(ColsumArgs a) {
  __shared__ float red[1024];
  int mi = 0;
  while (mi < 3 && (int)blockIdx.x >= a.block_begin[mi + 1]) ++mi;
  const int c0 = ((int)blockIdx.x - a.block_begin[mi]) * 32;
  const int lane = threadIdx.x & 31, grp = threadIdx.x >> 5;
  const int c = c0 + lane, R = a.rows[mi], Cn = a.cols[mi];
  float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
  if (c < Cn) {
    const float* p = a.m[mi] + c;
    int r = grp;
    for (; r + 96 < R; r += 128) {
      s0 += p[(long long)r * Cn];
      s1 += p[(long long)(r + 32) * Cn];
      s2 += p[(long long)(r + 64) * Cn];
      s3 += p[(long long)(r + 96) * Cn];
    }
    for (; r < R; r += 32) s0 += p[(long long)r * Cn];
  }
  red[threadIdx.x] = (s0 + s1) + (s2 + s3);
  __syncthreads();
  if (grp == 0 && c < Cn) {
    float t = 0.f;
#pragma unroll
    for (int g2 = 0; g2 < 32; ++g2) t += red[g2 * 32 + lane];
    a.out[mi][c] = t;
  }
}

// g_total = g * gscale + reg * p (where decay[i] != 0);  m, v, p updated in place (TF "epsilon hat" form).
// kNesterov: TF's NadamOptimizer (ApplyAdam with use_nesterov), the step takes b1 m + (1-b1) g_total in place of m.
template <bool kNesterov>
__global__ void k_adam_tf(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v,
                          const uint8_t* __restrict__ decay, const float* __restrict__ state, long long n, float b1,
                          float b2, float eps, float reg, float gscale) {
  const float lr_t = state[2];
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const float pi = p[i];
    float gi = g[i] * gscale;
    if (decay != nullptr && decay[i]) gi = fmaf(reg, pi, gi);
    const float mi = fmaf(1.f - b1, gi - m[i], m[i]);
    const float vi = fmaf(1.f - b2, gi * gi - v[i], v[i]);
    m[i] = mi;
    v[i] = vi;
    p[i] = pi - lr_t * (kNesterov ? fmaf(b1, mi, (1.f - b1) * gi) : mi) / (sqrtf(vi) + eps);
  }
}

}  // namespace gcnb

using namespace gcnb;

extern "C" {

int gcnb_softmax_xent_f32(const float* logits, const int64_t* labels, float* loss, float* dlogits, float* loss_rows,
                          int B, int C, float* adam_state, float lr, float beta1, float beta2, gcnb_stream_t stream) {
  GCNB_REQUIRE(logits && labels && loss && loss_rows && B >= 1 && C >= 1, "gcnb_softmax_xent_f32: bad arguments");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (B <= 64) {  // tiny batches: one CTA does everything (one launch)
    k_softmax_xent_1cta<<<1, 1024, 0, st>>>(logits, reinterpret_cast<const long long*>(labels), loss, dlogits, B, C,
                                            1.f / (float)B, adam_state, lr, beta1, beta2);
    GCNB_LAUNCH_CHECK("k_softmax_xent_1cta");
    return GCNB_OK;
  }
  k_softmax_xent<<<ceil_div(B * 32, 256), 256, 0, st>>>(logits, reinterpret_cast<const long long*>(labels), loss_rows,
                                                       dlogits, B, C, 1.f / (float)B);
  GCNB_LAUNCH_CHECK("k_softmax_xent");
  k_mean_rows<<<1, 256, 0, st>>>(loss_rows, loss, B, adam_state, lr, beta1, beta2);  // fixed-order mean + clock tick
  GCNB_LAUNCH_CHECK("k_mean_rows");
  return GCNB_OK;
}

int gcnb_relu_dropout_fwd_f32(float* x, long long rows, int cols, int ld, float keep, unsigned seed, const float* step,
                              gcnb_stream_t stream) {
  GCNB_REQUIRE(x && rows >= 1 && cols >= 1 && ld >= cols && keep > 0.f, "gcnb_relu_dropout_fwd_f32: bad arguments");
  const unsigned grid = (unsigned)std::max<long long>(1, std::min<long long>(ceil_div_ll(rows * cols, 256), 148 * 8));
  k_relu_dropout_fwd<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(x, rows, cols, ld, keep, 1.f / keep, seed, step);
  GCNB_LAUNCH_CHECK("k_relu_dropout_fwd");
  return GCNB_OK;
}

int gcnb_relu_dropout_bwd_f32(float* d, const float* act, long long rows, int cols, int ld_d, int ld_act, float keep,
                              gcnb_stream_t stream) {
  GCNB_REQUIRE(d && act && rows >= 1 && cols >= 1 && keep > 0.f, "gcnb_relu_dropout_bwd_f32: bad arguments");
  const unsigned grid = (unsigned)std::max<long long>(1, std::min<long long>(ceil_div_ll(rows * cols, 256), 148 * 8));
  k_relu_dropout_bwd<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(d, act, rows, cols, ld_d, ld_act,
                                                                           keep >= 1.f ? 1.f : 1.f / keep);
  GCNB_LAUNCH_CHECK("k_relu_dropout_bwd");
  return GCNB_OK;
}

int gcnb_colsum_multi_f32(const float* const* mats, float* const* outs, const int* rows, const int* cols, int count,
                          gcnb_stream_t stream) {
  GCNB_REQUIRE(mats && outs && rows && cols && count >= 1 && count <= 4, "gcnb_colsum_multi_f32: 1..4 matrices");
  ColsumArgs a;
  a.block_begin[0] = 0;
  for (int i = 0; i < 4; ++i) {
    const bool on = i < count;
    a.m[i] = on ? mats[i] : nullptr;
    a.out[i] = on ? outs[i] : nullptr;
    a.rows[i] = on ? rows[i] : 0;
    a.cols[i] = on ? cols[i] : 0;
    a.block_begin[i + 1] = a.block_begin[i] + (on ? ceil_div(cols[i], 32) : 0);
  }
  k_colsum_multi<<<a.block_begin[4], 1024, 0, static_cast<cudaStream_t>(stream)>>>(a);
  GCNB_LAUNCH_CHECK("k_colsum_multi");
  return GCNB_OK;
}

int gcnb_adam_tf_f32(float* p, const float* g, float* m, float* v, const uint8_t* decay, float* state, long long n,
                     float lr, float beta1, float beta2, float eps, float reg, float gscale, int tick,
                     gcnb_stream_t stream) {
  GCNB_REQUIRE(p && g && m && v && state && n >= 1, "gcnb_adam_tf_f32: bad arguments");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (tick) {
    k_adam_tick<<<1, 1, 0, st>>>(state, lr, beta1, beta2);
    GCNB_LAUNCH_CHECK("k_adam_tick");
  }
  const unsigned grid = (unsigned)std::max<long long>(1, std::min<long long>(ceil_div_ll(n, 256), 148 * 8));
  k_adam_tf<false><<<grid, 256, 0, st>>>(p, g, m, v, decay, state, n, beta1, beta2, eps, reg, gscale);
  GCNB_LAUNCH_CHECK("k_adam_tf");
  return GCNB_OK;
}

int gcnb_nadam_tf_f32(float* p, const float* g, float* m, float* v, const uint8_t* decay, float* state, long long n,
                      float lr, float beta1, float beta2, float eps, float reg, int tick, gcnb_stream_t stream) {
  GCNB_REQUIRE(p && g && m && v && state && n >= 1, "gcnb_nadam_tf_f32: bad arguments");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (tick) {
    k_adam_tick<<<1, 1, 0, st>>>(state, lr, beta1, beta2);
    GCNB_LAUNCH_CHECK("k_adam_tick");
  }
  const unsigned grid = (unsigned)std::max<long long>(1, std::min<long long>(ceil_div_ll(n, 256), 148 * 8));
  k_adam_tf<true><<<grid, 256, 0, st>>>(p, g, m, v, decay, state, n, beta1, beta2, eps, reg, 1.f);
  GCNB_LAUNCH_CHECK("k_adam_tf<true>");
  return GCNB_OK;
}

}  // extern "C"
