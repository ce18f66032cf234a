// extern "C" entry points of libgcnb200.so: argument validation, kernel-family dispatch, and the
// small stand-alone kernels (b1relu/b2relu, mpool1, perm gather, mean over filters).
#include <algorithm>
#include <cstdlib>
#include <atomic>
#include <mutex>

#include "common.cuh"

namespace gcnb {

static thread_local char g_err[512] = "no error";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

static std::atomic<unsigned long long> g_launches{0};
void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }

bool pdl_enabled() {
  static const bool on = [] {
    // Off by default: measured on the config-2 step (B200, CUDA graph) 0.343 ms with the attribute vs 0.338 ms
    // without -- back-to-back launches of ONE kernel gain 3-5 %, the mixed chain of the step loses it again.
    const char* v = getenv("GCNB_PDL");
    return v && v[0] == '1';
  }();
  return on;
}

// GCNB_UMMA_ADJ=0 sends the input gradient back to k_cheb_bwd_fused (A/B runs); read once.
static bool adjoint_umma_enabled() {
  static const bool on = [] {
    const char* v = getenv("GCNB_UMMA_ADJ");
    return !(v && v[0] == '0');
  }();
  return on;
}

int device_info(DeviceInfo* out) {
  static std::mutex mu;
  static DeviceInfo cache[64];
  static bool have[64] = {false};
  int dev = 0;
  GCNB_CUDA(cudaGetDevice(&dev));
  if (dev < 0 || dev >= 64) {
    set_error("device ordinal %d out of range", dev);
    return GCNB_ERR_INVALID;
  }
  std::lock_guard<std::mutex> lock(mu);
  if (!have[dev]) {
    GCNB_CUDA(cudaDeviceGetAttribute(&cache[dev].sm_count, cudaDevAttrMultiProcessorCount, dev));
    GCNB_CUDA(cudaDeviceGetAttribute(&cache[dev].smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    have[dev] = true;
  }
  *out = cache[dev];
  return GCNB_OK;
}

// ------------------------------------------------------------------------------------------------
// stand-alone elementwise kernels
// ------------------------------------------------------------------------------------------------
__global__ void k_brelu_fwd(const float* __restrict__ x, const float* __restrict__ bias, float* __restrict__ y,
                            long long total, int M, int F, int bias_mode) {
  const long long MF = (long long)M * F;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    float v = x[i];
    if (bias_mode == GCNB_BIAS_PER_FILTER) v += bias[i % F];
    else if (bias_mode == GCNB_BIAS_PER_VERTEX) v += bias[i % MF];
    y[i] = fmaxf(v, 0.f);
  }
}

__global__ void k_brelu_bwd(const float* __restrict__ dy, const float* __restrict__ y, float* __restrict__ dx,
                            long long total) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x)
    dx[i] = y[i] > 0.f ? dy[i] : 0.f;
}

// db2[m*F+o] = sum_b dx[b][m][o]  (fixed order over b)
__global__ void k_bias_grad_vertex(const float* __restrict__ dx, float* __restrict__ db2, int B, long long MF) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < MF; i += (long long)gridDim.x * blockDim.x) {
    float s = 0.f;
    for (int b = 0; b < B; ++b) s += dx[(long long)b * MF + i];
    db2[i] = s;
  }
}

__global__ void k_bias_grad_filter(const float* __restrict__ db2, float* __restrict__ db, int M, int F) {
  const int o = blockIdx.x * blockDim.x + threadIdx.x;
  if (o >= F) return;
  float s = 0.f;
  for (int m = 0; m < M; ++m) s += db2[(long long)m * F + o];
  db[o] = s;
}

__global__ void k_mpool_fwd(const float* __restrict__ x, float* __restrict__ y, uint8_t* __restrict__ argmax, int B,
                            int M, int F, int p) {
  const int Mo = (M + p - 1) / p;
  const int before = (Mo * p - M) / 2;
  const long long total = (long long)B * Mo * F;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int o = (int)(i % F);
    const int j = (int)((i / F) % Mo);
    const int b = (int)(i / ((long long)F * Mo));
    float best = -INFINITY;
    int bi = 0;
    for (int w = 0; w < p; ++w) {
      const int m = j * p - before + w;
      if (m < 0 || m >= M) continue;
      const float v = x[((long long)b * M + m) * F + o];
      if (v > best) { best = v; bi = w; }
    }
    y[i] = best;
    if (argmax) argmax[i] = (uint8_t)bi;
  }
}

__global__ void k_mpool_bwd(const float* __restrict__ dy, const uint8_t* __restrict__ argmax, float* __restrict__ dx,
                            int B, int M, int F, int p) {
  const int Mo = (M + p - 1) / p;
  const int before = (Mo * p - M) / 2;
  const long long total = (long long)B * Mo * F;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int o = (int)(i % F);
    const int j = (int)((i / F) % Mo);
    const int b = (int)(i / ((long long)F * Mo));
    const int am = argmax[i];
    const float g = dy[i];
    for (int w = 0; w < p; ++w) {
      const int m = j * p - before + w;
      if (m < 0 || m >= M) continue;
      dx[((long long)b * M + m) * F + o] = (w == am) ? g : 0.f;
    }
  }
}

__global__ void k_perm_gather(const float* __restrict__ x, const int32_t* __restrict__ perm, float* __restrict__ y,
                              int B, int M_in, int M_out, int F) {
  const long long total = (long long)B * M_out * F;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int f = (int)(i % F);
    const int m = (int)((i / F) % M_out);
    const int b = (int)(i / ((long long)F * M_out));
    const int src = perm[m];
    y[i] = (src >= 0 && src < M_in) ? x[((long long)b * M_in + src) * F + f] : 0.f;
  }
}

// y[r] = mean_f x[r][f]  -- one warp per row, shuffle tree (fixed order)
__global__ void k_mean_f_fwd(const float* __restrict__ x, float* __restrict__ y, long long rows, int F) {
  const int lane = threadIdx.x & 31;
  const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long r = warp; r < rows; r += nwarps) {
    float s = 0.f;
    for (int f = lane; f < F; f += 32) s += x[r * F + f];
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) s += __shfl_xor_sync(0xffffffffu, s, d);
    if (lane == 0) y[r] = s / (float)F;
  }
}

__global__ void k_mean_f_bwd(const float* __restrict__ dy, float* __restrict__ dx, long long rows, int F) {
  const long long total = rows * F;
  const float inv = 1.f / (float)F;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x)
    dx[i] = dy[i / F] * inv;
}

static inline unsigned grid_for(long long total, int block = 256) {
  return (unsigned)std::max<long long>(1, std::min<long long>(ceil_div_ll(total, block), 148 * 16));
}

int launch_mean_f(const float* x, float* y, long long rows, int F, cudaStream_t st) {
  k_mean_f_fwd<<<grid_for(rows * 32), 256, 0, st>>>(x, y, rows, F);
  GCNB_LAUNCH_CHECK("k_mean_f_fwd");
  return GCNB_OK;
}

int launch_mean_f_bwd(const float* dy, float* dx, long long rows, int F, cudaStream_t st) {
  k_mean_f_bwd<<<grid_for(rows * F), 256, 0, st>>>(dy, dx, rows, F);
  GCNB_LAUNCH_CHECK("k_mean_f_bwd");
  return GCNB_OK;
}

static bool is_pow2(int v) { return v >= 1 && (v & (v - 1)) == 0; }

static int check_layer(const char* who, const gcnb_csr* L, int B, int Fin, int Fout, int K, int p, int bias_mode,
                       const float* bias) {
  GCNB_REQUIRE(L != nullptr && L->rowptr && (L->nnz == 0 || (L->col && L->val)), "%s: NULL operator", who);
  GCNB_REQUIRE(L->M >= 1 && L->nnz >= 0, "%s: bad operator size M=%d nnz=%d", who, L->M, L->nnz);
  GCNB_REQUIRE(B >= 1 && Fin >= 1 && Fout >= 1, "%s: B, Fin, Fout must be >= 1 (got %d, %d, %d)", who, B, Fin, Fout);
  GCNB_REQUIRE(K >= 1, "%s: polynomial order K must be >= 1 (got %d)", who, K);
  GCNB_REQUIRE(is_pow2(p) && p <= 128, "%s: pooling size must be a power of 2 in [1,128] (got %d)", who, p);
  GCNB_REQUIRE(bias_mode >= GCNB_BIAS_NONE && bias_mode <= GCNB_BIAS_PER_VERTEX, "%s: bad bias_mode %d", who, bias_mode);
  GCNB_REQUIRE(bias_mode == GCNB_BIAS_NONE || bias != nullptr, "%s: bias is NULL but bias_mode=%d", who, bias_mode);
  return GCNB_OK;
}

}  // namespace gcnb

using namespace gcnb;

extern "C" {

int gcnb_version(void) { return 100; }

const char* gcnb_last_error_string(void) { return g_err; }

unsigned long long gcnb_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

// Layout of the saved Chebyshev stack: 1 = fused kernels' [K][B][M][FP], 2 = general path's vertex-major
// [K][M][B][Fin] (graphs the fused kernels cannot hold), 0 = this shape keeps no stack.
static int stack_layout(const LayerShape& s) {
  if (fused_fwd_supported(s)) return stack_dw_supported(s) ? 1 : 0;
  return 2;
}

int gcnb_cheb_stack_width(int B, int M, int nnz, int Fin, int Fout, int K, int p) {
  LayerShape s{B, M, nnz, Fin, Fout, K, p};
  const int layout = stack_layout(s);
  return layout == 1 ? fused_feature_pad(Fin) : layout == 2 ? Fin : 0;
}

int gcnb_cheb_fwd_describe(int B, int M, int nnz, int Fin, int Fout, int K, int p, char* out, size_t n) {
  if (!out || n == 0) return GCNB_ERR_INVALID;
  LayerShape s{B, M, nnz, Fin, Fout, K, p};
  if (umma_fwd_describe(s, out, n) > 0) return GCNB_OK;
  snprintf(out, n, "%s", fused_fwd_supported(s) ? "k_cheb_fwd_fused: mma.sync, shared-memory resident"
                                                  : "general path: HBM-resident state (k_spmm_tma + k_stack_contract)");
  return GCNB_OK;
}

int gcnb_cheb_fused_supported(int B, int M, int nnz, int Fin, int Fout, int K, int p, int backward, int need_dx) {
  LayerShape s{B, M, nnz, Fin, Fout, K, p};
  return backward ? (fused_bwd_supported(s, need_dx != 0) ? 1 : 0) : (fused_fwd_supported(s) ? 1 : 0);
}

size_t gcnb_cheb_workspace_bytes(int B, int M, int nnz, int Fin, int Fout, int K, int p, int backward, int need_dx,
                                 int algo) {
  LayerShape s{B, M, nnz, Fin, Fout, K, p};
  const bool fused_ok = backward ? fused_bwd_supported(s, need_dx != 0) : fused_fwd_supported(s);
  // given the fused kernels' saved basis, a backward without dx runs stack_dw even where the fused backward does not fit
  // (gcnb_cheb_bwd_f32): its workspace must be there on the FUSED-unsupported and the general branch too (for every
  // algo on the latter, so that AUTO keeps asking for exactly what one of the two families asks for)
  const size_t stack_only = backward && !need_dx && stack_layout(s) == 1 ? stack_dw_workspace(s) + 512 : 0;
  if (algo == GCNB_ALGO_FUSED || (algo == GCNB_ALGO_AUTO && fused_ok))
    return fused_ok ? fused_cheb_workspace(s, backward != 0, need_dx != 0) + (backward ? stack_dw_workspace(s) + 512 : 0)
                    : stack_only;
  return general_cheb_workspace(s, backward != 0, need_dx != 0) +
         (backward ? align_up((size_t)B * ceil_div(M, p) * Fout * sizeof(float), 256) + 256 : 0) + stack_only;
}

int gcnb_cheb_fwd_f32(const float* x, const int32_t* perm, int M_in, const gcnb_csr* L, const float* W,
                      const float* bias, float* y, uint8_t* argmax, float* y_mean, float* xstack, int B, int Fin,
                      int Fout, int K, int p, int bias_mode, int relu, int algo, void* workspace,
                      size_t workspace_bytes, gcnb_stream_t stream) {
  int rc = check_layer("gcnb_cheb_fwd_f32", L, B, Fin, Fout, K, p, bias_mode, bias);
  if (rc) return rc;
  GCNB_REQUIRE(x && W && y, "gcnb_cheb_fwd_f32: x, W and y must not be NULL");
  GCNB_REQUIRE(perm != nullptr || M_in == L->M, "gcnb_cheb_fwd_f32: without perm, M_in (%d) must equal M (%d)", M_in,
               L->M);
  GCNB_REQUIRE(M_in >= 1, "gcnb_cheb_fwd_f32: M_in must be >= 1");
  LayerShape s{B, L->M, L->nnz, Fin, Fout, K, p};
  Workspace ws(workspace, workspace_bytes);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const bool fused_ok = fused_fwd_supported(s);
  if (algo == GCNB_ALGO_FUSED && !fused_ok) {
    set_error("gcnb_cheb_fwd_f32: fused kernels do not support B=%d M=%d nnz=%d Fin=%d Fout=%d K=%d p=%d", B, s.M,
              s.nnz, Fin, Fout, K, p);
    return GCNB_ERR_INVALID;
  }
  const long long pooled_rows = (long long)B * ceil_div(s.M, p);
  if (algo == GCNB_ALGO_FUSED || (algo == GCNB_ALGO_AUTO && fused_ok)) {
    // tensor-core (tcgen05/TMEM) kernel when the shape fits it; it writes the same xstack layout as the mma.sync one
    if (umma_fwd_supported(s) && (xstack == nullptr || stack_layout(s) == 1))
      return umma_cheb_fwd(x, perm, M_in, *L, W, bias, y, argmax, y_mean, xstack, s, bias_mode, relu, st);
    rc = fused_cheb_fwd(x, perm, M_in, *L, W, bias, y, argmax, y_mean, xstack, s, bias_mode, relu, ws, st);
    if (rc == GCNB_OK && y_mean != nullptr && Fout > 32) rc = launch_mean_f(y, y_mean, pooled_rows, Fout, st);
    return rc;
  }
  GCNB_REQUIRE(xstack == nullptr || stack_layout(s) == 2,
               "gcnb_cheb_fwd_f32: the general path cannot produce the stack layout gcnb_cheb_stack_width() announced");
  rc = general_cheb_fwd(x, perm, M_in, *L, W, bias, y, argmax, xstack, s, bias_mode, relu, ws, st);
  if (rc == GCNB_OK && y_mean != nullptr) rc = launch_mean_f(y, y_mean, pooled_rows, Fout, st);
  return rc;
}

int gcnb_cheb_stack_supported(const gcnb_csr* L, int B, int F, int K, int nlayers) {
  if (!L || B < 1 || K < 1 || nlayers < 1 || nlayers > 8 || L->M < 1) return 0;
  return umma_stack_supported(LayerShape{B, L->M, L->nnz, F, F, K, 1}, *L) ? 1 : 0;
}

size_t gcnb_cheb_tap_image_bytes(int Fin, int Fout, int K) { return cheb_tap_image_bytes(Fin, Fout, K); }

int gcnb_cheb_tap_image_build(const float* W_host, int Fin, int Fout, int K, void* image_host, size_t image_bytes) {
  return cheb_tap_image_build(W_host, Fin, Fout, K, image_host, image_bytes);
}

int gcnb_cheb_stack_fwd_f32(const float* x, const gcnb_csr* L, const float* const* W, const float* const* bias,
                            const void* const* tap_images, float* y, int nlayers, int B, int F, int K, int bias_mode,
                            int relu, gcnb_stream_t stream) {
  GCNB_REQUIRE(nlayers >= 1 && nlayers <= 8 && W != nullptr, "gcnb_cheb_stack_fwd_f32: 1..8 layers, W must not be NULL");
  int rc = check_layer("gcnb_cheb_stack_fwd_f32", L, B, F, F, K, 1, bias_mode,
                       bias_mode == GCNB_BIAS_NONE ? reinterpret_cast<const float*>(1) : (bias ? bias[0] : nullptr));
  if (rc) return rc;
  GCNB_REQUIRE(x && y, "gcnb_cheb_stack_fwd_f32: x and y must not be NULL");
  for (int l = 0; l < nlayers; ++l)
    GCNB_REQUIRE(W[l] != nullptr && (bias_mode == GCNB_BIAS_NONE || (bias && bias[l] != nullptr)),
                 "gcnb_cheb_stack_fwd_f32: W / bias of layer %d is NULL", l);
  LayerShape s{B, L->M, L->nnz, F, F, K, 1};
  if (!umma_stack_supported(s, *L)) {
    set_error("gcnb_cheb_stack_fwd_f32: needs F = 32, M %% 4 = 0 and the operator image of this layer shape in L->image "
              "(gcnb_cheb_image_build); got F=%d M=%d image=%s", F, L->M, L->image ? "yes" : "none");
    return GCNB_ERR_INVALID;
  }
  return umma_cheb_stack_fwd(x, *L, W, bias, tap_images, y, nlayers, s, bias_mode, relu, static_cast<cudaStream_t>(stream));
}

size_t gcnb_cheb_image_bytes(const int32_t* rowptr, const int32_t* col, int B, int M, int nnz, int Fin, int Fout, int K,
                             int p, int adjoint) {
  if (!rowptr || !col || B < 1 || M < 1 || nnz < 0 || Fin < 1 || Fout < 1 || K < 1 || p < 1) return 0;
  return cheb_image_bytes(rowptr, col, LayerShape{B, M, nnz, Fin, Fout, K, p}, adjoint);
}

int gcnb_cheb_image_build(const int32_t* rowptr, const int32_t* col, const float* val, int B, int M, int nnz, int Fin,
                          int Fout, int K, int p, int adjoint, void* image_host, size_t image_bytes) {
  GCNB_REQUIRE(rowptr && col && val && image_host && B >= 1 && M >= 1 && nnz >= 0 && Fin >= 1 && Fout >= 1 && K >= 1 && p >= 1,
               "gcnb_cheb_image_build: bad arguments");
  return cheb_image_build(rowptr, col, val, LayerShape{B, M, nnz, Fin, Fout, K, p}, adjoint, image_host, image_bytes);
}

int gcnb_cheb_bwd_f32(const float* x, const int32_t* perm, int M_in, const float* y, const uint8_t* argmax,
                      const float* dy, int dy_is_mean, const float* xstack, const gcnb_csr* L,
                      const gcnb_csr* Lt, const float* W, float* dx, float* dW, float* db, int B, int Fin,
                      int Fout, int K, int p, int bias_mode, int relu, int algo, void* workspace,
                      size_t workspace_bytes, gcnb_stream_t stream) {
  int rc = check_layer("gcnb_cheb_bwd_f32", L, B, Fin, Fout, K, p, bias_mode, reinterpret_cast<const float*>(1));
  if (rc) return rc;
  GCNB_REQUIRE(x && y && dy && W && dW, "gcnb_cheb_bwd_f32: x, y, dy, W and dW must not be NULL");
  GCNB_REQUIRE(p == 1 || argmax != nullptr, "gcnb_cheb_bwd_f32: argmax is required when p > 1");
  GCNB_REQUIRE(perm != nullptr || M_in == L->M, "gcnb_cheb_bwd_f32: without perm, M_in (%d) must equal M (%d)", M_in,
               L->M);
  GCNB_REQUIRE(bias_mode == GCNB_BIAS_NONE || db != nullptr, "gcnb_cheb_bwd_f32: db is NULL but bias_mode=%d", bias_mode);
  GCNB_REQUIRE(dx == nullptr || K == 1 || (Lt && Lt->M == L->M && Lt->nnz == L->nnz),
               "gcnb_cheb_bwd_f32: dx needs the transposed operator Lt with the same M and nnz");
  LayerShape s{B, L->M, L->nnz, Fin, Fout, K, p};
  Workspace ws(workspace, workspace_bytes);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int layout = xstack ? stack_layout(s) : 0;
  GCNB_REQUIRE(xstack == nullptr || layout != 0, "gcnb_cheb_bwd_f32: no stack layout exists for this shape");
  if (layout == 1 && dx == nullptr && algo != GCNB_ALGO_GENERAL)
    return stack_dw(xstack, y, argmax, dy, dy_is_mean, dW, db, s, bias_mode, relu, ws, st);
  const bool fused_ok = layout != 2 && fused_bwd_supported(s, dx != nullptr);
  if (layout == 1 && dx != nullptr && algo != GCNB_ALGO_GENERAL && fused_ok) {
    // saved basis: the weight gradient is one streamed GEMM; the fused kernel only runs the adjoint recursion for dx
    rc = stack_dw(xstack, y, argmax, dy, dy_is_mean, dW, db, s, bias_mode, relu, ws, st);
    if (rc) return rc;
    // dx = sum_k T_k(L~^T) dZ W_k^T: the tcgen05 forward kernel run on the transposed operator (cheb_fwd_umma.cu)
    if (K > 1 && algo == GCNB_ALGO_AUTO && umma_adj_supported(s) && adjoint_umma_enabled())
      return umma_cheb_adj(dy, dy_is_mean, y, argmax, *Lt, W, dx, s, relu, st);
    Workspace ws2(static_cast<char*>(workspace) + align_up(ws.used, 256), workspace_bytes - align_up(ws.used, 256));
    return fused_cheb_bwd(x, perm, M_in, y, argmax, dy, *L, Lt, W, dx, dW, db, s, bias_mode, relu, dy_is_mean, true, ws2, st);
  }
  if (algo == GCNB_ALGO_FUSED && !fused_ok) {
    set_error("gcnb_cheb_bwd_f32: fused kernels do not support B=%d M=%d nnz=%d Fin=%d Fout=%d K=%d p=%d", B, s.M,
              s.nnz, Fin, Fout, K, p);
    return GCNB_ERR_INVALID;
  }
  if (algo == GCNB_ALGO_FUSED || (algo == GCNB_ALGO_AUTO && fused_ok))
    return fused_cheb_bwd(x, perm, M_in, y, argmax, dy, *L, Lt, W, dx, dW, db, s, bias_mode, relu, dy_is_mean, false, ws, st);
  if (dy_is_mean) {  // the general path works on the full gradient: expand dy/Fout over the filters first
    const long long pooled_rows = (long long)B * ceil_div(s.M, p);
    float* full = ws.take<float>((size_t)pooled_rows * Fout);
    if (!full) {
      set_error("gcnb_cheb_bwd_f32: workspace too small");
      return GCNB_ERR_WORKSPACE;
    }
    rc = launch_mean_f_bwd(dy, full, pooled_rows, Fout, st);
    if (rc) return rc;
    dy = full;
  }
  return general_cheb_bwd(x, perm, M_in, y, argmax, dy, *L, Lt, W, dx, dW, db, layout == 2 ? xstack : nullptr, s,
                          bias_mode, relu, ws, st);
}

int gcnb_brelu_fwd_f32(const float* x, const float* bias, float* y, int B, int M, int F, int bias_mode,
                       gcnb_stream_t stream) {
  GCNB_REQUIRE(x && y && B >= 1 && M >= 1 && F >= 1, "gcnb_brelu_fwd_f32: bad arguments");
  GCNB_REQUIRE(bias_mode == GCNB_BIAS_NONE || bias, "gcnb_brelu_fwd_f32: bias is NULL");
  const long long total = (long long)B * M * F;
  k_brelu_fwd<<<grid_for(total), 256, 0, static_cast<cudaStream_t>(stream)>>>(x, bias, y, total, M, F, bias_mode);
  GCNB_LAUNCH_CHECK("k_brelu_fwd");
  return GCNB_OK;
}

int gcnb_brelu_bwd_f32(const float* dy, const float* y, float* dx, float* db, int B, int M, int F, int bias_mode,
                       void* workspace, size_t workspace_bytes, gcnb_stream_t stream) {
  GCNB_REQUIRE(dy && y && dx && B >= 1 && M >= 1 && F >= 1, "gcnb_brelu_bwd_f32: bad arguments");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const long long total = (long long)B * M * F, MF = (long long)M * F;
  k_brelu_bwd<<<grid_for(total), 256, 0, st>>>(dy, y, dx, total);
  GCNB_LAUNCH_CHECK("k_brelu_bwd");
  if (bias_mode == GCNB_BIAS_NONE || db == nullptr) return GCNB_OK;
  float* db2 = db;
  if (bias_mode == GCNB_BIAS_PER_FILTER) {
    Workspace ws(workspace, workspace_bytes);
    db2 = ws.take<float>((size_t)MF);
    if (!db2) {
      set_error("gcnb_brelu_bwd_f32: b1relu needs a workspace of M*F floats (+256 B)");
      return GCNB_ERR_WORKSPACE;
    }
  }
  k_bias_grad_vertex<<<grid_for(MF), 256, 0, st>>>(dx, db2, B, MF);
  GCNB_LAUNCH_CHECK("k_bias_grad_vertex");
  if (bias_mode == GCNB_BIAS_PER_FILTER) {
    k_bias_grad_filter<<<ceil_div(F, 128), 128, 0, st>>>(db2, db, M, F);
    GCNB_LAUNCH_CHECK("k_bias_grad_filter");
  }
  return GCNB_OK;
}

int gcnb_mpool_fwd_f32(const float* x, float* y, uint8_t* argmax, int B, int M, int F, int p, gcnb_stream_t stream) {
  GCNB_REQUIRE(x && y && B >= 1 && M >= 1 && F >= 1, "gcnb_mpool_fwd_f32: bad arguments");
  GCNB_REQUIRE(is_pow2(p) && p <= 128, "gcnb_mpool_fwd_f32: pooling size must be a power of 2 in [1,128] (got %d)", p);
  const long long total = (long long)B * ceil_div(M, p) * F;
  k_mpool_fwd<<<grid_for(total), 256, 0, static_cast<cudaStream_t>(stream)>>>(x, y, argmax, B, M, F, p);
  GCNB_LAUNCH_CHECK("k_mpool_fwd");
  return GCNB_OK;
}

int gcnb_mpool_bwd_f32(const float* dy, const uint8_t* argmax, float* dx, int B, int M, int F, int p,
                       gcnb_stream_t stream) {
  GCNB_REQUIRE(dy && argmax && dx && B >= 1 && M >= 1 && F >= 1, "gcnb_mpool_bwd_f32: bad arguments");
  GCNB_REQUIRE(is_pow2(p) && p <= 128, "gcnb_mpool_bwd_f32: pooling size must be a power of 2 in [1,128] (got %d)", p);
  const long long total = (long long)B * ceil_div(M, p) * F;
  k_mpool_bwd<<<grid_for(total), 256, 0, static_cast<cudaStream_t>(stream)>>>(dy, argmax, dx, B, M, F, p);
  GCNB_LAUNCH_CHECK("k_mpool_bwd");
  return GCNB_OK;
}

int gcnb_perm_gather_f32(const float* x, const int32_t* perm, float* y, int B, int M_in, int M_out, int F,
                         gcnb_stream_t stream) {
  GCNB_REQUIRE(x && perm && y && B >= 1 && M_in >= 1 && M_out >= M_in && F >= 1,
               "gcnb_perm_gather_f32: bad arguments (need M_out >= M_in, coarsening.py:254)");
  const long long total = (long long)B * M_out * F;
  k_perm_gather<<<grid_for(total), 256, 0, static_cast<cudaStream_t>(stream)>>>(x, perm, y, B, M_in, M_out, F);
  GCNB_LAUNCH_CHECK("k_perm_gather");
  return GCNB_OK;
}

int gcnb_mean_f_fwd_f32(const float* x, float* y, int rows, int F, gcnb_stream_t stream) {
  GCNB_REQUIRE(x && y && rows >= 1 && F >= 1, "gcnb_mean_f_fwd_f32: bad arguments");
  k_mean_f_fwd<<<grid_for((long long)rows * 32), 256, 0, static_cast<cudaStream_t>(stream)>>>(x, y, rows, F);
  GCNB_LAUNCH_CHECK("k_mean_f_fwd");
  return GCNB_OK;
}

int gcnb_mean_f_bwd_f32(const float* dy, float* dx, int rows, int F, gcnb_stream_t stream) {
  GCNB_REQUIRE(dy && dx && rows >= 1 && F >= 1, "gcnb_mean_f_bwd_f32: bad arguments");
  k_mean_f_bwd<<<grid_for((long long)rows * F), 256, 0, static_cast<cudaStream_t>(stream)>>>(dy, dx, rows, F);
  GCNB_LAUNCH_CHECK("k_mean_f_bwd");
  return GCNB_OK;
}

}  // extern "C"
