// extern "C" entry points of libgcnb200.so: argument validation, kernel-family dispatch, and the
// small stand-alone kernels (b1relu/b2relu, mpool1, perm gather, mean over filters).
#include <algorithm>
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

// the adjoint of k_perm_gather for a permutation: dx[b][perm[m]] = dxp[b][m] where perm[m] < M_in (every raw row is
// written exactly once, the rows of fake vertices are dropped)
__global__ void k_perm_scatter(const float* __restrict__ dxp, const int32_t* __restrict__ perm, float* __restrict__ dx,
                               int B, int M, int M_in, int F) {
  const long long total = (long long)B * M * F;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int f = (int)(i % F);
    const int m = (int)((i / F) % M);
    const int b = (int)(i / ((long long)F * M));
    const int dst = perm[m];
    if (dst >= 0 && dst < M_in) dx[((long long)b * M_in + dst) * F + f] = dxp[i];
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

// ------------------------------------------------------------------------------------------------
// Chebyshev layer plan: the one place that decides which kernels a call runs and the workspace they take.  The
// dispatch (gcnb_cheb_fwd_f32 / gcnb_cheb_bwd_f32) and every query (workspace, basis width, fused support, describe)
// read it.
// ------------------------------------------------------------------------------------------------
enum ChebRoute {
  ROUTE_UNSUPPORTED,
  ROUTE_FWD_UMMA,        // k_cheb_fwd_umma (tcgen05 / TMEM)
  ROUTE_FWD_FUSED,       // k_cheb_fwd_fused (mma.sync, shared-memory resident)
  ROUTE_GENERAL,         // HBM-resident state, forward or backward
  ROUTE_STACK_DW,        // dW / db streamed from the saved basis, no dx
  ROUTE_STACK_ADJ,       // ... and dx through k_cheb_fwd_umma on L~^T
  ROUTE_STACK_FUSED_DX,  // ... and dx through k_cheb_bwd_fused
  ROUTE_FUSED_BWD,       // k_cheb_bwd_fused recomputes the basis
  ROUTE_ADJ_ONLY,        // input gradient only: k_cheb_fwd_umma (RAW) on L~^T, any input width, un-permuted in its store
  ROUTE_FUSED_DX,        // input gradient only: k_cheb_bwd_fused without the weight gradient
};

struct ChebPlan {
  ChebRoute route;
  // saved basis of the shape (only when the call passes one): 1 = the fused kernels' [K][B][M][FP], 2 = the general
  // path's vertex-major [K][M][B][Fin] for graphs the fused kernels cannot hold, 0 = none exists
  int layout;
  // workspace regions of the route, in order; each a multiple of 256 bytes.  The input-gradient-only routes that run a
  // backward kernel (dx_only) put its unwanted weight gradient in region 2 and the permuted dx in region 3.
  size_t region[4];
  const char* why;   // ROUTE_UNSUPPORTED: the reason, NULL when the fused kernels do not fit the shape
  size_t total() const { return region[0] + region[1] + region[2] + region[3]; }
};

// dx_only (backward, need_dx, no saved basis): the input gradient alone, gcnb_cheb_dx_f32
static ChebPlan plan_cheb(const LayerShape& s, bool backward, bool need_dx, bool saved, int algo, bool dx_only = false) {
  ChebPlan pl{ROUTE_UNSUPPORTED, 0, {0, 0, 0, 0}, nullptr};
  auto route = [&pl](ChebRoute r, size_t a, size_t b = 0, size_t c = 0, size_t d = 0) {
    pl.route = r;
    pl.region[0] = a;
    pl.region[1] = b;
    pl.region[2] = c;
    pl.region[3] = d;
    return pl;
  };
  if (dx_only) {
    // the tcgen05 adjoint takes any input width; ALGO_FUSED keeps dx on k_cheb_bwd_fused, as in the full backward
    if (algo == GCNB_ALGO_AUTO && umma_adj_raw_supported(s)) return route(ROUTE_ADJ_ONLY, 0);
    const size_t dxp = align_up((size_t)s.B * s.M * s.Fin * sizeof(float), 256) + 256;
    const bool bwd_ok = fused_bwd_supported(s, true);
    if (algo == GCNB_ALGO_FUSED && !bwd_ok) return pl;
    if (algo == GCNB_ALGO_FUSED || (algo == GCNB_ALGO_AUTO && bwd_ok))
      return route(ROUTE_FUSED_DX, fused_cheb_workspace(s, true, true), 0, 0, dxp);
    return route(ROUTE_GENERAL, general_cheb_workspace(s, true, true),
                 align_up((size_t)s.B * ceil_div(s.M, s.p) * s.Fout * sizeof(float), 256) + 256,
                 align_up((size_t)s.Fin * s.K * s.Fout * sizeof(float), 256) + 256, dxp);
  }
  const bool fwd_ok = fused_fwd_supported(s);
  if (saved) pl.layout = fwd_ok ? (stack_dw_supported(s) ? 1 : 0) : 2;
  if (!backward) {
    if (algo == GCNB_ALGO_FUSED && !fwd_ok) return pl;
    // the tcgen05 kernel writes the same basis layout as the mma.sync one, where that layout exists
    if (algo == GCNB_ALGO_FUSED || (algo == GCNB_ALGO_AUTO && fwd_ok))
      return route(umma_fwd_supported(s) && (!saved || pl.layout == 1) ? ROUTE_FWD_UMMA : ROUTE_FWD_FUSED,
                   fused_cheb_workspace(s, false, false));
    if (saved && pl.layout != 2) {
      pl.why = "the general path cannot produce the stack layout gcnb_cheb_stack_width() announced";
      return pl;
    }
    return route(ROUTE_GENERAL, general_cheb_workspace(s, false, false));
  }
  if (saved && pl.layout == 0) {
    pl.why = "no stack layout exists for this shape";
    return pl;
  }
  // the fused kernels' saved basis: the weight gradient is one streamed GEMM (ALGO_GENERAL recomputes instead), also
  // where the fused backward does not fit
  const bool stack = pl.layout == 1 && algo != GCNB_ALGO_GENERAL;
  const size_t sdw = stack ? stack_dw_workspace(s) + 512 : 0;
  if (stack && !need_dx) return route(ROUTE_STACK_DW, sdw);
  const bool bwd_ok = pl.layout != 2 && fused_bwd_supported(s, need_dx);
  const size_t fw = bwd_ok ? fused_cheb_workspace(s, true, need_dx) : 0;
  if (stack && bwd_ok) {  // only dx needs the adjoint recursion; ALGO_FUSED keeps it on k_cheb_bwd_fused
    if (s.K > 1 && algo == GCNB_ALGO_AUTO && umma_adj_supported(s)) return route(ROUTE_STACK_ADJ, sdw);
    return route(ROUTE_STACK_FUSED_DX, sdw, fw);
  }
  if (algo == GCNB_ALGO_FUSED && !bwd_ok) return pl;
  if (algo == GCNB_ALGO_FUSED || (algo == GCNB_ALGO_AUTO && bwd_ok)) return route(ROUTE_FUSED_BWD, fw);
  // the general path works on the full gradient: a dy given as the mean over the filters is expanded first
  return route(ROUTE_GENERAL, general_cheb_workspace(s, true, need_dx),
               align_up((size_t)s.B * ceil_div(s.M, s.p) * s.Fout * sizeof(float), 256) + 256);
}

// region i of the plan in the caller's workspace
static Workspace plan_region(const ChebPlan& pl, int i, void* workspace, size_t bytes) {
  size_t off = 0;
  for (int r = 0; r < i; ++r) off += pl.region[r];
  if (workspace == nullptr || off >= bytes) return Workspace(nullptr, 0);
  return Workspace(static_cast<char*>(workspace) + off, std::min(pl.region[i], bytes - off));
}

static int plan_error(const char* who, const ChebPlan& pl, const LayerShape& s) {
  if (pl.why)
    set_error("%s: %s", who, pl.why);
  else
    set_error("%s: fused kernels do not support B=%d M=%d nnz=%d Fin=%d Fout=%d K=%d p=%d", who, s.B, s.M, s.nnz, s.Fin,
              s.Fout, s.K, s.p);
  return GCNB_ERR_INVALID;
}

static void plan_describe(const ChebPlan& pl, const LayerShape& s, bool backward, char* out, size_t n) {
  switch (pl.route) {
    case ROUTE_FWD_UMMA:
      umma_fwd_describe(s, out, n);
      return;
    case ROUTE_FWD_FUSED:
      snprintf(out, n, "k_cheb_fwd_fused: mma.sync, shared-memory resident");
      return;
    case ROUTE_GENERAL:
      snprintf(out, n, "%s", backward ? "general path: HBM-resident state (k_spmm_tma + k_node_dw, k_dz_wt for dx)"
                                      : "general path: HBM-resident state (k_spmm_tma + k_stack_contract)");
      return;
    case ROUTE_STACK_DW:
      snprintf(out, n, "stack-dW: k_dw_from_stack + k_dw_from_partials");
      return;
    case ROUTE_STACK_ADJ:
      snprintf(out, n, "stack-dW + tcgen05 adjoint: k_dw_from_stack + k_dw_from_partials, dx by k_cheb_fwd_umma on L~^T");
      return;
    case ROUTE_STACK_FUSED_DX:
      snprintf(out, n, "stack-dW + fused dx: k_dw_from_stack + k_dw_from_partials, dx by k_cheb_bwd_fused");
      return;
    case ROUTE_FUSED_BWD:
      snprintf(out, n, "fused recompute: k_cheb_bwd_fused + k_dw_from_partials");
      return;
    default:
      snprintf(out, n, "unsupported: %s", pl.why ? pl.why : "the fused kernels do not fit this shape");
  }
}

}  // namespace gcnb

using namespace gcnb;

extern "C" {

int gcnb_version(void) { return 104; }

const char* gcnb_last_error_string(void) { return g_err; }

unsigned long long gcnb_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

int gcnb_cheb_stack_width(int B, int M, int nnz, int Fin, int Fout, int K, int p) {
  LayerShape s{B, M, nnz, Fin, Fout, K, p};
  const int layout = plan_cheb(s, false, false, true, GCNB_ALGO_AUTO).layout;
  return layout == 1 ? fused_feature_pad(Fin) : layout == 2 ? Fin : 0;
}

int gcnb_cheb_describe(int B, int M, int nnz, int Fin, int Fout, int K, int p, int backward, int need_dx, int saved_basis,
                       int algo, char* out, size_t n, size_t* route_workspace_bytes) {
  if (!out || n == 0) return GCNB_ERR_INVALID;
  LayerShape s{B, M, nnz, Fin, Fout, K, p};
  const ChebPlan pl = plan_cheb(s, backward != 0, need_dx != 0, saved_basis != 0, algo);
  plan_describe(pl, s, backward != 0, out, n);
  if (route_workspace_bytes) *route_workspace_bytes = pl.total();
  return GCNB_OK;
}

int gcnb_cheb_fused_supported(int B, int M, int nnz, int Fin, int Fout, int K, int p, int backward, int need_dx) {
  LayerShape s{B, M, nnz, Fin, Fout, K, p};
  return plan_cheb(s, backward != 0, need_dx != 0, false, GCNB_ALGO_FUSED).route != ROUTE_UNSUPPORTED;
}

size_t gcnb_cheb_workspace_bytes(int B, int M, int nnz, int Fin, int Fout, int K, int p, int backward, int need_dx,
                                 int algo) {
  LayerShape s{B, M, nnz, Fin, Fout, K, p};
  return std::max(plan_cheb(s, backward != 0, need_dx != 0, false, algo).total(),
                  plan_cheb(s, backward != 0, need_dx != 0, true, algo).total());
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
  const ChebPlan pl = plan_cheb(s, false, false, xstack != nullptr, algo);
  Workspace ws = plan_region(pl, 0, workspace, workspace_bytes);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const long long pooled_rows = (long long)B * ceil_div(s.M, p);
  switch (pl.route) {
    case ROUTE_FWD_UMMA:
      return umma_cheb_fwd(x, perm, M_in, *L, W, bias, y, argmax, y_mean, xstack, s, bias_mode, relu, st);
    case ROUTE_FWD_FUSED:
      rc = fused_cheb_fwd(x, perm, M_in, *L, W, bias, y, argmax, y_mean, xstack, s, bias_mode, relu, ws, st);
      if (rc == GCNB_OK && y_mean != nullptr && Fout > 32) rc = launch_mean_f(y, y_mean, pooled_rows, Fout, st);
      return rc;
    case ROUTE_GENERAL:
      rc = general_cheb_fwd(x, perm, M_in, *L, W, bias, y, argmax, xstack, s, bias_mode, relu, ws, st);
      if (rc == GCNB_OK && y_mean != nullptr) rc = launch_mean_f(y, y_mean, pooled_rows, Fout, st);
      return rc;
    default:
      return plan_error("gcnb_cheb_fwd_f32", pl, s);
  }
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
  const ChebPlan pl = plan_cheb(s, true, dx != nullptr, xstack != nullptr, algo);
  Workspace ws = plan_region(pl, 0, workspace, workspace_bytes), ws1 = plan_region(pl, 1, workspace, workspace_bytes);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  switch (pl.route) {
    case ROUTE_STACK_DW:
    case ROUTE_STACK_ADJ:
    case ROUTE_STACK_FUSED_DX:
      rc = stack_dw(xstack, y, argmax, dy, dy_is_mean, dW, db, s, bias_mode, relu, ws, st);
      if (rc || pl.route == ROUTE_STACK_DW) return rc;
      // dx = sum_k T_k(L~^T) dZ W_k^T: the tcgen05 forward kernel run on the transposed operator (cheb_fwd_umma.cu)
      if (pl.route == ROUTE_STACK_ADJ) return umma_cheb_adj(dy, dy_is_mean, y, argmax, *Lt, W, dx, s, relu, st);
      return fused_cheb_bwd(x, perm, M_in, y, argmax, dy, *L, Lt, W, dx, dW, db, s, bias_mode, relu, dy_is_mean, true, ws1, st);
    case ROUTE_FUSED_BWD:
      return fused_cheb_bwd(x, perm, M_in, y, argmax, dy, *L, Lt, W, dx, dW, db, s, bias_mode, relu, dy_is_mean, false, ws, st);
    case ROUTE_GENERAL:
      if (dy_is_mean) {
        const long long pooled_rows = (long long)B * ceil_div(s.M, p);
        float* full = ws1.take<float>((size_t)pooled_rows * Fout);
        if (!full) {
          set_error("gcnb_cheb_bwd_f32: workspace too small");
          return GCNB_ERR_WORKSPACE;
        }
        rc = launch_mean_f_bwd(dy, full, pooled_rows, Fout, st);
        if (rc) return rc;
        dy = full;
      }
      return general_cheb_bwd(x, perm, M_in, y, argmax, dy, *L, Lt, W, dx, dW, db, pl.layout == 2 ? xstack : nullptr, s,
                              bias_mode, relu, ws, st);
    default:
      return plan_error("gcnb_cheb_bwd_f32", pl, s);
  }
}

int gcnb_cheb_dx_describe(int B, int M, int nnz, int Fin, int Fout, int K, int p, int algo, char* out, size_t n,
                          size_t* workspace_bytes) {
  if (!out || n == 0) return GCNB_ERR_INVALID;
  LayerShape s{B, M, nnz, Fin, Fout, K, p};
  const ChebPlan pl = plan_cheb(s, true, true, false, algo, true);
  switch (pl.route) {
    case ROUTE_ADJ_ONLY: {
      const int w = snprintf(out, n, "tcgen05 adjoint only: ");
      if (w >= 0 && (size_t)w < n) umma_adj_describe(s, out + w, n - w);
      break;
    }
    case ROUTE_FUSED_DX:
      snprintf(out, n, "fused dx: k_cheb_bwd_fused without the weight gradient, k_perm_scatter with perm");
      break;
    case ROUTE_GENERAL:
      snprintf(out, n, "general path: HBM-resident state (k_spmm_tma, k_dz_wt for dx; dW to scratch), k_perm_scatter "
                       "with perm");
      break;
    default:
      plan_describe(pl, s, true, out, n);
  }
  if (workspace_bytes) *workspace_bytes = pl.total();
  return GCNB_OK;
}

int gcnb_cheb_dx_f32(const float* x, const int32_t* perm, int M_in, const float* y, const uint8_t* argmax,
                     const float* dy, int dy_is_mean, const gcnb_csr* L, const gcnb_csr* Lt, const float* W, float* dx,
                     int B, int Fin, int Fout, int K, int p, int relu, int algo, void* workspace, size_t workspace_bytes,
                     gcnb_stream_t stream) {
  int rc = check_layer("gcnb_cheb_dx_f32", L, B, Fin, Fout, K, p, GCNB_BIAS_NONE, nullptr);
  if (rc) return rc;
  GCNB_REQUIRE(y && dy && W && dx, "gcnb_cheb_dx_f32: y, dy, W and dx must not be NULL");
  GCNB_REQUIRE(p == 1 || argmax != nullptr, "gcnb_cheb_dx_f32: argmax is required when p > 1");
  GCNB_REQUIRE(M_in >= 1 && (perm != nullptr || M_in == L->M),
               "gcnb_cheb_dx_f32: without perm, M_in (%d) must equal M (%d)", M_in, L->M);
  GCNB_REQUIRE(K == 1 || (Lt && Lt->M == L->M && Lt->nnz == L->nnz),
               "gcnb_cheb_dx_f32: needs the transposed operator Lt with the same M and nnz");
  LayerShape s{B, L->M, L->nnz, Fin, Fout, K, p};
  const ChebPlan pl = plan_cheb(s, true, true, false, algo, true);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (pl.route == ROUTE_ADJ_ONLY) {
    // K = 1 applies no operator: L only provides the kernel's row tables (its image belongs to the forward shape)
    gcnb_csr op = Lt ? *Lt : *L;
    if (!Lt) op.image = nullptr, op.image_bytes = 0;
    return umma_cheb_adj_raw(dy, dy_is_mean, y, argmax, op, W, dx, perm, M_in, s, relu, st);
  }
  if (pl.route != ROUTE_FUSED_DX && pl.route != ROUTE_GENERAL) return plan_error("gcnb_cheb_dx_f32", pl, s);
  GCNB_REQUIRE(pl.route != ROUTE_GENERAL || x != nullptr,
               "gcnb_cheb_dx_f32: the general path recomputes the Chebyshev basis and needs x");
  Workspace ws = plan_region(pl, 0, workspace, workspace_bytes), ws1 = plan_region(pl, 1, workspace, workspace_bytes);
  Workspace ws2 = plan_region(pl, 2, workspace, workspace_bytes), ws3 = plan_region(pl, 3, workspace, workspace_bytes);
  float* dxp = perm ? ws3.take<float>((size_t)B * s.M * Fin) : dx;  // gradient w.r.t. the permuted input
  if (!dxp) {
    set_error("gcnb_cheb_dx_f32: workspace too small");
    return GCNB_ERR_WORKSPACE;
  }
  if (pl.route == ROUTE_FUSED_DX) {
    rc = fused_cheb_bwd(x, perm, M_in, y, argmax, dy, *L, Lt, W, dxp, nullptr, nullptr, s, GCNB_BIAS_NONE, relu, dy_is_mean,
                        true, ws, st);
  } else {
    float* dW = ws2.take<float>((size_t)Fin * K * Fout);
    float* full = dy_is_mean ? ws1.take<float>((size_t)B * ceil_div(s.M, p) * Fout) : nullptr;
    if (!dW || (dy_is_mean && !full)) {
      set_error("gcnb_cheb_dx_f32: workspace too small");
      return GCNB_ERR_WORKSPACE;
    }
    if (dy_is_mean) {
      rc = launch_mean_f_bwd(dy, full, (long long)B * ceil_div(s.M, p), Fout, st);
      if (rc) return rc;
      dy = full;
    }
    rc = general_cheb_bwd(x, perm, M_in, y, argmax, dy, *L, Lt, W, dxp, dW, nullptr, nullptr, s, GCNB_BIAS_NONE, relu, ws,
                          st);
  }
  if (rc || !perm) return rc;
  k_perm_scatter<<<grid_for((long long)B * s.M * Fin), 256, 0, st>>>(dxp, perm, dx, B, s.M, M_in, Fin);
  GCNB_LAUNCH_CHECK("k_perm_scatter");
  return GCNB_OK;
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
