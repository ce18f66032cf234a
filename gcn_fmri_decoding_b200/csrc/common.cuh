// Shared helpers of the gcnb200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/gcnb200.h"

namespace gcnb {

void set_error(const char* fmt, ...);
void count_launch();  // diagnostic counter behind gcnb_launch_count()

#define GCNB_REQUIRE(cond, ...)      \
  do {                               \
    if (!(cond)) {                   \
      gcnb::set_error(__VA_ARGS__);  \
      return GCNB_ERR_INVALID;       \
    }                                \
  } while (0)

#define GCNB_CUDA(expr)                                                         \
  do {                                                                          \
    cudaError_t e_ = (expr);                                                    \
    if (e_ != cudaSuccess) {                                                    \
      gcnb::set_error("%s failed: %s", #expr, cudaGetErrorString(e_));          \
      return GCNB_ERR_CUDA;                                                     \
    }                                                                           \
  } while (0)

// Launch errors are surfaced right after enqueue; no synchronisation.
#define GCNB_LAUNCH_CHECK(name)                                                 \
  do {                                                                          \
    gcnb::count_launch();                                                       \
    cudaError_t e_ = cudaGetLastError();                                        \
    if (e_ != cudaSuccess) {                                                    \
      gcnb::set_error("launch of %s failed: %s", name, cudaGetErrorString(e_)); \
      return GCNB_ERR_CUDA;                                                     \
    }                                                                           \
  } while (0)

__host__ __device__ static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }
static inline int ceil_div(int a, int b) { return (a + b - 1) / b; }
static inline long long ceil_div_ll(long long a, long long b) { return (a + b - 1) / b; }

// Bump allocator over the caller's workspace.
struct Workspace {
  char* base;
  size_t size;
  size_t used;
  Workspace(void* p, size_t n) : base(static_cast<char*>(p)), size(n), used(0) {}
  template <typename T>
  T* take(size_t count) {
    size_t off = align_up(used, 256);
    size_t end = off + count * sizeof(T);
    used = end;
    if (end > size || base == nullptr) return nullptr;
    return reinterpret_cast<T*>(base + off);
  }
};

struct LayerShape {
  int B, M, nnz, Fin, Fout, K, p;
};

// Device properties the dispatch needs, queried once per device.
struct DeviceInfo {
  int sm_count;
  int smem_optin;
};
int device_info(DeviceInfo* out);

// ---- general (HBM-resident) path, general.cu ------------------------------------------------
size_t general_cheb_workspace(const LayerShape& s, bool backward, bool need_dx);
int general_cheb_fwd(const float* x, const int32_t* perm, int M_in, const gcnb_csr& L, const float* W,
                     const float* bias, float* y, uint8_t* argmax, float* xstack, const LayerShape& s, int bias_mode,
                     int relu, Workspace& ws, cudaStream_t st);
int general_cheb_bwd(const float* x, const int32_t* perm, int M_in, const float* y, const uint8_t* argmax, const float* dy, const gcnb_csr& L,
                     const gcnb_csr* Lt, const float* W, float* dx, float* dW, float* db, const float* xstack,
                     const LayerShape& s, int bias_mode, int relu, Workspace& ws, cudaStream_t st);

// pieces shared with the spectral path
int launch_to_node_major(const float* x, const int32_t* perm, float* X0, int B, int M, int M_in, int F,
                         cudaStream_t st);
int launch_from_node_major(const float* Xn, float* x, int B, int M, int F, cudaStream_t st);
int launch_epilogue(const float* Zn, const float* bias, float* y, uint8_t* argmax, int B, int M, int F, int p,
                    int bias_mode, int relu, cudaStream_t st);
// dZn rows (m*B + b) have a stride of ldz floats (>= F; padded for the tensor-core kernels of the general path)
int launch_dz(const float* dy, const float* y, const uint8_t* argmax, float* dZn, int ldz, int B, int M, int F, int p,
              int relu, cudaStream_t st);
size_t db_scratch_floats(int M, int F);
int launch_db(const float* dZn, int ldz, float* db, float* scratch, int B, int M, int F, int bias_mode, cudaStream_t st);

// ---- tensor-core contractions of the general path, general_mma.cu ---------------------------------
int node_mma_ldz(int Fout);
bool node_contract_supported(const LayerShape& s);
int node_contract(const float* Xs, long long slab, const float* W, const float* bias, float* out, const LayerShape& s,
                  int bias_mode, int relu, int direct, cudaStream_t st);
bool node_dw_supported(const LayerShape& s);
int node_dw_blocks(const LayerShape& s);
int node_dw(const float* Xs, long long slab, const float* dZ, float* part, const LayerShape& s, cudaStream_t st);
bool node_dz_wt_supported(const LayerShape& s);
int node_dz_wt(const float* dZ, const float* W, float* Gs, long long slab, const LayerShape& s, cudaStream_t st);

// ---- TMA-staged sparse recursion step for HBM-resident state, spmm_tma.cu -------------------------
bool spmm_tma_supported(const gcnb_csr& L, long long C, const float* src, const float* add, const float* add2,
                        const float* out);
int spmm_tma(const gcnb_csr& L, const float* src, const float* add, const float* add2, float* out, long long C,
             float alpha, float beta, float beta2, cudaStream_t st);

// ---- gradient w.r.t. the operator L~ (edge saliency), sddmm_tma.cu + general.cu ---------------------------------
// dval[b][e] (L~'s CSR order) and ddiag[b][i] from the basis stack X and the Clenshaw stack Bk (both [K][M][B*Fin],
// with 16 bytes of readable slack behind each); K >= 2
int sddmm_tma(const gcnb_csr& L, const float* X, const float* Bk, float* dval, float* ddiag, int accumulate,
              const LayerShape& s, cudaStream_t st);
size_t general_cheb_dL_workspace(const LayerShape& s);
int general_cheb_dL(const float* x, const int32_t* perm, int M_in, const float* y, const uint8_t* argmax, const float* dy,
                    const gcnb_csr& L, const gcnb_csr* Lt, const float* W, float* dval, float* ddiag, int accumulate,
                    float* dx, const LayerShape& s, int relu, Workspace& ws, cudaStream_t st);

// ---- gradient w.r.t. the adjacency (the chain through the normalisation and the coarsening), adjacency_grad.cu ----
size_t adjacency_grad_workspace(const gcnb_adj_level* levels, int nlevels, int B);
int adjacency_grad(const gcnb_adj_level* levels, int nlevels, const int32_t* edges, int E, float* out, int B,
                   int absolute, Workspace& ws, cudaStream_t st);

// ---- tcgen05 / TMEM forward for shared-memory resident graphs, cheb_fwd_umma.cu -------------------------
bool umma_fwd_supported(const LayerShape& s);
int umma_fwd_describe(const LayerShape& s, char* out, size_t n);  // 0 when the shape is not supported
int umma_cheb_fwd(const float* x, const int32_t* perm, int M_in, const gcnb_csr& L, const float* W, const float* bias,
                  float* y, uint8_t* argmax, float* y_mean, float* xstack, const LayerShape& s, int bias_mode, int relu,
                  cudaStream_t st);

// host-built operator image of the row-blocked kernels (layer = the layer's shape; adjoint: image of the transpose)
size_t cheb_image_bytes(const int32_t* rowptr, const int32_t* col, const LayerShape& layer, int adjoint);
int cheb_image_build(const int32_t* rowptr, const int32_t* col, const float* val, const LayerShape& layer, int adjoint,
                     void* out, size_t bytes);
// a stack of identical layers (p = 1, 32 -> 32, same operator image) in one launch
bool umma_stack_supported(const LayerShape& s, const gcnb_csr& L);
int umma_cheb_stack_fwd(const float* x, const gcnb_csr& L, const float* const* W, const float* const* bias,
                        const void* const* tap_images, float* y, int nlayers, const LayerShape& s, int bias_mode, int relu,
                        cudaStream_t st);
size_t cheb_tap_image_bytes(int Fin, int Fout, int K);
int cheb_tap_image_build(const float* W, int Fin, int Fout, int K, void* out, size_t bytes);
// input gradient dx of a layer through the same kernel (operator L~^T, taps W_k^T, dZ rebuilt from dy / y / argmax)
bool umma_adj_supported(const LayerShape& s);
int umma_cheb_adj(const float* dy, int dy_is_mean, const float* y, const uint8_t* argmax, const gcnb_csr& Lt, const float* W,
                  float* dx, const LayerShape& s, int relu, cudaStream_t st);
// ... for any input width Fin in [4, 32], dx stored row by row, row m to raw row perm[m] (perm nullable; rows with
// perm[m] >= M_in dropped): the input gradient of a first layer
bool umma_adj_raw_supported(const LayerShape& s);
int umma_adj_describe(const LayerShape& s, char* out, size_t n);  // 0 when the shape is not supported
int umma_cheb_adj_raw(const float* dy, int dy_is_mean, const float* y, const uint8_t* argmax, const gcnb_csr& Lt,
                      const float* W, float* dx, const int32_t* perm, int M_in, const LayerShape& s, int relu, cudaStream_t st);

// ---- fused (shared-memory resident) path, fused_fwd.cu / fused_bwd.cu ------------------------
bool fused_fwd_supported(const LayerShape& s);
bool fused_bwd_supported(const LayerShape& s, bool need_dx);
size_t fused_cheb_workspace(const LayerShape& s, bool backward, bool need_dx);
int fused_cheb_fwd(const float* x, const int32_t* perm, int M_in, const gcnb_csr& L, const float* W,
                   const float* bias, float* y, uint8_t* argmax, float* y_mean, float* xstack, const LayerShape& s,
                   int bias_mode, int relu, Workspace& ws, cudaStream_t st);
// padded feature width of the fused kernels' slabs / of the X_k stack (8, 16 or 32; 0 = not supported)
int fused_feature_pad(int Fin);
int launch_dw_from_partials(const float* part, float* dW, int nblocks, int K, int MT, int NT, int Fin, int Fout,
                            const float* db_part, float* db, int FoP, cudaStream_t st);
size_t db_vertex_workspace(const LayerShape& s);
int launch_db_vertex(const float* dy, const float* y, const uint8_t* argmax, float* db, const LayerShape& s, int relu,
                     int dy_is_mean, Workspace& ws, cudaStream_t st);
bool stack_dw_supported(const LayerShape& s);
size_t stack_dw_workspace(const LayerShape& s);
int stack_dw(const float* xstack, const float* y, const uint8_t* argmax, const float* dy, int dy_is_mean, float* dW,
             float* db, const LayerShape& s, int bias_mode, int relu, Workspace& ws, cudaStream_t st);
int fused_cheb_bwd(const float* x, const int32_t* perm, int M_in, const float* y, const uint8_t* argmax, const float* dy, const gcnb_csr& L,
                   const gcnb_csr* Lt, const float* W, float* dx, float* dW, float* db, const LayerShape& s,
                   int bias_mode, int relu, int dy_is_mean, bool skip_dw, Workspace& ws, cudaStream_t st);
int launch_gemm(const float* A, const float* B, float* C, const float* bias, int M, int N, int K, int lda, int ldb, int ldc,
                int ta, int tb, cudaStream_t st);
// GEMM with a fused element-wise epilogue (gemm.cu): GCNB_EPI_RELU_DROPOUT / GCNB_EPI_MASK, see gcnb_gemm_epilogue_f32
int launch_gemm_epi(const float* A, const float* B, float* C, const float* bias, int M, int N, int K, int lda, int ldb,
                    int ldc, int ta, int tb, int epilogue, const float* aux, int ld_aux, float keep, unsigned seed,
                    const float* step, cudaStream_t st);

// ---- counter-based dropout mask shared by k_relu_dropout_fwd (head.cu) and the GEMM epilogue (gemm.cu) ----------
__device__ __forceinline__ uint32_t mix32(uint32_t x) {  // murmur3 finaliser
  x ^= x >> 16;
  x *= 0x85ebca6bu;
  x ^= x >> 13;
  x *= 0xc2b2ae35u;
  x ^= x >> 16;
  return x;
}
// key of one (layer seed, optimiser step) pair; step = the Adam state vector (element 3 = step count) or NULL
__device__ __forceinline__ uint32_t dropout_key(uint32_t seed, const float* step) {
  return mix32(seed ^ mix32((uint32_t)(step ? step[3] : 0.f) + 0x9e3779b9u));
}
__device__ __forceinline__ uint32_t dropout_threshold(float keep) {
  return keep >= 1.f ? 0xffffffffu : (uint32_t)(keep * 4294967296.0);
}
// element i (row-major index within the activation matrix) survives iff this is true
__device__ __forceinline__ bool dropout_keeps(uint32_t i, uint32_t key, uint32_t thresh) {
  return mix32(i * 0x9e3779b1u + key) < thresh;
}
// ---- the classifier head as one persistent cooperative kernel, head_fused.cu ---------------------------------------
struct HeadParams {
  const float* a0;
  const long long* labels;
  const float *W1, *b1, *W2, *b2, *W3, *b3;
  float *logits, *loss;
  float *gW1, *gb1, *gW2, *gb2, *gW3, *gb3, *d0;
  // scratch
  float *h1, *h2, *d1, *d2, *d3, *part2, *partW2, *loss_rows, *part3, *part1, *part0;
  int B, n0, n1, n2, C;  // widths: a0 [B x n0], h1 [B x n1], h2 [B x n2], logits [B x C]
  float keep, inv_keep;
  unsigned seed1, seed2;
  float* state;  // optimiser clock {b1^t, b2^t, lr_t, t} (nullable); element 3 keys the dropout masks
  float lr, beta1, beta2;
  int tick;
};

bool head_step_supported(int B, int n0, int n1, int n2, int C);
size_t head_step_workspace(int B, int n0, int n1, int n2, int C);
int head_step(const HeadParams& P, Workspace& ws, cudaStream_t st);

int launch_mean_f(const float* x, float* y, long long rows, int F, cudaStream_t st);
int launch_mean_f_bwd(const float* dy, float* dx, long long rows, int F, cudaStream_t st);

}  // namespace gcnb
