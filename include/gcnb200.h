/*
 * gcnb200.h -- C ABI of the B200 (sm_100a) graph-convolution kernels.
 *
 * This is the drop-in boundary for the graph-convolution hot path of
 * zhangyu2ustc/GCN_fmri_decoding.  The reference has no FFI: its layers are Python
 * methods that emit TensorFlow-1.x ops (lib_new/models_gcn.py).  Each entry point below
 * replaces the TF op sequence of one reference method (cited per function); the Python
 * host side (gcn_fmri_decoding_b200/_lib.py, ops.py) binds them with ctypes and mirrors
 * the reference's method names and arguments.  INTEGRATION.md shows the stub a
 * maintainer of the reference would add.
 *
 * Conventions
 *  - plain pointers and sizes only; every pointer is a DEVICE pointer unless named h_*.
 *  - tensors are dense, row-major, fp32: x[B][M][Fin], y[B][Mo][Fout] with Mo = ceil(M/p).
 *  - the caller owns every buffer, including the workspace (size from *_workspace_bytes);
 *    the library never allocates or frees device memory and keeps no pointer after return.
 *  - all work is enqueued on `stream` (a cudaStream_t); no host synchronisation, no
 *    allocation, no stream creation inside: every call is CUDA-graph capturable.
 *  - return value: GCNB_OK (0) or a negative code; gcnb_last_error_string() (thread local)
 *    describes the last failure.  Nothing throws or aborts.
 *  - re-entrant; no global mutable state besides the thread-local error string and the
 *    one-time per-device kernel attribute setup.
 */
#ifndef GCNB200_H
#define GCNB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define GCNB_API __attribute__((visibility("default")))
#else
#define GCNB_API
#endif

#define GCNB_OK 0
#define GCNB_ERR_INVALID (-1)   /* bad argument / unsupported shape */
#define GCNB_ERR_WORKSPACE (-2) /* workspace too small or misaligned */
#define GCNB_ERR_CUDA (-3)      /* a CUDA runtime call or launch failed */

/* bias_mode: how the bias of b1relu / b2relu is indexed (models_gcn.py:619-629) */
#define GCNB_BIAS_NONE 0
#define GCNB_BIAS_PER_FILTER 1 /* b1relu: bias[Fout]    */
#define GCNB_BIAS_PER_VERTEX 2 /* b2relu: bias[M][Fout] */

/* algo: kernel family selection.  AUTO picks FUSED when the graph and a tile of samples
 * fit in shared memory, GENERAL (HBM-resident operator and state) otherwise. */
#define GCNB_ALGO_AUTO 0
#define GCNB_ALGO_GENERAL 1
#define GCNB_ALGO_FUSED 2

typedef void* gcnb_stream_t; /* cudaStream_t */

/* A rescaled Laplacian L~ = L/(lmax/2) - I in CSR (graph.py:146-152 output, rows sorted by
 * column as tf.sparse_reorder leaves them, models_gcn.py:593-596).  Device arrays. */
typedef struct gcnb_csr {
  const int32_t* rowptr; /* [M+1] */
  const int32_t* col;    /* [nnz] */
  const float* val;      /* [nnz] */
  int32_t M;
  int32_t nnz;
  /* Optional (NULL / 0 = none): operator image pre-built on the host by gcnb_cheb_image_build for ONE layer shape
   * and uploaded by the caller (16-byte aligned device memory).  The tcgen05 kernels then copy it instead of
   * re-deriving their row-blocked work lists from the CSR arrays in every launch.  The CSR arrays stay mandatory
   * (other kernels read them) and must describe the same matrix. */
  const void* image;
  size_t image_bytes;
} gcnb_csr;

GCNB_API int gcnb_version(void);
GCNB_API const char* gcnb_last_error_string(void);
/* Number of kernels this library has enqueued in this process so far (diagnostic; monotonic). */
GCNB_API unsigned long long gcnb_launch_count(void);

/* 1 if the fused shared-memory kernels can take this layer shape, else 0 (no reference counterpart: dispatch query). */
GCNB_API int gcnb_cheb_fused_supported(int B, int M, int nnz, int Fin, int Fout, int K, int p, int backward, int need_dx);

/* Human-readable description of the route gcnb_cheb_fwd_f32 (backward = 0) or gcnb_cheb_bwd_f32 (backward = 1) takes
 * for this shape: "<route>: <its kernels>" (diagnostics, bench records).  saved_basis: the call passes `xstack`.
 * route_workspace_bytes (nullable) receives the workspace that route takes; gcnb_cheb_workspace_bytes is the largest
 * of these over saved_basis = 0 and 1. */
GCNB_API int gcnb_cheb_describe(int B, int M, int nnz, int Fin, int Fout, int K, int p, int backward, int need_dx,
                                int saved_basis, int algo, char* out, size_t n, size_t* route_workspace_bytes);

/*
 * Operator image of a layer (see gcnb_csr.image) -- the counterpart of turning the rescaled Laplacian into a
 * tf.SparseTensor once per graph build (models_gcn.py:590-596).  rowptr / col / val are HOST arrays of the rescaled Laplacian the
 * layer is called with -- for adjoint != 0 of its TRANSPOSE, and the image then serves the input gradient of
 * gcnb_cheb_bwd_f32 (pass it in Lt->image).  The shape arguments are the layer's (the same as in the fwd / bwd call);
 * an image is only valid for that shape on that device model.  gcnb_cheb_image_bytes returns 0 when no image-based
 * kernel exists for the shape (the calls then work without an image).  No CUDA calls besides a device-property query.
 */
GCNB_API size_t gcnb_cheb_image_bytes(const int32_t* rowptr, const int32_t* col, int B, int M, int nnz, int Fin, int Fout,
                                      int K, int p, int adjoint);
GCNB_API int gcnb_cheb_image_build(const int32_t* rowptr, const int32_t* col, const float* val, int B, int M, int nnz,
                                   int Fin, int Fout, int K, int p, int adjoint, void* image_host, size_t image_bytes);

/*
 * A stack of `nlayers` (1..8) identical ChebyNet layers in ONE launch -- the reference's production network is six
 * such layers (model.py:271-274; conv loop models_gcn.py:658-668): same operator, p = 1 (no pooling), F -> F filters
 * with F = 32, the same K / bias mode / ReLU, weights W[l] [F*K, F] and biases bias[l] per layer (host arrays of
 * device pointers).  x [B, M, F] -> y [B, M, F]; the activations between the layers stay on the SM.  Needs the
 * operator image of the layer shape in L->image (gcnb_cheb_image_build(..., Fin = Fout = F, p = 1, adjoint = 0));
 * results are bit-identical to nlayers calls of gcnb_cheb_fwd_f32.  Inference only (no arg-max, no saved basis).
 * tap_images (NULL, or a host array of nlayers device pointers, entries may be NULL): pre-split tap images of the
 * layers' weights (gcnb_cheb_tap_image_build, uploaded by the caller, 16-byte aligned) -- the kernel then copies a
 * layer's taps with one bulk copy instead of splitting W at every layer boundary.  An image belongs to the weight
 * values it was built from.
 */
GCNB_API int gcnb_cheb_stack_supported(const gcnb_csr* L, int B, int F, int K, int nlayers);
GCNB_API int gcnb_cheb_stack_fwd_f32(const float* x, const gcnb_csr* L, const float* const* W, const float* const* bias,
                                     const void* const* tap_images, float* y, int nlayers, int B, int F, int K,
                                     int bias_mode, int relu, gcnb_stream_t stream);
/* Host side: the three tap arrays of a layer (tf32 hi / lo parts and the bf16 image of W [Fin*K, Fout]) in the
 * kernel's shared-memory layout, bit for bit what the kernel derives from W itself.  _bytes returns 0 for widths the
 * tcgen05 kernel does not take. */
GCNB_API size_t gcnb_cheb_tap_image_bytes(int Fin, int Fout, int K);
GCNB_API int gcnb_cheb_tap_image_build(const float* W_host, int Fin, int Fout, int K, void* image_host, size_t image_bytes);

/* Feature width FP of the saved-basis buffer `xstack` (K*B*M*FP floats, layout private to the library: [K][B][M][FP]
 * with padded FP for graphs the fused kernels hold in shared memory, vertex-major [K][M][B][Fin] for vertex-level
 * graphs on the general path), or 0 when this shape keeps no basis. */
GCNB_API int gcnb_cheb_stack_width(int B, int M, int nnz, int Fin, int Fout, int K, int p);

/* Bytes of workspace gcnb_cheb_{fwd,bwd}_f32 need for this shape and algo, with or without a saved basis (256-byte
 * aligned pointer). */
GCNB_API size_t gcnb_cheb_workspace_bytes(int B, int M, int nnz, int Fin, int Fout, int K, int p, int backward, int need_dx,
                                 int algo);

/*
 * Fused ChebyNet layer, forward:  filter -> bias -> ReLU -> max-pool.
 * Replaces cgcnn.chebyshev5 (models_gcn.py:587-617) / cgcnn.chebyshev2 (:558-585, same math)
 * followed by b1relu/b2relu (:619-629) and mpool1 (:631-639), i.e. one iteration of the
 * conv loop at :658-668.
 *
 *   X_0 = x, X_1 = L~ X_0, X_k = 2 L~ X_{k-1} - X_{k-2}
 *   z[b,m,o] = sum_{f,k} X_k[b,m,f] * W[f*K + k, o]          (W row order of :611-615)
 *   a = relu ? max(z + bias, 0) : z + bias
 *   y[b,j,o] = max_{i<p} a[b, j*p+i, o],  argmax[b,j,o] = first i attaining it (uint8)
 *
 * perm (nullable): if given, x is the un-permuted data x_raw[B][M_in][Fin] and the kernel reads
 *   row perm[m] (zero when perm[m] >= M_in) -- coarsening.perm_data_3d (coarsening.py:244-265)
 *   fused into the load.  With perm == NULL, M_in must equal M.
 * bias (nullable iff bias_mode == NONE); argmax (nullable: not written); p >= 1, power of 2.
 * y_mean (nullable): also write mean_o y[b,j,o] as [B][M/p] -- tf.reduce_mean(x, -1) of the last conv layer
 *   (models_gcn.py:673) fused into the epilogue.
 * xstack (nullable, training): also keep the Chebyshev basis X_k, k < K, in a caller buffer of K*B*M*FP floats (FP
 *   from gcnb_cheb_stack_width) so that the backward pass can skip recomputing the recursion.
 */
GCNB_API int gcnb_cheb_fwd_f32(const float* x, const int32_t* perm, int M_in, const gcnb_csr* L, const float* W,
                      const float* bias, float* y, uint8_t* argmax, float* y_mean, float* xstack, int B, int Fin,
                      int Fout, int K, int p, int bias_mode, int relu, int algo, void* workspace,
                      size_t workspace_bytes, gcnb_stream_t stream);

/*
 * Backward of the fused layer (what tf.gradients builds for it, models_gcn.py:298-303).
 *   g  = dy * [y > 0] (if relu)            routed to row j*p + argmax (MaxPoolGrad), dz elsewhere 0
 *   db = sum_b,m dz (PER_FILTER) | sum_b dz (PER_VERTEX)
 *   dW[f*K+k, o] = sum_{b,m} X_k[b,m,f] dz[b,m,o]           (X_k recomputed from x)
 *   dx = sum_k T_k(L~^T) (dz W_k^T)                          (needs Lt = CSR of L~^T; skipped if dx NULL)
 * x / perm / M_in as in the forward (the gather is repeated when X_k is recomputed); dx, if
 * requested, is the gradient w.r.t. the permuted layer input [B][M][Fin].
 * dW / db are overwritten (not accumulated).  db may be NULL when bias_mode == NONE.
 * dy_is_mean != 0: dy is [B][M/p], the gradient of the mean over filters (every filter receives dy/Fout);
 *   the adjoint of y_mean above.
 * xstack (nullable): the basis saved by the forward (dW becomes one streamed tall-skinny GEMM; only the adjoint
 *   recursion for dx is left).
 */
GCNB_API int gcnb_cheb_bwd_f32(const float* x, const int32_t* perm, int M_in, const float* y, const uint8_t* argmax,
                      const float* dy, int dy_is_mean, const float* xstack, const gcnb_csr* L,
                      const gcnb_csr* Lt, const float* W, float* dx, float* dW, float* db, int B, int Fin,
                      int Fout, int K, int p, int bias_mode, int relu, int algo, void* workspace,
                      size_t workspace_bytes, gcnb_stream_t stream);

/*
 * Input gradient of the fused layer only (no dW, no db): dx = sum_k T_k(L~^T) (dz W_k^T) with dz rebuilt from dy / y /
 * argmax as in gcnb_cheb_bwd_f32 -- what a gradient saliency map of a trained network needs of each conv layer.
 * perm (nullable): the first layer's Graclus ordering, which must be a permutation of [0, M) (every raw vertex appears
 *   exactly once; entries >= M_in are fake vertices).  dx is then the gradient w.r.t. the UN-permuted input
 *   x_raw[B][M_in][Fin]: row m goes to raw row perm[m], fake vertices are dropped.  Without perm dx is [B][M][Fin].
 * x [B][M_in][Fin] (the layer input, as in the forward) may be NULL where the route never reads it: the general path
 *   recomputes the Chebyshev basis and refuses a NULL x.  Lt is required when K > 1; an operator image in Lt->image
 *   (gcnb_cheb_image_build with adjoint != 0) serves the tcgen05 route.  No bias argument: the bias does not enter dx.
 * gcnb_cheb_dx_describe names the route ("<route>: <its kernels>") and returns the workspace it takes (256-byte aligned
 * pointer).  Routes: the tcgen05 adjoint (k_cheb_fwd_umma on L~^T, any Fin in [4, 32], ALGO_AUTO), k_cheb_bwd_fused
 * without the weight gradient, or the general path (dW to workspace scratch); the last two un-permute in a second launch.
 */
GCNB_API int gcnb_cheb_dx_describe(int B, int M, int nnz, int Fin, int Fout, int K, int p, int algo, char* out, size_t n,
                                   size_t* workspace_bytes);
GCNB_API int gcnb_cheb_dx_f32(const float* x, const int32_t* perm, int M_in, const float* y, const uint8_t* argmax,
                              const float* dy, int dy_is_mean, const gcnb_csr* L, const gcnb_csr* Lt, const float* W,
                              float* dx, int B, int Fin, int Fout, int K, int p, int relu, int algo, void* workspace,
                              size_t workspace_bytes, gcnb_stream_t stream);

/*
 * Gradient of a ChebyNet layer w.r.t. the entries of its operator L~ (edge saliency maps), per window.  With dz rebuilt
 * from dy / y / argmax as in gcnb_cheb_bwd_f32, G_k = dz W_k^T and the Clenshaw states of the adjoint
 *   b_{K-1} = G_{K-1},  b_k = G_k + 2 L~^T b_{k+1} - b_{k+2}  (k = K-2 .. 1),
 * the gradient of <dy, layer(x)> is
 *   dL~[b][i][j] = sum_f b_1[i][b][f] X_0[j][b][f] + sum_{k=2}^{K-1} 2 sum_f b_k[i][b][f] X_{k-1}[j][b][f]
 * (X_k the Chebyshev basis of the permuted input), on L~'s pattern and on the diagonal:
 *   dval  [B][nnz]  entry e of L~'s CSR order (may be NULL when nnz = 0)
 *   ddiag [B][M]    entry (i, i), whether or not L~ stores it
 * L~ = L - I (lmax = 2), so these are also the gradients w.r.t. the entries of the Laplacian L.  K = 1 gives zeros.
 * accumulate != 0 adds onto dval / ddiag instead of overwriting them (layers that share an operator).  dx (nullable) is
 * the layer's input gradient, as gcnb_cheb_dx_f32 computes it on the general path (bit for bit), un-permuted through
 * perm to [B][M_in][Fin] when perm is given.  No dW, no db.  Lt is required when K > 1.  No allocation and no
 * synchronisation: the call can be captured in a CUDA graph.  Runs on the general path (HBM-resident stacks) and
 * k_sddmm_tma; the workspace is gcnb_cheb_dL_describe's (256-byte aligned pointer).
 */
GCNB_API int gcnb_cheb_dL_describe(int B, int M, int nnz, int Fin, int Fout, int K, int p, char* out, size_t n,
                                   size_t* workspace_bytes);
GCNB_API int gcnb_cheb_dL_f32(const float* x, const int32_t* perm, int M_in, const float* y, const uint8_t* argmax,
                              const float* dy, int dy_is_mean, const gcnb_csr* L, const gcnb_csr* Lt, const float* W,
                              float* dval, float* ddiag, int accumulate, float* dx, int B, int Fin, int Fout, int K,
                              int p, int relu, void* workspace, size_t workspace_bytes, gcnb_stream_t stream);

/*
 * Gradient w.r.t. the edge weights of the adjacency A the Laplacians were built from (edge saliency maps in ROI
 * coordinates), per window, from the per-level operator gradients G_l of gcnb_cheb_dL_f32.  Per level l, with A_l the
 * level's adjacency (zero diagonal), d_b = sum_a A_l[a][b], s = d^-1/2 and L~_l = -s_a A_ab s_b off the diagonal:
 *   r_b = sum_j G_bj L~_bj,  c_b = sum_i G_ib L~_ib  (stored entries)
 *   T_l[(a, b)] = -G_ab s_a s_b - (r_b + c_b) / (2 d_b) + T_next[parent[(a, b)]]
 * where T_next is the next entry of `levels` (a coarser level: the Graclus coarsening sums the entries of merged vertex
 * pairs, so its gradient flows back by a gather) and parent is -1 for a pair inside one cluster.  Then for every
 * undirected edge k of A:  out[b][k] = T_0[b][edges[2k]] + T_0[b][edges[2k + 1]]  (|.| with absolute != 0), the two
 * entries being (a, b) and (b, a) of level 0.  levels[0] is the finest level, levels[nlevels - 1] the coarsest; a
 * level no layer uses (G = 0) is skipped by composing the parent maps across it.  The diagonal of L is constant, so
 * gcnb_cheb_dL_f32's ddiag does not enter.  Every output is written by one thread in a fixed order: bit-reproducible.
 * No allocation and no synchronisation (capturable); the workspace holds T_l, [B][nnz_l] per level.
 */
#define GCNB_ADJ_MAX_LEVELS 16
typedef struct gcnb_adj_level {
  const float* dval;        /* [B][nnz] G_l in L~_l's CSR order (may be NULL when nnz = 0) */
  const int32_t* rowptr;    /* [M+1] L~_l's CSR (rows sorted by column, as gcnb_csr) */
  const float* val;         /* [nnz] L~_l's values */
  const int32_t* rowptr_t;  /* [M+1] CSR of L~_l^T */
  const int32_t* tpos;      /* [nnz] entry t of L~_l^T's CSR order is entry tpos[t] of L~_l's */
  const float* ss;          /* [nnz] s_a s_b of entry (a, b) */
  const float* hinv;        /* [M] 1 / (2 d_b), 0 for an isolated vertex */
  const int32_t* parent;    /* [nnz] entry of levels[l + 1], or -1; NULL for the last level */
  int32_t M;
  int32_t nnz;
} gcnb_adj_level;
GCNB_API size_t gcnb_adjacency_grad_workspace_bytes(const gcnb_adj_level* levels, int nlevels, int B);
GCNB_API int gcnb_adjacency_grad_f32(const gcnb_adj_level* levels, int nlevels, const int32_t* edges, int E, float* out,
                                     int B, int absolute, void* workspace, size_t workspace_bytes,
                                     gcnb_stream_t stream);

/*
 * Spectral layer (cgcnn.fourier + filter_in_fourier, models_gcn.py:512-539) with the same fused
 * bias/ReLU/pool epilogue.  Ut[M][M] is the transposed eigenvector matrix (row i = i-th
 * eigenvector), exactly the constant the reference builds at :536.  W[M][Fout][Fin].
 *   xh = Ut x ; yh[b,m,o] = sum_f W[m,o,f] xh[b,m,f] ; z = Ut^T yh
 */
GCNB_API size_t gcnb_spectral_workspace_bytes(int B, int M, int Fin, int Fout, int p, int backward);
GCNB_API int gcnb_spectral_fwd_f32(const float* x, const float* Ut, const float* W, const float* bias, float* y,
                          uint8_t* argmax, int B, int M, int Fin, int Fout, int p, int bias_mode, int relu,
                          void* workspace, size_t workspace_bytes, gcnb_stream_t stream);
GCNB_API int gcnb_spectral_bwd_f32(const float* x, const float* y, const uint8_t* argmax, const float* dy, const float* Ut,
                          const float* W, float* dx, float* dW, float* db, int B, int M, int Fin, int Fout, int p,
                          int bias_mode, int relu, void* workspace, size_t workspace_bytes, gcnb_stream_t stream);

/* Stand-alone pieces, for callers that invoke the reference methods one by one. */
/* b1relu / b2relu (models_gcn.py:619-629): y = max(x + bias, 0). */
GCNB_API int gcnb_brelu_fwd_f32(const float* x, const float* bias, float* y, int B, int M, int F, int bias_mode,
                       gcnb_stream_t stream);
/* dx = dy * [y > 0]; db as above.  workspace: M*F floats (PER_FILTER only), may be NULL otherwise. */
GCNB_API int gcnb_brelu_bwd_f32(const float* dy, const float* y, float* dx, float* db, int B, int M, int F, int bias_mode,
                       void* workspace, size_t workspace_bytes, gcnb_stream_t stream);
/* mpool1 (models_gcn.py:631-639): tf.nn.max_pool SAME over the vertex axis, any M (ragged tail padded). */
GCNB_API int gcnb_mpool_fwd_f32(const float* x, float* y, uint8_t* argmax, int B, int M, int F, int p, gcnb_stream_t stream);
GCNB_API int gcnb_mpool_bwd_f32(const float* dy, const uint8_t* argmax, float* dx, int B, int M, int F, int p,
                       gcnb_stream_t stream);
/* coarsening.perm_data_3d (coarsening.py:244-265) on the device, fp32 in / fp32 out. */
GCNB_API int gcnb_perm_gather_f32(const float* x, const int32_t* perm, float* y, int B, int M_in, int M_out, int F,
                         gcnb_stream_t stream);

/* Head pieces ("next" rows of the scope table): reduce_mean over the filter axis (models_gcn.py:673). */
GCNB_API int gcnb_mean_f_fwd_f32(const float* x, float* y, int rows, int F, gcnb_stream_t stream);
GCNB_API int gcnb_mean_f_bwd_f32(const float* dy, float* dx, int rows, int F, gcnb_stream_t stream);

/*
 * Sparse softmax cross-entropy, forward and backward in one pass (models_gcn.py:253-259):
 *   loss = mean_b (logsumexp(logits[b]) - logits[b][labels[b]]);  dlogits = (softmax - onehot) / B  (nullable).
 * loss_rows[B] is scratch for the per-row losses (fixed-order mean).
 * adam_state (nullable): if given, the kernel also advances the optimiser clock {b1^t, b2^t, lr_t, t} of
 *   gcnb_adam_tf_f32 (one launch less per training step); pass the same lr/beta1/beta2 as to the update.
 */
GCNB_API int gcnb_softmax_xent_f32(const float* logits, const int64_t* labels, float* loss, float* dlogits,
                          float* loss_rows, int B, int C, float* adam_state, float lr, float beta1, float beta2,
                          gcnb_stream_t stream);

/*
 * The classifier head of one training step in ONE launch (a persistent cooperative kernel, grid barriers between the
 * six dependent stages): cgcnn.fc x2 with ReLU + dropout (models_gcn.py:650-656, :674-677), the logits layer (:680-681),
 * the mean sparse-softmax cross-entropy (:253-259) and the whole backward pass tf.gradients builds for them (:298-303).
 *   h1 = dropout(relu(a0 W1 + b1)), h2 = dropout(relu(h1 W2 + b2)), logits = h2 W3 + b3, loss = mean CE(logits, labels)
 *   gW*, gb* = gradients of the loss (overwritten); d0 [B][n0] = gradient w.r.t. a0 (the mean over the filters of the
 *   last conv layer, i.e. the dy of gcnb_cheb_bwd_f32 with dy_is_mean = 1).
 * a0 [B][n0], W1 [n0][n1], W2 [n1][n2], W3 [n2][C], logits [B][C], loss [1]; n0 <= 32, C <= 32, n2 <= 2048.
 * Dropout: keep-probability `keep` (1 = none), counter-based masks keyed by (seed1 | seed2, adam_state[3]) -- the masks
 * gcnb_relu_dropout_fwd_f32 draws -- so CUDA-graph replays draw fresh masks.  tick != 0 advances the optimiser clock
 * {b1^t, b2^t, lr_t, t} in adam_state (as gcnb_softmax_xent_f32 does) after the masks of this step have been drawn.
 * A label outside [0, C) contributes neither loss nor gradient.  64x64 tiles on the tensor cores with both operands
 * split (3xTF32: fp32-level products), fp32 epilogues, fixed-order reductions.
 */
GCNB_API size_t gcnb_head_step_workspace_bytes(int B, int n0, int n1, int n2, int C); /* 0: sizes not supported */
GCNB_API int gcnb_head_step_f32(const float* a0, const int64_t* labels, const float* W1, const float* b1, const float* W2,
                                const float* b2, const float* W3, const float* b3, float* logits, float* loss,
                                float* gW1, float* gb1, float* gW2, float* gb2, float* gW3, float* gb3, float* d0, int B,
                                int n0, int n1, int n2, int C, float keep, unsigned seed1, unsigned seed2,
                                float* adam_state, float lr, float beta1, float beta2, int tick, void* workspace,
                                size_t workspace_bytes, gcnb_stream_t stream);

/* C[M x N] = op(A) op(B) (+ bias[N]); row-major, fp32 in/out, tensor cores with a 3-pass TF32 split (fp32-level
 * accuracy): tf.matmul of the spectral transforms (models_gcn.py:516-527) and of cgcnn.fc (:654) when the head runs
 * launch by launch. */
GCNB_API int gcnb_gemm_f32(const float* A, const float* B, float* C, const float* bias, int M, int N, int K, int lda,
                  int ldb, int ldc, int transA, int transB, gcnb_stream_t stream);

/* The same GEMM with the FC layer's element-wise step fused into the store (one launch less per layer and pass):
 *   GCNB_EPI_RELU_DROPOUT: C = dropout(relu(op(A) op(B) + bias)) -- cgcnn.fc, models_gcn.py:650-656 + tf.nn.dropout :677;
 *     the mask is the one gcnb_relu_dropout_fwd_f32 draws for the same (keep, seed, *step) on a [M x N] matrix;
 *   GCNB_EPI_MASK: C = aux[m][n] > 0 ? (op(A) op(B)) / keep : 0 -- its adjoint applied to dx = d W^T, aux = the
 *     forward activation (what gcnb_relu_dropout_bwd_f32 does in a separate pass). */
enum { GCNB_EPI_NONE = 0, GCNB_EPI_RELU_DROPOUT = 1, GCNB_EPI_MASK = 2 };
GCNB_API int gcnb_gemm_epilogue_f32(const float* A, const float* B, float* C, const float* bias, int M, int N, int K,
                                    int lda, int ldb, int ldc, int transA, int transB, int epilogue, const float* aux,
                                    int ld_aux, float keep, unsigned seed, const float* step, gcnb_stream_t stream);

/* y = dropout(relu(x)) in place on x[rows][ld] (first `cols` columns): keep-probability `keep`, kept values scaled by
 * 1/keep (tf.nn.relu + tf.nn.dropout, models_gcn.py:655,677).  Counter-based generator keyed by (seed, *step, index);
 * step is a device counter so that CUDA-graph replays draw fresh masks.  keep >= 1 is a plain ReLU. */
GCNB_API int gcnb_relu_dropout_fwd_f32(float* x, long long rows, int cols, int ld, float keep, unsigned seed,
                              const float* step, gcnb_stream_t stream);
/* d = (act > 0) ? d / keep : 0 in place (act = output of the forward; act > 0 <=> ReLU active and kept). */
GCNB_API int gcnb_relu_dropout_bwd_f32(float* d, const float* act, long long rows, int cols, int ld_d, int ld_act,
                              float keep, gcnb_stream_t stream);
/* out_i[c] = sum_r m_i[r][c] for up to 4 row-major matrices in one launch: the bias gradients tf.gradients builds for
 * the `+ b` of cgcnn.fc (models_gcn.py:653-654, :298-303). */
GCNB_API int gcnb_colsum_multi_f32(const float* const* mats, float* const* outs, const int* rows, const int* cols,
                          int count, gcnb_stream_t stream);
/* out[g][c] = sum over the rows r with group[r] == g of X[r][c] (|X[r][c]| with absolute != 0), X row-major
 * [rows][cols], out [n_groups][cols]: per-group sums of per-window saliency maps (one row per window).  Rows whose group
 * is < 0 or >= n_groups contribute nothing; rows of out whose group occurs in no row are NOT written.  1 <= rows <= 8192,
 * cols >= 1, 1 <= n_groups <= rows.  Fixed summation order that depends only on (rows, group): bit-reproducible, no
 * float atomics, no allocation, no synchronisation, CUDA-graph capturable.  The work grows with rows x cols and not with
 * n_groups, so a caller may pass a capacity. */
GCNB_API int gcnb_group_colsum_f32(const float* X, int rows, int cols, const int32_t* group, int n_groups,
                                   int absolute, float* out, gcnb_stream_t stream);

/*
 * tf.train.AdamOptimizer step (models_gcn.py:294, TF-1.x "epsilon hat" form) over one flat buffer of n parameters:
 *   g' = g * gscale + reg * p (only where decay[i] != 0; the L2 term of models_gcn.py:260-262)
 *   m = b1 m + (1-b1) g';  v = b2 v + (1-b2) g'^2;  p -= lr sqrt(1-b2^t)/(1-b1^t) * m / (sqrt(v) + eps)
 * state[4] (device) holds {b1^t, b2^t, lr_t, t}; initialise to {1, 1, 0, 0}.  The step counter lives on the device so
 * that a captured CUDA graph can replay the step.  tick != 0: advance the clock here (an extra 1-thread launch);
 * tick == 0: the clock was already advanced this step by gcnb_softmax_xent_f32.
 */
GCNB_API int gcnb_adam_tf_f32(float* p, const float* g, float* m, float* v, const uint8_t* decay, float* state,
                     long long n, float lr, float beta1, float beta2, float eps, float reg, float gscale, int tick,
                     gcnb_stream_t stream);

/*
 * tf.contrib.opt.NadamOptimizer step (TF's ApplyAdam with use_nesterov = true) over one flat buffer of n parameters --
 * the optimiser of the fine-tuning model (models_gcn.py:685-933).  Same clock state[4], decay mask and tick rule as
 * gcnb_adam_tf_f32, no gradient scale:
 *   g' = g + reg * p (only where decay[i] != 0);  m = b1 m + (1-b1) g';  v = b2 v + (1-b2) g'^2
 *   p -= lr sqrt(1-b2^t)/(1-b1^t) * (b1 m + (1-b1) g') / (sqrt(v) + eps)
 * (not Dozat's momentum schedule of Keras' Nadam / torch.optim.NAdam).
 */
GCNB_API int gcnb_nadam_tf_f32(float* p, const float* g, float* m, float* v, const uint8_t* decay, float* state,
                               long long n, float lr, float beta1, float beta2, float eps, float reg, int tick,
                               gcnb_stream_t stream);

/*
 * Data-parallel training: the gradient all-reduce FUSED into the optimiser update (one ordinary launch; replaces
 * ncclAllReduce + gcnb_adam_tf_f32 on the step's critical path).  Every rank's flat gradient buffer is peer-mapped;
 * the kernel raises one flag per peer over NVLink, waits for all peers' flags, reads all ranks' gradients straight from
 * peer memory, sums them in rank order (bit-identical on every rank, so replicas never drift) and applies the Adam
 * step above with gscale = 1 / world.  `state` must already hold this step's clock.
 * peer_grad[q] / peer_flags[q] (HOST arrays of `world` DEVICE pointers, mapped into this process, e.g. torch symmetric
 * memory or CUDA IPC): rank q's flat gradient of THIS step and its flag array of gcnb_adam_allreduce_flag_bytes() bytes
 * (zero-filled once).  The caller must alternate between two gradient buffers on successive steps (a peer may still
 * be reading the previous one); the flag arrays stay the same.
 */
GCNB_API size_t gcnb_adam_allreduce_flag_bytes(void);
GCNB_API int gcnb_adam_tf_allreduce_f32(float* p, float* m, float* v, const uint8_t* decay, const float* state,
                                        long long n, float beta1, float beta2, float eps, float reg,
                                        const void* const* peer_grad, void* const* peer_flags, int rank, int world,
                                        gcnb_stream_t stream);

/*
 * The same fused exchange for the fine-tuning optimiser: gcnb_nadam_tf_f32's update (TF's NadamOptimizer) on the
 * rank-order sum of every rank's gradient scaled by gscale = 1 / world.  Arguments, flag arrays, the alternating
 * gradient buffers, the L2 fold and the decay mask are those of gcnb_adam_tf_allreduce_f32; both calls may share one
 * flag array only if they never run at the same time.
 */
GCNB_API int gcnb_nadam_tf_allreduce_f32(float* p, float* m, float* v, const uint8_t* decay, const float* state,
                                         long long n, float beta1, float beta2, float eps, float reg,
                                         const void* const* peer_grad, void* const* peer_flags, int rank, int world,
                                         gcnb_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* GCNB200_H */
