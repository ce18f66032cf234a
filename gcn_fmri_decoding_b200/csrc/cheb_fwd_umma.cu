// Fused ChebyNet forward on the Blackwell tensor cores (tcgen05 + TMEM) for graphs that fit in shared memory:
//   (perm gather) -> T_k(L~) recursion -> contraction with the taps -> bias -> ReLU -> max-pool (+ mean over filters)
// Replaces cgcnn.chebyshev5 / chebyshev2 + b1relu / b2relu + mpool1 (models_gcn.py:587-617, 558-585, 619-639).
//
// One persistent CTA per SM, 25 warps with three roles:
//   * 20 "sparse" warps (24 measured slower: the recursion is bound by shared-memory wavefronts, not by warps) run the recursion X_k = 2 L~ X_{k-1} - X_{k-2} out of shared memory.  The state of a tile
//     of windows lives in two ping-pong slabs of 128-byte rows (row = vertex, 32 floats = G windows x FP features,
//     SWIZZLE_128B): a neighbour row is one conflict-free LDS.128 per lane, 8 lanes per row, 4 rows per warp step.
//     Rows are sorted by length once per CTA and dealt to the warps in groups of four (snake order) so that the
//     lanes of a warp stay in lock step and the warps finish together.
//   * 1 MMA warp: after every order, one elected thread issues z += X_k W_k as tcgen05.mma (M = 128 vertices,
//     N = 32 filters) straight from the slab the sparse warps just wrote -- no operand copy, no fragment loads, no
//     accumulator registers.  fp32-level accuracy from a 3-term split on the tensor cores:
//       trunc_tf32(X) * tf32(W)  +  trunc_tf32(X) * tf32(W - tf32(W))  +  bf16(X - trunc_tf32(X)) * bf16(W)
//     (the hardware truncation of kind::tf32 IS the "hi" part of X; only the bf16 remainder is stored separately).
//     Accumulators stay in TMEM across all K orders, double-buffered across tiles.
//   * 4 epilogue warps drain the finished tile of the PREVIOUS iteration from TMEM while the sparse warps already
//     work on the next one.  State rows are kept SIBLING-MAJOR: vertex v = p*j + i of window-slab s lives in row
//     i*BQ + s*Q + j, so the p members of a pooling window sit in the SAME TMEM lane of p different accumulator
//     blocks and mpool1 is a thread-local running maximum (first-maximum rule of MaxPoolGrad) -- no shuffles, no
//     shared-memory transpose; thread = pooled vertex, 32 filters: bias, ReLU, y / arg-max / mean-over-filters.
// x is read from HBM once, y written once; the K-stack only goes to HBM when the caller asks for it (training).
#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <type_traits>
#include <vector>

#include "umma.cuh"

namespace gcnb {

using namespace um;

static constexpr int kSparseWarps = 20;
static constexpr int kEpiWarps = 4;   // warps 0..3: warp w may only touch TMEM lanes 32w..32w+31
static constexpr int kMmaWarp = 4;    // warp 4
static constexpr int kThreads = (kSparseWarps + kEpiWarps + 1) * 32;
static_assert(kSparseWarps % 4 == 0, "the tail epilogue deals the sparse warps to the four TMEM lane quarters");
static constexpr uint32_t kImgMagic = 0x494e4347u;  // "GCNI"
static constexpr uint32_t kImgPair = 144;            // bytes of one pair of steps in the entry stream of an operator image
static constexpr int kBarOrder = 1;   // named barrier: sparse warps + MMA warp, once per Chebyshev order
static constexpr int kBarLayer = 2;   // named barrier: all warps, between two layers of a stack (see UmmaFwdParams::nlayers)

#ifdef GCNB_TRACE
// debug builds only (-DGCNB_TRACE): clock64 stamps of CTA 0's roles, read back by gcnb_debug_read_trace
__device__ long long g_trace[4][512];
#define TRACE(region, cond)                                                        \
  do {                                                                             \
    if (blockIdx.x == 0 && lane == 0 && (cond) && tr_n < 512) g_trace[region][tr_n++] = clock64(); \
  } while (0)
// per sparse warp, one chosen order (n == 2) of CTA 0: g_trace[1][64 + sw * 16 + slot]
#define TRACEW(slot)                                                                              \
  do {                                                                                            \
    if (blockIdx.x == 0 && lane == 0 && n == 2) g_trace[1][64 + sw * 16 + (slot)] = clock64();     \
  } while (0)
#else
#define TRACE(region, cond) do { } while (0)
#define TRACEW(slot) do { } while (0)
#endif
#ifdef GCNB_TRACE
// order 0 of CTA 0's first two tiles, per sparse warp: g_trace[3][64 + (tile index) * 160 + sw * 8 + slot]
#define TRACE0(slot)                                                                                     \
  do {                                                                                                   \
    if (blockIdx.x == 0 && lane == 0 && n <= (uint32_t)K) g_trace[3][64 + (n ? 160 : 0) + sw * 8 + (slot)] = clock64(); \
  } while (0)
#else
#define TRACE0(slot) do { } while (0)
#endif
#ifdef GCNB_TRACE
// first layer boundary of a stack, per warp w (sparse warps 0..19, epilogue warps 20..23): g_trace[0][256 + w * 8 + slot]
#define TRACEB(w, slot) do { if (blockIdx.x == 0 && lane == 0 && it == 0) g_trace[0][256 + (w) * 8 + (slot)] = clock64(); } while (0)
#else
#define TRACEB(w, slot) do { } while (0)
#endif
#ifdef GCNB_TRACE
#define TRACE_NOSPILL ((P.debug & 4) != 0)  // image kernels: skip the basis stores
#define TRACE_NOLOAD ((P.debug & 8) != 0)   // image kernels: order 0 is all zeros (no global loads)
#else
#define TRACE_NOSPILL false
#define TRACE_NOLOAD false
#endif

struct UmmaFwdParams {
  const float* x;
  const int32_t* perm;
  int M_in;
  const int32_t* rowptr;
  const int32_t* col;
  const float* val;
  int nnz;
  const float* W;
  const float* bias;
  float* y;
  uint8_t* argmax;
  float* y_mean;
  float* xstack;
  int B, M, Fin, Fout, K, p, log2p, bias_mode, relu;
  int NS;        // window-slabs per tile (each holds G windows side by side in its rows)
  int S;         // windows per tile = NS * G
  int Q;         // rows of one window-slab inside a sibling block = M/p rounded up to 8
  int BQ;        // rows of one sibling block = NS * Q
  int T;         // 128-row MMA tiles per sibling block
  int NG;        // groups of 4 rows
  int ntiles;
  int nlo;       // lo buffers per slab (2, or 1 when shared memory is short)
  int nacc;      // TMEM accumulator buffers (2, or 1)
  int acc_cols;  // TMEM columns of one accumulator buffer = G * p * T * 32
  int tmem_cols; // allocated columns (power of two)
  int slab_rows; // rows of one state buffer incl. the zero row (multiple of 8)
  int debug;     // GCNB_TRACE builds only: bit0 skip the gathers, bit1 skip the tcgen05.mma issue
  // Adjoint mode (the layer's input gradient): dx = sum_k T_k(L~^T) dZ W_k^T is the SAME computation as the forward
  // with the transposed operator, the transposed taps and dZ as the input.  dZ (MaxPoolGrad o ReluGrad of the layer's
  // output gradient) is rebuilt on the fly from the pooled tensors while order 0 is loaded; x / perm are unused.
  int adj;              // 1: adjoint mode; Fin = the layer's Fout (contraction width), Fout = the layer's Fin
  const float* adj_dy;  // [B][Mo][Fin], or [B][Mo] when adj_mean (gradient of the mean over filters)
  const float* adj_y;   // [B][Mo][Fin] pooled layer output (ReLU mask), used when adj_relu
  const uint8_t* adj_arg;  // [B][Mo][Fin] arg-max offsets, used when the layer pools (adj_log2p > 0)
  int adj_log2p, adj_relu, adj_mean, adj_Mo;
  // Pre-built operator image (IMG kernels, see "operator image" below): copied to shared memory as is.
  const unsigned char* image;
  int img_bytes;     // multiple of 16
  int stage;         // image kernels, forward: the raw windows of a tile are staged with one TMA bulk copy
  // Layer stack (image kernels, inference): nlayers > 1 runs a stack of identical layers (same graph, p = 1,
  // Fin = Fout = 32, same K / bias mode / ReLU) on a tile back to back -- the output of a layer is written from TMEM
  // straight into the state buffer as order 0 of the next one and never leaves the SM.  Layer l reads Wl[l] / biasl[l];
  // W / bias above are layer 0's / the last layer's.
  int nlayers;
  const float* Wl[8];
  const float* biasl[8];
  // Pre-split tap images (gcnb_cheb_tap_image_build): the exact bytes of the three tap arrays of a layer (tf32 hi, tf32 lo,
  // bf16) in their shared-memory layout.  tapimg[l] != NULL: copied by TMA instead of being split from W in the kernel.
  const unsigned char* tapimg[8];
  int tap_bytes;  // 2.5 x K * FP * 32 * 4
  unsigned img_sig;  // geometry signature the image must carry
  int n_groups;      // groups of 4 row blocks
  int off_img, off_grp, off_blk;  // shared-memory offsets of the image copy, its group table and its block table
  // byte offsets into dynamic shared memory
  int off_lo, off_wh, off_wl, off_wb, off_ent, off_grow, off_grho, off_gslot, off_glen, off_src, off_rlen, off_sorted, off_bias,
      off_bar, off_rp;
};

// ---------------------------------------------------------------------------------------------------------------
// STACK: the layer-stack variant (UmmaFwdParams::nlayers > 1); the single-layer instances carry none of its code.
// RAW: adjoint mode writing the input gradient of a first layer -- output rows of any width (Fout need not be a multiple
// of 4: element stores), row m sent to raw row perm[m] when perm is given (fake vertices dropped), MMA N = 16 for
// outputs of at most 16 columns.  The other instances carry none of its code.
template <int FP, int MAXI, bool IMG, bool STACK, bool RAW>
__global__ void __launch_bounds__(kThreads, 1) k_cheb_fwd_umma(const UmmaFwdParams P) {
  extern __shared__ __align__(1024) unsigned char smem[];
  constexpr int G = 32 / FP;    // windows per 128-byte row
  constexpr int CPW = FP / 4;   // 16-byte chunks per window
  const uint32_t sb = smem_u32(smem);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int M = P.M, K = P.K, NS = P.NS, Q = P.Q, BQ = P.BQ;
  const int pm1 = P.p - 1, log2p = P.log2p;
  const uint32_t buf_bytes = (uint32_t)P.slab_rows * 128u, lo_bytes = (uint32_t)P.slab_rows * 64u;
  // state buffer u at sb + u*buf_bytes ; remainder (lo) buffer u at sb + off_lo + u*lo_bytes
  int* grow = reinterpret_cast<int*>(smem + P.off_grow);       // [NG*4] vertex of (group, slot), -1 = none
  int* grho = reinterpret_cast<int*>(smem + P.off_grho);       // [NG*4] its state row inside window-slab 0
  int2* gslot = reinterpret_cast<int2*>(smem + P.off_gslot);   // [NG*4] (first entry pair, row length)
  int* glen = reinterpret_cast<int*>(smem + P.off_glen);       // [NG] entry pairs of the longest row of the group
  int* src_row = reinterpret_cast<int*>(smem + P.off_src);     // [M] source row of the raw window, -1 = zero
  int* rlen = reinterpret_cast<int*>(smem + P.off_rlen);       // [NG*4]
  int* sorted = reinterpret_cast<int*>(smem + P.off_sorted);   // [NG*4]
  int* rp = reinterpret_cast<int*>(smem + P.off_rp);           // [M+1] row pointers
  float* bias_s = reinterpret_cast<float*>(smem + P.off_bias); // [nlayers][32]; the epilogue of the last layer reads the last row
  const uint32_t bar0 = sb + P.off_bar;
  auto bar_mma = [bar0](uint32_t i) { return bar0 + i * 8u; };          // tcgen05.mma of order n done (n & 1)
  auto bar_full = [bar0](uint32_t i) { return bar0 + 16u + i * 8u; };   // accumulator buffer i complete
  auto bar_empty = [bar0](uint32_t i) { return bar0 + 32u + i * 8u; };  // accumulator buffer i drained
  const uint32_t bar_stage = bar0 + 56u;                                 // raw windows of a tile staged (TMA)
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem + P.off_bar + 48);
  // state row of vertex v inside window-slab 0 (sibling-major)
  auto rho = [=](int v) { return (v & pm1) * BQ + (v >> log2p); };

  // ---- prologue (all warps) ---------------------------------------------------------------------------------
#ifdef GCNB_TRACE
  int tr_p = 0;
#define TRACEP() do { if (blockIdx.x == 0 && tid == 160) g_trace[1][tr_p++] = clock64(); } while (0)
#else
#define TRACEP() do { } while (0)
#endif
  TRACEP();
  if ((sb & 1023u) != 0) __trap();  // the swizzled operand layouts need a 1 KB aligned base
  if (tid == 0) {
    mbar_init(bar_mma(0), 1); mbar_init(bar_mma(1), 1);
    mbar_init(bar_full(0), 1); mbar_init(bar_full(1), 1);
    mbar_init(bar_empty(0), kEpiWarps); mbar_init(bar_empty(1), kEpiWarps);
    mbar_init(bar_stage, 1);
    mbar_init_fence();
  }
  if constexpr (IMG) {
    // the operator image was built once on the host (gcnb_cheb_image_build): ONE TMA bulk copy brings it in as it is
    // while the rest of the prologue runs (first phase of the staging barrier)
    if (tid == 0) {
      const bool tap0 = STACK && P.tapimg[0] != nullptr;
      mbar_expect_tx(bar_stage, (uint32_t)P.img_bytes + (tap0 ? (uint32_t)P.tap_bytes : 0u));
      bulk_g2s(sb + P.off_img, P.image, (uint32_t)P.img_bytes, bar_stage);
      if (tap0) bulk_g2s(sb + P.off_wh, P.tapimg[0], (uint32_t)P.tap_bytes, bar_stage);
    }
  }
  if (warp == kMmaWarp) tmem_alloc(sb + P.off_bar + 48, (uint32_t)P.tmem_cols);
  // taps: tf32 hi / lo and bf16 images, contraction index kk = k*FP + f  (W row = f*K + k, models_gcn.py:611-615).
  // The global loads of the first batch (and of the permutation / bias) are in flight while the state buffers are zeroed.
  // element idx -> (filter o, contraction index kk): the 32 lanes of a warp cover (o & 7) x (kk & 3), i.e. all 32 banks of
  // the tap images (the natural order, lane = filter, stores with 4-way bank conflicts)
  auto tap_o = [](int idx) { return (idx & 7) | (((idx >> 5) & 3) << 3); };
  auto tap_kk = [](int idx) { return ((idx >> 3) & 3) | ((idx >> 7) << 2); };
  // (nt threads with index t share the conversion: the whole CTA in the prologue, the sparse warps between layers)
  auto tap_load = [&](const float* Wsrc, int i0, int t, int nt, float (&wv)[4]) {
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int idx = i0 + u * nt + t;
      const int o = tap_o(idx), kk = tap_kk(idx), k = kk / FP, f = kk - k * FP;
      wv[u] = (idx < K * FP * 32 && f < P.Fin && o < P.Fout)
                  ? __ldg(Wsrc + (P.adj ? ((long long)o * K + k) * P.Fin + f : ((long long)f * K + k) * P.Fout + o))
                  : 0.f;
    }
  };
  auto tap_store = [&](int i0, int t, int nt, const float (&wv)[4]) {
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int idx = i0 + u * nt + t;
      if (idx < K * FP * 32) {
        const int o = tap_o(idx), kk = tap_kk(idx);
        const float w = wv[u], hi = tf32_rna(w), lo = tf32_rna(w - hi);
        *reinterpret_cast<float*>(smem + P.off_wh + tap_off_tf32(kk, o)) = hi;
        *reinterpret_cast<float*>(smem + P.off_wl + tap_off_tf32(kk, o)) = lo;
        *reinterpret_cast<__nv_bfloat16*>(smem + P.off_wb + tap_off_bf16(kk, o)) = __float2bfloat16_rn(w);
      }
    }
  };
  auto taps_of = [&](const float* Wsrc, int t, int nt) {  // all tap images of one layer
    for (int i0 = 0; i0 < K * FP * 32; i0 += nt * 4) {
      float wv[4];
      tap_load(Wsrc, i0, t, nt, wv);
      tap_store(i0, t, nt, wv);
    }
  };
  const bool split_taps0 = !(STACK && IMG && P.tapimg[0] != nullptr);  // else: layer 0's taps arrive by TMA (above)
  float wv0[4] = {0.f, 0.f, 0.f, 0.f};
  if (split_taps0) tap_load(P.W, 0, tid, kThreads, wv0);
  int perm0 = tid;
  if (P.perm && tid < M) perm0 = __ldg(P.perm + tid);
  const int nlayers = STACK ? P.nlayers : 1;
  float bias0 = 0.f;
  if (tid < 32 * nlayers && P.bias_mode == GCNB_BIAS_PER_FILTER && (tid & 31) < P.Fout)
    bias0 = __ldg((nlayers > 1 ? P.biasl[tid >> 5] : P.bias) + (tid & 31));
  // zero the state buffers: the zero row behind every buffer and the padding rows of the blocks stay zero (the
  // remainder buffers need no initialisation -- garbage there only reaches accumulator rows nobody reads -- and
  // host the prologue's scratch tables rlen / sorted / rp until the first order overwrites them)
  for (uint32_t a = tid * 16u; a < (uint32_t)P.off_lo; a += kThreads * 16u) sts128(sb + a, make_float4(0.f, 0.f, 0.f, 0.f));
  if (split_taps0) {
    tap_store(0, tid, kThreads, wv0);
    for (int i0 = kThreads * 4; i0 < K * FP * 32; i0 += kThreads * 4) {
      float wv[4];
      tap_load(P.W, i0, tid, kThreads, wv);
      tap_store(i0, tid, kThreads, wv);
    }
  }
  for (int r = tid; r < M; r += kThreads) {
    int s = r == tid ? perm0 : r;
    if (P.perm) { if (r != tid) s = __ldg(P.perm + r); if (s < 0 || s >= P.M_in) s = -1; }
    src_row[r] = s;
  }
  if (tid < 32 * nlayers) bias_s[tid] = bias0;
  if constexpr (IMG) {
    __syncthreads();          // (thread 0 initialised the barrier: nobody may poll it before that is certain)
    mbar_wait(bar_stage, 0);  // the image has landed
    const uint32_t* hdr = reinterpret_cast<const uint32_t*>(smem + P.off_img);
    if (hdr[0] != kImgMagic || hdr[1] != P.img_sig || hdr[2] != (uint32_t)P.img_bytes) __trap();  // image of another geometry
  } else {
    // operator image: rows sorted by decreasing length; entries re-encoded as (gather code, value) in CSR order,
    // every row starting on an even entry so that one LDS.128 fetches two entries
    const int M4 = P.NG * 4;
    int* bins = sorted;  // [M + 3]: bin b counts rows of length (M - b); the padding rows (length -1) come last;
                         // bins[M + 2] = longest row.  (`sorted` itself is no longer materialised.)
    for (int r = tid; r <= M; r += kThreads) rp[r] = __ldg(P.rowptr + r);
    for (int i = tid; i < M + 3; i += kThreads) bins[i] = 0;
    {
      const int npairs = (P.nnz + M + 2) >> 1;  // zero entries everywhere (padding entry of odd rows: zero row, 0.0)
      const uint32_t zc = gather_code(P.p * BQ);
      int4* e4 = reinterpret_cast<int4*>(smem + P.off_ent);
      for (int i = tid; i < npairs; i += kThreads) e4[i] = make_int4((int)zc, 0, (int)zc, 0);
    }
    TRACEP();
    __syncthreads();
    TRACEP();
    for (int r = tid; r < M4; r += kThreads) {
      const int l = r < M ? rp[r + 1] - rp[r] : -1;
      rlen[r] = l;
      atomicAdd(&bins[M - l], 1);
      if (l > 0) atomicMax(&bins[M + 2], l);
    }
    {
      // one thread per entry, eight at a time: all loads issued first, then eight independent bisections of rp
      int2* ent = reinterpret_cast<int2*>(smem + P.off_ent);
      for (int e0 = 0; e0 < P.nnz; e0 += kThreads * 8) {
        int cc[8], lo[8];
        float vv[8];
  #pragma unroll
        for (int u = 0; u < 8; ++u) {
          const int e = e0 + u * kThreads + tid;
          cc[u] = e < P.nnz ? __ldg(P.col + e) : 0;
          vv[u] = e < P.nnz ? __ldg(P.val + e) : 0.f;
          lo[u] = 0;
        }
        // largest r with rp[r] <= e: fixed-trip bisection over [0, 2^s) so that the eight chains interleave
        for (int step = 1 << (31 - __clz(max(M, 1))); step > 0; step >>= 1) {
  #pragma unroll
          for (int u = 0; u < 8; ++u) {
            const int cand = lo[u] + step;
            if (cand <= M && rp[min(cand, M)] <= e0 + u * kThreads + tid) lo[u] = cand;
          }
        }
  #pragma unroll
        for (int u = 0; u < 8; ++u) {
          const int e = e0 + u * kThreads + tid;
          if (e < P.nnz) {
            const int r = min(lo[u], M - 1);
            ent[((rp[r] + r + 1) & ~1) + (e - rp[r])] = make_int2((int)gather_code(rho(cc[u])), __float_as_int(vv[u]));
          }
        }
      }
    }
    TRACEP();
    __syncthreads();
    TRACEP();
    if (warp == 0) {
      // exclusive prefix over the occupied bins [M - longest, M + 1] (rows sorted by decreasing length), one warp
      const int first = M - bins[M + 2];
      int carry = 0;
      for (int b0 = first; b0 < M + 2; b0 += 32) {
        const int i = b0 + lane;
        const int v = i < M + 2 ? bins[i] : 0;
        int x = v;
  #pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
          const int y = __shfl_up_sync(0xffffffffu, x, d);
          if (lane >= d) x += y;
        }
        if (i < M + 2) bins[i] = carry + x - v;
        carry += __shfl_sync(0xffffffffu, x, 31);
      }
    }
    __syncthreads();
    // every row takes its place in the sorted order (the order inside a bin is whatever the atomics give: it only
    // decides which rows share a warp step, never a sum) and fills the group tables there
    for (int r = tid; r < M4; r += kThreads) {
      const int l = rlen[r];
      const int i = atomicAdd(&bins[M - l], 1);
      if (r < M) {
        grow[i] = r;
        grho[i] = rho(r);
        gslot[i] = make_int2(((rp[r] + r + 1) & ~1) >> 1, l);
      } else {
        grow[i] = -1;
        grho[i] = 0;
        gslot[i] = make_int2(0, 0);
      }
    }
    __syncthreads();
    for (int g = tid; g < P.NG; g += kThreads) glen[g] = (gslot[g * 4].y + 1) >> 1;  // slot 0 holds the group's longest row
  }
  TRACEP();
  fence_async_smem();  // the zeroed state buffers are about to be written through the async proxy (staging copy)
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  TRACEP();

#ifdef GCNB_TRACE
  int tr_n = 0;
#endif
  const int NI = P.NG * NS;  // work items (row group, window-slab) of one order
  const int nsync = (kSparseWarps + 1) * 32;

  // ---- one epilogue task: halves [h0, h1) of the 32 filters of accumulator block (g, t) for TMEM lane quarter e -------
  // thread = (window-slab, pooled vertex); the p sibling vertices of its pooling window sit in the same TMEM lane of p
  // accumulator blocks: running maximum with the first-maximum rule, bias, ReLU, y / arg-max / mean stores
  const int Mo = M >> log2p;
  auto epi_task = [&](int tile, int buf, int e, int g, int t, int h0, int h1) {
    const int p = P.p;
    const bool pool_relu_fix = P.relu && p > 1;
          const int rb0 = t * 128 + e * 32;
          if (rb0 >= BQ) return;
          const int rb = rb0 + lane;             // row inside a sibling block = (window-slab, pooled vertex)
          const int s = rb / Q, j = rb - s * Q;
          const int b = tile * P.S + s * G + g;
          const bool valid = rb < BQ && j < Mo && b < P.B;
          const long long orow = (long long)b * Mo + j;
          const uint32_t tbase = tmem + ((uint32_t)(e * 32) << 16) + (uint32_t)(buf * P.acc_cols + (g * p * P.T + t) * 32);
          if constexpr (RAW) {
            // p = 1, no bias / ReLU: row j of the layer's vertex order is the gradient of raw row src_row[j] (perm[j], or
            // -1 for a fake vertex, whose gradient is dropped).  Every raw row has exactly one such j: plain stores, no
            // zero fill.  A row of Fout floats need not be 16-byte aligned: element stores.
            const int dst = valid ? src_row[j] : -1;
            float* dxp = dst >= 0 ? P.y + ((long long)b * P.M_in + dst) * P.Fout : nullptr;
            for (int h = h0; h < h1 && h * 16 < P.Fout; ++h) {
              float m[16];
              tmem_ld16(tbase + h * 16, m);
              if (dxp) {
#pragma unroll
                for (int o = 0; o < 16; ++o)
                  if (h * 16 + o < P.Fout) dxp[h * 16 + o] = m[o];
              }
            }
            return;
          }
          float msum = 0.f;
          for (int h = h0; h < h1; ++h) {
            float m[16];
            int idx[16];
            tmem_ld16(tbase + h * 16, m);
            if (P.bias_mode == GCNB_BIAS_PER_VERTEX && valid) {
              const float* bp = P.bias + (long long)(j << log2p) * P.Fout + h * 16;
#pragma unroll
              for (int c4 = 0; c4 < 4; ++c4) {
                if (h * 16 + c4 * 4 < P.Fout) {
                  const float4 bv = __ldg(reinterpret_cast<const float4*>(bp + c4 * 4));
                  m[c4 * 4] += bv.x; m[c4 * 4 + 1] += bv.y; m[c4 * 4 + 2] += bv.z; m[c4 * 4 + 3] += bv.w;
                }
              }
            }
#pragma unroll
            for (int o = 0; o < 16; ++o) idx[o] = 0;
            for (int i = 1; i < p; ++i) {
              float a[16];
              tmem_ld16(tbase + (uint32_t)(i * P.T * 32) + h * 16, a);
              if (P.bias_mode == GCNB_BIAS_PER_VERTEX && valid) {
                const float* bp = P.bias + (long long)((j << log2p) + i) * P.Fout + h * 16;
#pragma unroll
                for (int c4 = 0; c4 < 4; ++c4) {
                  if (h * 16 + c4 * 4 < P.Fout) {
                    const float4 bv = __ldg(reinterpret_cast<const float4*>(bp + c4 * 4));
                    a[c4 * 4] += bv.x; a[c4 * 4 + 1] += bv.y; a[c4 * 4 + 2] += bv.z; a[c4 * 4 + 3] += bv.w;
                  }
                }
              }
#pragma unroll
              for (int o = 0; o < 16; ++o) {
                const bool gt = a[o] > m[o];  // strict: the first maximum wins (MaxPoolGrad)
                m[o] = gt ? a[o] : m[o];
                idx[o] = gt ? i : idx[o];
              }
            }
            if (P.bias_mode == GCNB_BIAS_PER_FILTER) {
#pragma unroll
              for (int c4 = 0; c4 < 4; ++c4) {
                const float4 bv = *reinterpret_cast<const float4*>(bias_s + (nlayers - 1) * 32 + h * 16 + c4 * 4);
                m[c4 * 4] += bv.x; m[c4 * 4 + 1] += bv.y; m[c4 * 4 + 2] += bv.z; m[c4 * 4 + 3] += bv.w;
              }
            }
            if (P.relu) {
#pragma unroll
              for (int o = 0; o < 16; ++o) {
                // a window whose maximum is clipped is a tie of zeros after the ReLU: the first vertex is the arg-max
                if (pool_relu_fix && !(m[o] > 0.f)) idx[o] = 0;
                m[o] = fmaxf(m[o], 0.f);
              }
            }
            if (valid) {
              float* yp = P.y + orow * P.Fout + h * 16;
#pragma unroll
              for (int c4 = 0; c4 < 4; ++c4)
                if (h * 16 + c4 * 4 < P.Fout)
                  *reinterpret_cast<float4*>(yp + c4 * 4) = make_float4(m[c4 * 4], m[c4 * 4 + 1], m[c4 * 4 + 2], m[c4 * 4 + 3]);
              if (P.argmax && p > 1) {
                uint8_t* ap = P.argmax + orow * P.Fout + h * 16;
#pragma unroll
                for (int c4 = 0; c4 < 4; ++c4)
                  if (h * 16 + c4 * 4 < P.Fout)
                    *reinterpret_cast<uint32_t*>(ap + c4 * 4) = (uint32_t)idx[c4 * 4] | ((uint32_t)idx[c4 * 4 + 1] << 8) |
                                                                ((uint32_t)idx[c4 * 4 + 2] << 16) |
                                                                ((uint32_t)idx[c4 * 4 + 3] << 24);
              }
            }
#pragma unroll
            for (int o = 0; o < 16; ++o)
              if (h * 16 + o < P.Fout) msum += m[o];
          }
          if (P.y_mean && valid && h0 == 0 && h1 == 2) P.y_mean[orow] = msum / (float)P.Fout;
  };
  // tasks of one tile per lane quarter; the LAST tile of a CTA is shared between the epilogue warp of the quarter and
  // the kSparseWarps / 4 sparse warps that can reach the same TMEM lanes (they have nothing left to do)
  const bool split_halves = P.y_mean == nullptr;  // the mean over filters needs both halves in one thread
  const int ntask = G * P.T * (split_halves ? 2 : 1);
  constexpr int kTailShare = 1 + kSparseWarps / 4;
  auto tail_tasks = [&](int tile, int buf, int e, int j) {  // participant j of kTailShare in quarter e
    for (int k = j; k < ntask; k += kTailShare) {
      const int gt = split_halves ? (k >> 1) : k;
      const int g = gt / P.T, t = gt - g * P.T;
      if (split_halves) epi_task(tile, buf, e, g, t, k & 1, (k & 1) + 1);
      else epi_task(tile, buf, e, g, t, 0, 2);
    }
  };
  // Between two layers of a stack (p = 1, 32 -> 32): one half (16 filters) of accumulator tile t for TMEM lane quarter e.
  // thread = vertex: bias of layer l, ReLU, and the row goes straight into the state buffer (+ its bf16 remainder) as
  // order 0 of layer l + 1.
  // (the bias of the task is loaded separately so that a caller can have it in flight before the accumulators are final)
  auto inner_bias = [&](int e, int t, int h, int l, float (&bv)[16]) {
    const int rb = t * 128 + e * 32 + lane;
#pragma unroll
    for (int o = 0; o < 16; ++o) bv[o] = 0.f;
    if (rb >= M || t * 128 + e * 32 >= BQ) return;
    if (P.bias_mode == GCNB_BIAS_PER_VERTEX) {
      const float* bp = P.biasl[l] + (long long)rb * P.Fout + h * 16;
#pragma unroll
      for (int c4 = 0; c4 < 4; ++c4) {
        const float4 q4 = __ldg(reinterpret_cast<const float4*>(bp + c4 * 4));
        bv[c4 * 4] = q4.x; bv[c4 * 4 + 1] = q4.y; bv[c4 * 4 + 2] = q4.z; bv[c4 * 4 + 3] = q4.w;
      }
    } else if (P.bias_mode == GCNB_BIAS_PER_FILTER) {
#pragma unroll
      for (int o = 0; o < 16; ++o) bv[o] = bias_s[l * 32 + h * 16 + o];
    }
  };
  auto inner_task = [&](int buf, int e, int t, int h, const float (&bv)[16], uint32_t dst, uint32_t dlo) {
    if (t * 128 + e * 32 >= BQ) return;
    const int rb = t * 128 + e * 32 + lane;  // row = vertex
    float m[16];
    tmem_ld16(tmem + ((uint32_t)(e * 32) << 16) + (uint32_t)(buf * P.acc_cols + t * 32 + h * 16), m);
    if (rb >= M) return;
#pragma unroll
    for (int c4 = 0; c4 < 4; ++c4) {
      float4 v = make_float4(m[c4 * 4] + bv[c4 * 4], m[c4 * 4 + 1] + bv[c4 * 4 + 1], m[c4 * 4 + 2] + bv[c4 * 4 + 2],
                             m[c4 * 4 + 3] + bv[c4 * 4 + 3]);
      if (P.relu) v = make_float4(fmaxf(v.x, 0.f), fmaxf(v.y, 0.f), fmaxf(v.z, 0.f), fmaxf(v.w, 0.f));
      const int c = h * 4 + c4;
      store_state_at(dst + slab_off(rb, c), dlo + lo_off(rb, c), v);
    }
  };
  // this participant's share of the drain between two layers; the bias of its first task is already in bv0
  auto inner_share = [&](int buf, int e, int j, int l, const float (&bv0)[16], uint32_t dst, uint32_t dlo) {
    if (j < P.T * 2) inner_task(buf, e, j >> 1, j & 1, bv0, dst, dlo);
    for (int k2 = j + kTailShare; k2 < P.T * 2; k2 += kTailShare) {
      float bv[16];
      inner_bias(e, k2 >> 1, k2 & 1, l, bv);
      inner_task(buf, e, k2 >> 1, k2 & 1, bv, dst, dlo);
    }
  };
  int my_tiles = 0;
  for (int tile = blockIdx.x; tile < P.ntiles; tile += gridDim.x) ++my_tiles;
  const int my_iters = my_tiles * nlayers;  // (tile, layer) passes of this CTA

  if (warp > kMmaWarp) {
    // =========================================== sparse warps ==================================================
    const int sw = warp - (kMmaWarp + 1);
    const int q = lane >> 3, c = lane & 7;
    const uint32_t c16 = (uint32_t)c << 4;
    const int gw = c / CPW, fc = c - gw * CPW;  // window inside the row, feature chunk inside the window
    // lo offset of the same chunk (64-byte rows, SWIZZLE_64B), from the state offset
    auto lo_of = [c](uint32_t off) {
      const uint32_t rr = off >> 7;
      return rr * 64u + ((((uint32_t)(c >> 1) ^ ((rr >> 1) & 3u)) << 4) | ((uint32_t)(c & 1) << 3));
    };
    // value of element (vertex vtx, window b, features 4 fc .. 4 fc + 3) of order 0: the gathered, zero padded raw
    // window, or (adjoint mode) dZ rebuilt from the pooled gradient, the ReLU mask and the arg-max
    auto load_x0 = [&](int vtx, int b) -> float4 {
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (vtx < 0 || b >= P.B) return v;
      if (P.adj) {
        if (fc * 4 < P.Fin) {
          const int jj = vtx >> P.adj_log2p, ii = vtx & ((1 << P.adj_log2p) - 1);
          const long long prow = (long long)b * P.adj_Mo + jj, gi = prow * P.Fin + fc * 4;
          if (P.adj_mean) {
            const float m = __ldg(P.adj_dy + prow) / (float)P.Fin;
            v = make_float4(m, m, m, m);
          } else {
            v = __ldg(reinterpret_cast<const float4*>(P.adj_dy + gi));
          }
          if (P.adj_relu) {
            const float4 yv = __ldg(reinterpret_cast<const float4*>(P.adj_y + gi));
            if (!(yv.x > 0.f)) v.x = 0.f;
            if (!(yv.y > 0.f)) v.y = 0.f;
            if (!(yv.z > 0.f)) v.z = 0.f;
            if (!(yv.w > 0.f)) v.w = 0.f;
          }
          if (P.adj_log2p > 0) {
            const uint32_t am = __ldg(reinterpret_cast<const uint32_t*>(P.adj_arg + gi));
            if ((int)(am & 0xff) != ii) v.x = 0.f;
            if ((int)((am >> 8) & 0xff) != ii) v.y = 0.f;
            if ((int)((am >> 16) & 0xff) != ii) v.z = 0.f;
            if ((int)(am >> 24) != ii) v.w = 0.f;
          }
        }
      } else {
        const int src = src_row[vtx];
        if (src >= 0) {
          const float* xp = P.x + ((long long)b * P.M_in + src) * P.Fin + fc * 4;
          const int nf = P.Fin - fc * 4;
          if (nf > 0) v.x = __ldg(xp);
          if (nf > 1) v.y = __ldg(xp + 1);
          if (nf > 2) v.z = __ldg(xp + 2);
          if (nf > 3) v.w = __ldg(xp + 3);
        }
      }
      return v;
    };
    if constexpr (IMG) {
      // ---- row-blocked recursion over a host-built operator image -------------------------------------------
      // Work item = (group of four row blocks, window-slab): quarter-warp q owns block q of the group = four
      // consecutive vertices (the siblings of the Graclus ordering share most of their neighbours), lane c of the
      // quarter owns the 16-byte chunk c of their rows.  The entry stream of a group lists, per step, one
      // neighbour of each block (the union of its rows' neighbour sets, ascending) with the four weights of that
      // neighbour (zero where a row does not have it): one gathered row feeds four rows.  Items are dealt to the
      // warps in snake order of the length-sorted groups.
      const uint32_t grp_tab = sb + P.off_grp, img0 = sb + P.off_img;
      const uint16_t* blk = reinterpret_cast<const uint16_t*>(smem + P.off_blk);
      auto item_of = [sw](int u) { return u * kSparseWarps + ((u & 1) ? kSparseWarps - 1 - sw : sw); };
      auto row_of = [=](int vtx, int s) { return (vtx & pm1) * BQ + s * Q + (vtx >> log2p); };
      uint32_t n = 0;  // orders issued so far (all tiles)
      uint32_t stage_phase = 1;  // phase 0 of the staging barrier brought the operator image in
      int base = 0, it = 0;
      TRACE(0, sw == 0);
      for (int tile = blockIdx.x; tile < P.ntiles; tile += gridDim.x)
      for (int l = 0; l < nlayers; ++l, ++it) {
        // ---- order 0 (first layer of a stack: from HBM; later layers: written by the drain of the layer before) ----
        if (l == 0) {
          if (STACK && nlayers > 1 && it > 0) {
            // the tap images still hold the last layer's: rebuild layer 0's once the tensor cores are done with them
            mbar_wait(bar_mma((n - 1) & 1), ((n - 1) >> 1) & 1);
            if (P.tapimg[0] != nullptr) {
              if (sw == 0 && lane == 0) {
                mbar_expect_tx(bar_stage, (uint32_t)P.tap_bytes);
                bulk_g2s(sb + P.off_wh, P.tapimg[0], (uint32_t)P.tap_bytes, bar_stage);
              }
              mbar_wait(bar_stage, stage_phase);
              stage_phase ^= 1u;
            } else {
              taps_of(P.Wl[0], sw * 32 + lane, kSparseWarps * 32);
            }
          }
          const uint32_t lo_u = P.nlo == 2 ? (n & 1u) : 0u;
          if (P.nlo == 1 && n > 0) mbar_wait(bar_mma((n - 1) & 1), ((n - 1) >> 1) & 1);
          const uint32_t dst = sb + (uint32_t)base * buf_bytes, dlo = sb + P.off_lo + lo_u * lo_bytes;
          if (P.stage) {
            // Forward, staged: ONE TMA bulk copy brings the tile's raw windows (contiguous in HBM) into the state buffer
            // this order does not write -- it held X_{K-1} of the previous tile and is dead once that tile's last MMA has
            // read it -- and the Graclus gather + zero padding happens shared -> shared.  (Block-wise global loads of
            // 60-byte rows cost four scalar loads per lane, eight cache lines per instruction: measured 10-15 K cycles
            // per tile against ~4 K for the copy.)
            TRACE0(0);
            const int b0 = tile * P.S, nw = min(P.S, P.B - b0);
            const uint32_t stage = sb + (uint32_t)(base ^ 1) * buf_bytes;
            const uint32_t wbytes = (uint32_t)(P.M_in * P.Fin) * 4u;
            if (sw == 0 && lane == 0) {
              if (n > 0) mbar_wait(bar_mma((n - 1) & 1), ((n - 1) >> 1) & 1);  // the tensor cores are done with that buffer
              mbar_expect_tx(bar_stage, (uint32_t)nw * wbytes);
              bulk_g2s(stage, P.x + (long long)b0 * P.M_in * P.Fin, (uint32_t)nw * wbytes, bar_stage);
            }
            mbar_wait(bar_stage, stage_phase);
            stage_phase ^= 1u;
            TRACE0(1);
            for (int u = 0, ii; (ii = item_of(u)) < NI; ++u) {
              const int g = ii / NS, s = ii - g * NS;
              const int beta = blk[g * 4 + q];
              if (beta == 0xffff) continue;
              const int w = s * G + gw, b = b0 + w;
              const int nf = P.Fin - fc * 4;
#pragma unroll
              for (int i = 0; i < 4; ++i) {
                const int vtx = beta * 4 + i;
                const int src = src_row[vtx];
                float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                if (src >= 0 && w < nw && nf > 0 && !TRACE_NOLOAD) {
                  const uint32_t a = stage + (uint32_t)w * wbytes + (uint32_t)(src * P.Fin + fc * 4) * 4u;
                  if (nf > 3 && (a & 15u) == 0) {
                    v = lds128(a);
                  } else {
                    v.x = lds32(a);
                    if (nf > 1) v.y = lds32(a + 4);
                    if (nf > 2) v.z = lds32(a + 8);
                    if (nf > 3) v.w = lds32(a + 12);
                  }
                }
                const uint32_t off = slab_off(row_of(vtx, s), c);
                store_state_at(dst + off, dlo + lo_of(off), v);
                if (P.xstack && b < P.B && !TRACE_NOSPILL)
                  *reinterpret_cast<float4*>(P.xstack + ((long long)b * M + vtx) * FP + fc * 4) = v;
              }
              TRACE0(2 + u);
            }
          } else
          for (int u = 0, ii; (ii = item_of(u)) < NI; ++u) {
            const int g = ii / NS, s = ii - g * NS;
            const int beta = blk[g * 4 + q];
            if (beta == 0xffff) continue;
            const int b = tile * P.S + s * G + gw;
            float4 v[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) v[i] = load_x0(beta * 4 + i, TRACE_NOLOAD ? P.B : b);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const int vtx = beta * 4 + i;
              const uint32_t off = slab_off(row_of(vtx, s), c);
              store_state_at(dst + off, dlo + lo_of(off), v[i]);
              if (P.xstack && b < P.B && !TRACE_NOSPILL)
                *reinterpret_cast<float4*>(P.xstack + ((long long)b * M + vtx) * FP + fc * 4) = v[i];
            }
          }
          TRACE(0, sw == 0);
          TRACE0(5);
          fence_async_smem();
          TRACE0(6);
          named_bar_sync(kBarOrder, nsync);
          TRACE0(7);
          ++n;
        }
        // ---- orders 1 .. K-1 ----------------------------------------------------------------------------------
        for (int k = 1; k < K; ++k) {
          const int cur = (base + k) & 1;
          const uint32_t lo_u = P.nlo == 2 ? (n & 1u) : 0u;
          bool lo_free = P.nlo == 2;  // single remainder buffer: the tensor cores must be done with order n-1 first
          float* spill = (P.xstack && !TRACE_NOSPILL) ? P.xstack + (long long)k * P.B * M * FP : nullptr;
          const uint32_t dlo = sb + P.off_lo + lo_u * lo_bytes;
          const uint32_t srcb = sb + (uint32_t)(cur ^ 1) * buf_bytes, dst = sb + (uint32_t)cur * buf_bytes;
          if (k == K - 1 && !P.adj && l == nlayers - 1 && tile + (int)gridDim.x < P.ntiles) {
            // pull the next tile's raw windows into L2 while this order computes
            for (int u = 0, ii; (ii = item_of(u)) < NI; ++u) {
              const int g = ii / NS, s = ii - g * NS;
              const int beta = blk[g * 4 + q];
              const int b = (tile + (int)gridDim.x) * P.S + s * G + gw;
              if (beta != 0xffff && b < P.B && fc * 4 < P.Fin) {
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                  const int src = src_row[beta * 4 + i];
                  if (src >= 0)
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(P.x + ((long long)b * P.M_in + src) * P.Fin + fc * 4));
                }
              }
            }
          }
          TRACEW(0);
          // With a single remainder buffer the lo stores of this order must not land before the tensor cores are done
          // with order n-1: since the MMAs of an order take ~400 cycles (issued right after the barrier) that wait is over
          // long before the first item reaches its stores.
          auto do_item = [&](int u, int ii) {
            const int g = ii / NS, s = ii - g * NS;
            const uint2 gr = lds64u(grp_tab + (uint32_t)g * 8u);  // (offset of the entry stream in the image, steps)
            const int beta = blk[g * 4 + q];
            const uint32_t srcs = srcb + ((uint32_t)(s * Q) << 7);  // window-slab offset keeps the swizzle phase
            uint32_t wa = img0 + gr.x + (uint32_t)q * 16u, ca = img0 + gr.x + 128u + (uint32_t)q * 4u;
            // accumulators packed by PAIRS OF ROWS: c01[f] = (row 0, row 1) of feature f, c23[f] = (row 2, row 3).  One
            // fma.rn.f32x2 (two IEEE fp32 FMAs, bit-identical to fmaf) multiplies the weight pair of two rows -- adjacent
            // words of the entry stream -- by a duplicated gathered value: 12 issue slots per gathered row instead of 16
            // (the loop is issue-bound).
            uint64_t c01[4] = {0ull, 0ull, 0ull, 0ull}, c23[4] = {0ull, 0ull, 0ull, 0ull};
            int steps = (int)gr.y;
#ifdef GCNB_TRACE
            if (P.debug & 1) steps = 0;
#endif
            // software pipeline: the codes and weights of the next pair of steps are in flight while this pair's two
            // gathers return (the read past the last pair of a group stays inside the image / the tables behind it)
            uint32_t cc = lds32u(ca);  // two 16-bit row codes: (row * 8 + (row & 7)) << 4 is the gather code
            float4 w0 = lds128(wa), w1 = lds128(wa + 64u);
#pragma unroll 1
            for (int j = 0; j < steps; j += 2) {
              const float4 v0 = lds128(srcs + (((cc & 0xffffu) << 4) ^ c16));
              const float4 v1 = lds128(srcs + (((cc >> 12) & 0xffff0u) ^ c16));
              wa += kImgPair;
              ca += kImgPair;
              const uint32_t ccn = lds32u(ca);
              const float4 w0n = lds128(wa), w1n = lds128(wa + 64u);
              {
                const uint64_t wl = pack2(w0.x, w0.y), wh = pack2(w0.z, w0.w);
                const uint64_t x = pack2(v0.x, v0.x), y = pack2(v0.y, v0.y), z = pack2(v0.z, v0.z), w = pack2(v0.w, v0.w);
                c01[0] = fma2(wl, x, c01[0]); c23[0] = fma2(wh, x, c23[0]);
                c01[1] = fma2(wl, y, c01[1]); c23[1] = fma2(wh, y, c23[1]);
                c01[2] = fma2(wl, z, c01[2]); c23[2] = fma2(wh, z, c23[2]);
                c01[3] = fma2(wl, w, c01[3]); c23[3] = fma2(wh, w, c23[3]);
              }
              {
                const uint64_t wl = pack2(w1.x, w1.y), wh = pack2(w1.z, w1.w);
                const uint64_t x = pack2(v1.x, v1.x), y = pack2(v1.y, v1.y), z = pack2(v1.z, v1.z), w = pack2(v1.w, v1.w);
                c01[0] = fma2(wl, x, c01[0]); c23[0] = fma2(wh, x, c23[0]);
                c01[1] = fma2(wl, y, c01[1]); c23[1] = fma2(wh, y, c23[1]);
                c01[2] = fma2(wl, z, c01[2]); c23[2] = fma2(wh, z, c23[2]);
                c01[3] = fma2(wl, w, c01[3]); c23[3] = fma2(wh, w, c23[3]);
              }
              cc = ccn; w0 = w0n; w1 = w1n;
            }
            float4 a0, a1, a2, a3;
            unpack2(c01[0], a0.x, a1.x); unpack2(c01[1], a0.y, a1.y); unpack2(c01[2], a0.z, a1.z); unpack2(c01[3], a0.w, a1.w);
            unpack2(c23[0], a2.x, a3.x); unpack2(c23[1], a2.y, a3.y); unpack2(c23[2], a2.z, a3.z); unpack2(c23[3], a2.w, a3.w);
            TRACEW(1 + u * 3);
            if (!lo_free) {
              mbar_wait(bar_mma((n - 1) & 1), ((n - 1) >> 1) & 1);
              lo_free = true;
            }
            TRACEW(2 + u * 3);
            if (beta != 0xffff) {
              const int b = tile * P.S + s * G + gw;
              const float4 acc[4] = {a0, a1, a2, a3};
#pragma unroll
              for (int i = 0; i < 4; ++i) {
                const int vtx = beta * 4 + i;
                const uint32_t off = slab_off(row_of(vtx, s), c);
                float4 o = acc[i];
                if (k > 1) {
                  const float4 own = lds128(dst + off);
                  o = make_float4(fmaf(2.f, o.x, -own.x), fmaf(2.f, o.y, -own.y), fmaf(2.f, o.z, -own.z), fmaf(2.f, o.w, -own.w));
                }
                sts128(dst + off, o);
                const float rx = o.x - tf32_trunc(o.x), ry = o.y - tf32_trunc(o.y);
                const float rz = o.z - tf32_trunc(o.z), rw = o.w - tf32_trunc(o.w);
                const uint2 rem = make_uint2(pack_bf16(rx, ry), pack_bf16(rz, rw));
                sts64(dlo + lo_of(off), rem.x, rem.y);
                if (spill && b < P.B) *reinterpret_cast<float4*>(spill + ((long long)b * M + vtx) * FP + fc * 4) = o;
              }
            }
            TRACEW(3 + u * 3);
          };
          for (int u = 0, ii; (ii = item_of(u)) < NI; ++u) do_item(u, ii);
          TRACE(0, sw == 0);
          TRACEW(13);
          fence_async_smem();
          TRACEW(14);
          named_bar_sync(kBarOrder, nsync);
          TRACEW(15);
          ++n;
        }
        base = (base + K) & 1;
        if (STACK && l + 1 < nlayers) {
          // ---- layer boundary: taps of the next layer, accumulators -> order 0 of the next layer ---------------------
          const int buf = P.nacc == 2 ? (it & 1) : 0;
          const int use = P.nacc == 2 ? (it >> 1) : it;
          const int e = warp & 3;
          const int j = 1 + (warp - (5 + ((e + 3) & 3))) / 4;  // sparse warps of TMEM lane quarter e, in warp order
          // static data first: the next layer's taps and this warp's bias rows are in flight while the last MMA finishes
          constexpr int nt = kSparseWarps * 32;
          const int t_ = sw * 32 + lane;
          float w0[4] = {0.f, 0.f, 0.f, 0.f}, w1[4] = {0.f, 0.f, 0.f, 0.f}, bv0[16];
          const bool tap_tma = P.tapimg[l + 1] != nullptr;  // pre-split taps: one TMA bulk copy instead of the re-split
          TRACEB(sw, 0);
          if (!tap_tma) {
            tap_load(P.Wl[l + 1], 0, t_, nt, w0);
            tap_load(P.Wl[l + 1], nt * 4, t_, nt, w1);
          }
          inner_bias(e, j >> 1, j & 1, l, bv0);
          TRACEB(sw, 1);
          mbar_wait(bar_full(buf), (uint32_t)use & 1u);  // the layer's last MMA is complete: taps and remainder free
          tc_fence_after();
          TRACEB(sw, 2);
          if (tap_tma) {
            if (sw == 0 && lane == 0) {
              mbar_expect_tx(bar_stage, (uint32_t)P.tap_bytes);
              bulk_g2s(sb + P.off_wh, P.tapimg[l + 1], (uint32_t)P.tap_bytes, bar_stage);
            }
          } else {
            tap_store(0, t_, nt, w0);
            tap_store(nt * 4, t_, nt, w1);
            for (int i0 = 2 * nt * 4; i0 < K * FP * 32; i0 += nt * 4) {
              float wv[4];
              tap_load(P.Wl[l + 1], i0, t_, nt, wv);
              tap_store(i0, t_, nt, wv);
            }
          }
          const uint32_t dst = sb + (uint32_t)base * buf_bytes, dlo = sb + P.off_lo + (P.nlo == 2 ? (n & 1u) : 0u) * lo_bytes;
          TRACEB(sw, 3);
          inner_share(buf, e, j, l, bv0, dst, dlo);
          if (tap_tma) {  // the copy ran beside the drain
            mbar_wait(bar_stage, stage_phase);
            stage_phase ^= 1u;
          }
          TRACEB(sw, 4);
          tc_fence_before();
          fence_async_smem();
          TRACEB(sw, 5);
          named_bar_sync(kBarLayer, kThreads);
          TRACEB(sw, 6);
          ++n;
        }
      }
    } else {
      // The rows a lane works on never change: keep what the order loop needs of each of its (up to MAXI) items in
      // registers -- state offset of its 16-byte chunk, address of its entry list, lengths, vertex id.
      uint32_t it_off[MAXI], it_ent[MAXI], it_pk[MAXI];  // pk: own pairs | group pairs << 8 | window-in-tile << 16
      int it_row[MAXI];                                   // vertex (-1: no work), for the global addresses
  #pragma unroll
      for (int u = 0; u < MAXI; ++u) {
        const int ii = u * kSparseWarps + ((u & 1) ? kSparseWarps - 1 - sw : sw);  // snake deal of the sorted groups
        it_row[u] = -1;
        it_off[u] = 0; it_ent[u] = sb + P.off_ent; it_pk[u] = 0;
        if (ii < NI) {
          const int g = ii / NS, s = ii - g * NS;
          const int2 meta = gslot[g * 4 + q];
          const int rr = grho[g * 4 + q] + s * Q;
          it_row[u] = grow[g * 4 + q];
          it_off[u] = slab_off(rr, c);
          it_ent[u] = sb + P.off_ent + (uint32_t)meta.x * 16u;
          it_pk[u] = (uint32_t)((meta.y + 1) >> 1) | ((uint32_t)glen[g] << 8) | ((uint32_t)(s * G + gw) << 16) |
                     ((uint32_t)s << 24);
        }
      }
      uint32_t n = 0;  // orders issued so far (all tiles)
      int base = 0;
      TRACE(0, sw == 0);
      for (int tile = blockIdx.x; tile < P.ntiles; tile += gridDim.x) {
        // ---- order 0: the (gathered, zero padded) raw windows -----------------------------------------------
        {
          const uint32_t lo_u = P.nlo == 2 ? (n & 1u) : 0u;
          if (P.nlo == 1 && n > 0) mbar_wait(bar_mma((n - 1) & 1), ((n - 1) >> 1) & 1);
          const uint32_t dst = sb + (uint32_t)base * buf_bytes, dlo = sb + P.off_lo + lo_u * lo_bytes;
          float4 v[MAXI];
  #pragma unroll
          for (int u = 0; u < MAXI; ++u) {
            v[u] = load_x0(it_row[u], tile * P.S + (int)((it_pk[u] >> 16) & 0xff));
          }
#pragma unroll
          for (int u = 0; u < MAXI; ++u) {
            if (it_row[u] >= 0) {
              store_state_at(dst + it_off[u], dlo + lo_of(it_off[u]), v[u]);
              const int b = tile * P.S + (int)((it_pk[u] >> 16) & 0xff);
              if (P.xstack && b < P.B)
                *reinterpret_cast<float4*>(P.xstack + ((long long)b * M + it_row[u]) * FP + fc * 4) = v[u];
            }
          }
          TRACE(0, sw == 0);
          fence_async_smem();
          named_bar_sync(kBarOrder, nsync);
          ++n;
        }
        // ---- orders 1 .. K-1 --------------------------------------------------------------------------------
        for (int k = 1; k < K; ++k) {
          const int cur = (base + k) & 1;
          const uint32_t lo_u = P.nlo == 2 ? (n & 1u) : 0u;
          if (P.nlo == 1) mbar_wait(bar_mma((n - 1) & 1), ((n - 1) >> 1) & 1);
          float* spill = P.xstack ? P.xstack + (long long)k * P.B * M * FP : nullptr;
          const uint32_t dlo = sb + P.off_lo + lo_u * lo_bytes;
          const uint32_t srcb = sb + (uint32_t)(cur ^ 1) * buf_bytes, dst = sb + (uint32_t)cur * buf_bytes;
          if (k == K - 1 && !P.adj && tile + (int)gridDim.x < P.ntiles) {
            // pull the next tile's raw windows into L2 while this order computes
  #pragma unroll
            for (int u = 0; u < MAXI; ++u) {
              const int b = (tile + (int)gridDim.x) * P.S + (int)((it_pk[u] >> 16) & 0xff);
              if (it_row[u] >= 0 && b < P.B && fc * 4 < P.Fin) {
                const int src = src_row[it_row[u]];
                if (src >= 0)
                  asm volatile("prefetch.global.L2 [%0];" ::"l"(P.x + ((long long)b * P.M_in + src) * P.Fin + fc * 4));
              }
            }
          }
          // Two work items at a time (the snake deal makes neighbours in the list near-equal in length): twice the
          // independent shared-memory loads in flight per warp.
          auto finish = [&](int row, uint32_t off, uint32_t pk, float a0, float a1, float a2, float a3) {
            if (row >= 0) {
              float4 o;
              if (k == 1) {
                o = make_float4(a0, a1, a2, a3);
              } else {
                const float4 own = lds128(dst + off);
                o = make_float4(fmaf(2.f, a0, -own.x), fmaf(2.f, a1, -own.y), fmaf(2.f, a2, -own.z), fmaf(2.f, a3, -own.w));
              }
              store_state_at(dst + off, dlo + lo_of(off), o);
              const int b = tile * P.S + (int)((pk >> 16) & 0xff);
              if (spill && b < P.B) *reinterpret_cast<float4*>(spill + ((long long)b * M + row) * FP + fc * 4) = o;
            }
          };
  #pragma unroll
          for (int u = 0; u < MAXI; u += 2) {
            const bool two = u + 1 < MAXI;
            const int u1 = two ? u + 1 : u;
            const uint32_t pka = it_pk[u], pkb = two ? it_pk[u1] : 0u;
            const int owna = (int)(pka & 0xff), ownb = (int)(pkb & 0xff);
            int lim = max((int)((pka >> 8) & 0xff), (int)((pkb >> 8) & 0xff));
  #ifdef GCNB_TRACE
            if (P.debug & 1) lim = 0;
  #endif
            const uint32_t srca = srcb + ((pka >> 24) * (uint32_t)Q << 7);  // window-slab offset keeps the swizzle phase
            const uint32_t srcq = srcb + ((pkb >> 24) * (uint32_t)Q << 7);
            const uint32_t ea = it_ent[u], eb = it_ent[u1];
            const int lasta = max(owna - 1, 0), lastb = max(ownb - 1, 0);
            float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f, b0 = 0.f, b1 = 0.f, b2 = 0.f, b3 = 0.f;
            // Branch-free over the longest row of the two groups: a lane whose own row is shorter re-reads its last
            // entry pair with zero weights.
            for (int j = 0; j < lim; ++j) {
              const int4 e = lds128i(ea + (uint32_t)min(j, lasta) * 16u);
              const int4 f = lds128i(eb + (uint32_t)min(j, lastb) * 16u);
              const float4 v0 = lds128(srca + ((uint32_t)e.x ^ c16));
              const float4 v1 = lds128(srca + ((uint32_t)e.z ^ c16));
              const float4 x0 = lds128(srcq + ((uint32_t)f.x ^ c16));
              const float4 x1 = lds128(srcq + ((uint32_t)f.z ^ c16));
              const bool la = j < owna, lb = two && j < ownb;
              const float w0 = la ? __int_as_float(e.y) : 0.f, w1 = la ? __int_as_float(e.w) : 0.f;
              const float z0 = lb ? __int_as_float(f.y) : 0.f, z1 = lb ? __int_as_float(f.w) : 0.f;
              a0 = fmaf(w0, v0.x, a0); a1 = fmaf(w0, v0.y, a1); a2 = fmaf(w0, v0.z, a2); a3 = fmaf(w0, v0.w, a3);
              b0 = fmaf(z0, x0.x, b0); b1 = fmaf(z0, x0.y, b1); b2 = fmaf(z0, x0.z, b2); b3 = fmaf(z0, x0.w, b3);
              a0 = fmaf(w1, v1.x, a0); a1 = fmaf(w1, v1.y, a1); a2 = fmaf(w1, v1.z, a2); a3 = fmaf(w1, v1.w, a3);
              b0 = fmaf(z1, x1.x, b0); b1 = fmaf(z1, x1.y, b1); b2 = fmaf(z1, x1.z, b2); b3 = fmaf(z1, x1.w, b3);
            }
            finish(it_row[u], it_off[u], pka, a0, a1, a2, a3);
            if (two) finish(it_row[u1], it_off[u1], pkb, b0, b1, b2, b3);
          }
          TRACE(0, sw == 0);
          fence_async_smem();
          named_bar_sync(kBarOrder, nsync);
          ++n;
        }
        base = (base + K) & 1;
      }
    }
    // the CTA's last tile: help the epilogue warp of this warp's TMEM lane quarter
    if (my_tiles > 0) {
      const int it = my_iters - 1;
      const int buf = P.nacc == 2 ? (it & 1) : 0;
      const int use = P.nacc == 2 ? (it >> 1) : it;
      const int e = warp & 3;
      const int j = 1 + (warp - (5 + ((e + 3) & 3))) / 4;  // sparse warps of quarter e, in warp order
      mbar_wait(bar_full(buf), (uint32_t)use & 1u);
      tc_fence_after();
      tail_tasks(blockIdx.x + (my_tiles - 1) * (int)gridDim.x, buf, e, j);
      tc_fence_before();
    }
  } else if (warp == kMmaWarp) {
    // =========================================== MMA warp ======================================================
    uint32_t n = 0;
    int base = 0, it = 0;
    for (int tile = blockIdx.x; tile < P.ntiles; tile += gridDim.x)
    for (int l = 0; l < nlayers; ++l, ++it) {
      const int buf = P.nacc == 2 ? (it & 1) : 0;
      const int use = P.nacc == 2 ? (it >> 1) : it;  // earlier uses of this accumulator buffer
      if (use > 0) mbar_wait(bar_empty(buf), (uint32_t)(use - 1) & 1u);
      for (int k = 0; k < K; ++k) {
        // X_k (and its remainder) is complete in shared memory; order 0 of a later layer comes from the drain
        if (STACK && k == 0 && l > 0) named_bar_sync(kBarLayer, kThreads);
        else named_bar_sync(kBarOrder, nsync);
        TRACE(2, true);
        tc_fence_after();
        {
          // The whole warp walks the (warp-uniform) issue loop and only the tcgen05 instructions themselves are
          // predicated on the elected lane: descriptor arithmetic then stays in the uniform datapath instead of a
          // per-instruction register -> uniform-register waterfall inside a divergent branch.
          const bool leader = elect_one();
          // ONE thread issues every MMA of the order.  Inside an `if (lane == 0)` branch ptxas wraps every tcgen05.mma in
          // a register -> uniform-register waterfall loop (~18 instructions each); under the load of the sparse warps that
          // made the issue of the 40 MMAs of an order take 5-8 K cycles, i.e. as long as the sparse phase itself (clock64
          // trace of CTA 0).  With the elect.sync predicate the sequence is a handful of uniform adds per instruction and
          // the tensor-core work of an order (issue + execution) is ~400 cycles, off the critical path.
          const int cur = (base + k) & 1;
          const uint32_t lo_u = P.nlo == 2 ? (n & 1u) : 0u;
          const uint32_t sbuf = sb + (uint32_t)cur * buf_bytes, lbuf = sb + P.off_lo + lo_u * lo_bytes;
          uint64_t bh[FP / 8], bl[FP / 8], bb[FP / 16];
#pragma unroll
          for (int j = 0; j < FP / 8; ++j) {
            bh[j] = smem_desc(kDescTaps, sb + P.off_wh + (uint32_t)(k * (FP / 4) * 4) * 128u + j * 1024);
            bl[j] = smem_desc(kDescTaps, sb + P.off_wl + (uint32_t)(k * (FP / 4) * 4) * 128u + j * 1024);
          }
#pragma unroll
          for (int j = 0; j < FP / 16; ++j)
            bb[j] = smem_desc(kDescTaps, sb + P.off_wb + (uint32_t)(k * (FP / 8) * 4) * 128u + j * 1024);
          const uint32_t first_acc = k != 0;
          const uint32_t d0 = tmem + (uint32_t)(buf * P.acc_cols);
          uint32_t idesc_tf32 = kIdescTf32, idesc_bf16 = kIdescBf16;
          if constexpr (RAW) {
            // at most 16 output columns: the zero tap columns 16..31 are not multiplied (the epilogue never reads them)
            if (P.Fout <= 16) idesc_tf32 = kIdescTf32N16, idesc_bf16 = kIdescBf16N16;
          }
#ifdef GCNB_TRACE
          const bool t_tf32 = !(P.debug & 16), t_lo = !(P.debug & 64), t_bf16 = !(P.debug & 32);
          if (!(P.debug & 2))
#else
          constexpr bool t_tf32 = true, t_lo = true, t_bf16 = true;
#endif
#pragma unroll
          for (int g = 0; g < G; ++g) {
            // descriptor start-address fields (16-byte units) of block (g, i = 0, t = 0)
            uint32_t ai = ((sbuf + (uint32_t)(g * FP * 4)) >> 4) & 0x3fffu, li = ((lbuf + (uint32_t)(g * FP * 2)) >> 4) & 0x3fffu;
            uint32_t d = d0 + (uint32_t)(g * P.p * P.T * 32);
            for (int i = 0; i < P.p; ++i) {
              uint32_t at = ai, lt = li;
              for (int t = 0; t < P.T; ++t) {
                const uint64_t da = kDescSlab | at, dl = kDescLo | lt;
                if (leader) {
#pragma unroll
                  for (int j = 0; j < FP / 8; ++j)
                    if (t_tf32) mma_tf32(d, da + 2 * j, bh[j], idesc_tf32, j ? 1u : first_acc);
#pragma unroll
                  for (int j = 0; j < FP / 8; ++j)
                    if (t_tf32 && t_lo) mma_tf32(d, da + 2 * j, bl[j], idesc_tf32, 1);
#pragma unroll
                  for (int j = 0; j < FP / 16; ++j)
                    if (t_bf16) mma_bf16(d, dl + 2 * j, bb[j], idesc_bf16, 1);
                }
                d += 32;
                at += 128 * 128 / 16;  // the next 128 rows of the block
                lt += 128 * 64 / 16;
              }
              ai += (uint32_t)BQ * 128 / 16;  // the next sibling block
              li += (uint32_t)BQ * 64 / 16;
            }
          }
          if (leader) {
            mma_commit(bar_mma(n & 1));
            if (k == K - 1) mma_commit(bar_full(buf));
          }
        }
        __syncwarp();
        TRACE(2, true);
        // X_k's buffer and remainder may be overwritten two orders from now: only pass the next barrier once the
        // tensor cores have finished reading them
        mbar_wait(bar_mma(n & 1), (n >> 1) & 1);
        TRACE(2, true);
        ++n;
      }
      base = (base + K) & 1;
    }
  } else {
    // =========================================== epilogue warps =================================================
    const int e = warp;  // TMEM lane quarter
    int it = 0;
    for (int tile = blockIdx.x; tile < P.ntiles; tile += gridDim.x)
    for (int l = 0; l < nlayers; ++l, ++it) {
      const int buf = P.nacc == 2 ? (it & 1) : 0;
      const int use = P.nacc == 2 ? (it >> 1) : it;
      float bv0[16];
      if (STACK && l + 1 < nlayers) inner_bias(e, 0, 0, l, bv0);  // static: loaded before the accumulators are final
      mbar_wait_relaxed(bar_full(buf), (uint32_t)use & 1u);
      TRACE(3, e == 0);
      tc_fence_after();
      if (STACK && l + 1 < nlayers) {
        // layer boundary: this warp's share of the drain into order 0 of the next layer (participant 0 of its quarter)
        const uint32_t n_next = (uint32_t)(it + 1) * (uint32_t)K;
        const uint32_t dst = sb + (n_next & 1u) * buf_bytes, dlo = sb + P.off_lo + (P.nlo == 2 ? (n_next & 1u) : 0u) * lo_bytes;
        TRACEB(20 + e, 2);
        inner_share(buf, e, 0, l, bv0, dst, dlo);
        TRACEB(20 + e, 4);
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(bar_empty(buf));
        fence_async_smem();
        TRACEB(20 + e, 5);
        named_bar_sync(kBarLayer, kThreads);
        TRACEB(20 + e, 6);
        continue;
      }
      if (it + 1 == my_iters) {
        tail_tasks(tile, buf, e, 0);
      } else {
#pragma unroll
        for (int g = 0; g < G; ++g)
          for (int t = 0; t < P.T; ++t) epi_task(tile, buf, e, g, t, 0, 2);
      }
      TRACE(3, e == 0);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_empty(buf));
    }
  }

  // ---- teardown -----------------------------------------------------------------------------------------------
  tc_fence_before();
  __syncthreads();
  if (warp == kMmaWarp) {
    tc_fence_after();
    tmem_dealloc(tmem, (uint32_t)P.tmem_cols);
  }
}

// ---------------------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------------------
// Operator image (gcnb_cheb_image_build, consumed by the IMG kernels).  Vertices are taken in blocks of four
// consecutive rows (in the Graclus ordering: siblings, which share most of their neighbours); a block's entry list is
// the ascending union of its rows' neighbour sets with the four weights per neighbour.  Blocks are sorted by list
// length and grouped by four (one block per quarter-warp).  Layout, all offsets from the start of the image:
//   [0, 64)    header: magic, signature, bytes, groups
//   grp_off    groups x {u32 offset of the entry stream, u32 steps (even)}
//   blk_off    groups x 4 x u16 block index (0xffff: no block in this quarter)
//   ent_off    per group, per pair of steps (144 B): weights of step j for the 4 quarters (4 x 16 B), of step j+1
//              (4 x 16 B), 16-bit row codes of (j, j+1) for the 4 quarters (4 x 4 B); code = row * 8 + (row & 7), i.e. the
//              gather code (row * 128 + swizzle phase) >> 4.  Padding steps gather the zero row.
struct ImgGeom {
  int nb, ng;
  size_t grp_off, blk_off, ent_off;
};
static ImgGeom img_geom(int M) {
  ImgGeom g;
  g.nb = M / 4;
  g.ng = ceil_div(g.nb, 4);
  g.grp_off = 64;
  g.blk_off = g.grp_off + align_up((size_t)g.ng * 8, 16);
  g.ent_off = g.blk_off + align_up((size_t)g.ng * 8, 16);
  return g;
}

struct UmmaFwdPlan {
  bool ok, img;
  int FP, G, NS, Q, BQ, T, NG, nlo, nacc, acc_cols, tmem_cols, slab_rows, MAXI;
  size_t smem, img_bytes;
  int off_lo, off_wh, off_wl, off_wb, off_ent, off_grow, off_grho, off_gslot, off_glen, off_src, off_rlen, off_sorted,
      off_bias, off_bar, off_rp, off_img;
};

// ent_bytes < 0: the kernel builds its own (CSR-ordered) operator image in the prologue; otherwise the entry streams of
// a host-built image take ent_bytes.  raw: the adjoint instances that store rows of any width (RAW), Fout % 4 != 0 too.
static UmmaFwdPlan plan_umma_fwd(const LayerShape& s, int sm_count, int smem_optin, long long ent_bytes = -1,
                                 bool raw = false) {
  UmmaFwdPlan pl{};
  pl.ok = false;
  pl.img = ent_bytes >= 0;
  if (s.Fin <= 8 || s.Fin > 32 || s.Fout < 4 || s.Fout > 32 || (!raw && (s.Fout & 3))) return pl;
  if (s.p != 1 && s.p != 2 && s.p != 4 && s.p != 8) return pl;
  if (s.M % s.p != 0 || s.M < 1 || s.M > 2048 || s.K < 1 || s.B < 1) return pl;
  if (pl.img && (s.M & 3)) return pl;
  pl.FP = s.Fin <= 16 ? 16 : 32;
  pl.G = 32 / pl.FP;
  pl.NG = pl.img ? img_geom(s.M).ng : ceil_div(s.M, 4);
  pl.Q = (int)align_up((size_t)(s.M / s.p), 8);
  pl.img_bytes = pl.img ? img_geom(s.M).ent_off + (size_t)ent_bytes : 0;
  const size_t taps = (size_t)s.K * pl.FP * 32 * 4;  // one tf32 image
  const size_t ent = pl.img ? pl.img_bytes : align_up(((size_t)s.nnz + s.M + 2) * 8, 16);
  const size_t small = align_up((size_t)s.M * 4, 16) /*src*/ + 8 * 128 /*bias rows of up to 8 stacked layers*/ + 64 /*barriers*/;
  const size_t tables = pl.img ? small : 2 * (size_t)pl.NG * 16 /*grow, grho*/ + (size_t)pl.NG * 32 /*gslot*/ +
                                             align_up((size_t)pl.NG * 4, 16) + small;
  // prologue-only scratch (rlen, sorted, rp) lives in the first remainder buffer
  const size_t scratch =
      pl.img ? 0 : 2 * (size_t)pl.NG * 16 + align_up((size_t)(s.M + 3) * 4, 16) + align_up((size_t)(s.M + 1) * 4, 16);
  const size_t budget = std::min<size_t>((size_t)smem_optin, 227 * 1024);
  double best = 1e30;
  for (int ns = 1; ns <= 8; ++ns) {
    const int BQ = ns * pl.Q, T = ceil_div(BQ, 128);
    const int acc_cols = pl.G * s.p * T * 32;
    if (acc_cols > 512) continue;
    const int rows = (int)align_up((size_t)s.p * BQ + 1, 8);
    if ((size_t)rows * 128 >= (1u << 18)) continue;          // descriptors address 256 KB
    if (!pl.img && pl.NG * ns > 5 * kSparseWarps) continue;  // a lane keeps at most 5 work items in registers
    for (int nlo = 2; nlo >= 1; --nlo) {
      const size_t need = 2 * (size_t)rows * 128 + (size_t)nlo * rows * 64 + 2 * taps + taps / 2 + ent + tables;
      // the last MMA tile of the last block reads up to row (p-1)*BQ + T*128: those bytes must exist in the allocation
      const long long over = ((long long)(s.p - 1) * BQ + T * 128 - rows) * 128;
      // a second remainder buffer is a convenience (no waiting for the previous order's MMAs, which take ~400 cycles): only
      // when it leaves 8 KB of the SM's shared memory free -- tools that instrument a launch (ncu --set full) need some
      if (nlo == 2 && need + 8192 > budget) continue;
      if (need > budget || 2 * (size_t)rows * 128 + (over > 0 ? (size_t)over : 0) > need || scratch > (size_t)rows * 64) continue;
      const int tiles = ceil_div(s.B, ns * pl.G);
      // rounds of tiles over the SMs x work per tile; MMA rows wasted by a nearly empty last tile of a block count a little
      const double cost = std::ceil((double)tiles / sm_count) * ns * (nlo == 2 || pl.img ? 1.0 : 1.08) + 0.02 * T * 128.0 / BQ - 0.001 * ns;
      if (cost < best) {
        best = cost;
        pl.NS = ns; pl.BQ = BQ; pl.T = T; pl.nlo = nlo; pl.acc_cols = acc_cols; pl.slab_rows = rows; pl.smem = need;
      }
      break;
    }
  }
  if (best > 1e29) return pl;
  pl.nacc = 2 * pl.acc_cols <= 512 ? 2 : 1;
  pl.MAXI = pl.img ? 1 : (ceil_div(pl.NG * pl.NS, kSparseWarps) <= 3 ? 3 : 5);
  int cols = 32;
  while (cols < pl.nacc * pl.acc_cols) cols *= 2;
  pl.tmem_cols = cols;
  size_t off = 2 * (size_t)pl.slab_rows * 128;
  pl.off_lo = (int)off; off += (size_t)pl.nlo * pl.slab_rows * 64;
  pl.off_wh = (int)off; off += taps;
  pl.off_wl = (int)off; off += taps;
  pl.off_wb = (int)off; off += taps / 2;
  if (pl.img) {
    pl.off_img = (int)off; off += pl.img_bytes;
  } else {
    pl.off_ent = (int)off; off += ent;
    pl.off_grow = (int)off; off += (size_t)pl.NG * 16;
    pl.off_grho = (int)off; off += (size_t)pl.NG * 16;
    pl.off_gslot = (int)off; off += (size_t)pl.NG * 32;
    pl.off_glen = (int)off; off += align_up((size_t)pl.NG * 4, 16);
  }
  pl.off_src = (int)off; off += align_up((size_t)s.M * 4, 16);
  pl.off_bias = (int)off; off += 8 * 128;
  pl.off_bar = (int)off; off += 64;
  pl.off_rlen = pl.off_lo;
  pl.off_sorted = pl.off_rlen + pl.NG * 16;
  pl.off_rp = pl.off_sorted + pl.NG * 16 + (int)align_up((size_t)(s.M + 3) * 4, 16);  // sorted doubles as the bins
  if (off > pl.smem) return pl;
  pl.ok = true;
  return pl;
}

static void plan_device(DeviceInfo* di) {
  if (device_info(di) != GCNB_OK) {  // no device visible (shape queries on a CPU box): assume a B200
    di->sm_count = 148;
    di->smem_optin = 227 * 1024;
  }
}

// what an image must agree on with the kernel that reads it
static unsigned img_signature(const LayerShape& s, const UmmaFwdPlan& pl) {
  unsigned h = 2166136261u;
  const int v[] = {3 /*layout version*/, s.M, s.nnz, s.p, pl.FP, pl.NS, pl.Q, pl.BQ, pl.NG, (int)pl.img_bytes, kSparseWarps};
  for (int x : v) {
    h ^= (unsigned)x;
    h *= 16777619u;
  }
  return h;
}

bool umma_fwd_supported(const LayerShape& s) {
  DeviceInfo di;
  plan_device(&di);
  return plan_umma_fwd(s, di.sm_count, di.smem_optin).ok;
}

int umma_fwd_describe(const LayerShape& s, char* out, size_t n) {
  DeviceInfo di;
  plan_device(&di);
  const UmmaFwdPlan pl = plan_umma_fwd(s, di.sm_count, di.smem_optin);
  if (!pl.ok) return 0;
  return snprintf(out, n,
                  "k_cheb_fwd_umma<FP=%d>: tcgen05/TMEM, %d windows/tile (%d slabs x %d), sibling block %d rows (Q=%d), "
                  "%d MMA tiles/block, %d remainder buffers, %d accumulator buffers x %d TMEM columns, %zu B smem, %d tiles",
                  pl.FP, pl.NS * pl.G, pl.NS, pl.G, pl.BQ, pl.Q, pl.T, pl.nlo, pl.nacc, pl.acc_cols, pl.smem,
                  ceil_div(s.B, pl.NS * pl.G));
}

// ---- host-side image builder ----------------------------------------------------------------------------------
struct BlockList {
  std::vector<int> cols;
  std::vector<float> w;  // 4 per column
};

static void block_lists(const int32_t* rowptr, const int32_t* col, const float* val, int M, std::vector<BlockList>* out) {
  const int nb = M / 4;
  out->assign(nb, BlockList());
  for (int b = 0; b < nb; ++b) {
    std::vector<int>& c = (*out)[b].cols;
    for (int r = 4 * b; r < 4 * b + 4; ++r) c.insert(c.end(), col + rowptr[r], col + rowptr[r + 1]);
    std::sort(c.begin(), c.end());
    c.erase(std::unique(c.begin(), c.end()), c.end());
    if (val) {
      std::vector<float>& w = (*out)[b].w;
      w.assign(c.size() * 4, 0.f);
      for (int i = 0; i < 4; ++i) {
        const int r = 4 * b + i;
        for (int e = rowptr[r]; e < rowptr[r + 1]; ++e) {
          const size_t at = std::lower_bound(c.begin(), c.end(), col[e]) - c.begin();
          w[at * 4 + i] += val[e];  // duplicate entries of a row (never produced by scipy) add up
        }
      }
    }
  }
}

// blocks by decreasing list length (ties: by index), grouped by four; steps of a group = its longest list, made even
static void group_blocks(const std::vector<BlockList>& bl, std::vector<int>* order, std::vector<int>* steps) {
  const int nb = (int)bl.size();
  order->resize(nb);
  for (int i = 0; i < nb; ++i) (*order)[i] = i;
  std::stable_sort(order->begin(), order->end(), [&](int a, int b) { return bl[a].cols.size() > bl[b].cols.size(); });
  steps->clear();
  for (int g = 0; g * 4 < nb; ++g) steps->push_back((int)((bl[(*order)[g * 4]].cols.size() + 1) & ~(size_t)1));
}

static bool csr_rows_valid(const int32_t* rowptr, const int32_t* col, int M, int nnz) {
  if (!rowptr || !col || rowptr[0] != 0 || rowptr[M] != nnz) return false;
  for (int r = 0; r < M; ++r)
    if (rowptr[r + 1] < rowptr[r]) return false;
  for (int e = 0; e < nnz; ++e)
    if (col[e] < 0 || col[e] >= M) return false;
  return true;
}

static LayerShape adjoint_shape(const LayerShape& s) { return LayerShape{s.B, s.M, s.nnz, s.Fout, s.Fin, s.K, 1}; }

size_t cheb_image_bytes(const int32_t* rowptr, const int32_t* col, const LayerShape& layer, int adjoint) {
  const LayerShape s = adjoint ? adjoint_shape(layer) : layer;
  if (s.M < 4 || (s.M & 3) || !csr_rows_valid(rowptr, col, s.M, s.nnz)) return 0;
  std::vector<BlockList> bl;
  block_lists(rowptr, col, nullptr, s.M, &bl);
  std::vector<int> order, steps;
  group_blocks(bl, &order, &steps);
  long long ent = 0;
  for (int st : steps) ent += (long long)(st / 2) * kImgPair;
  DeviceInfo di;
  plan_device(&di);
  const UmmaFwdPlan pl = plan_umma_fwd(s, di.sm_count, di.smem_optin, ent, adjoint != 0);
  return pl.ok ? pl.img_bytes : 0;
}

int cheb_image_build(const int32_t* rowptr, const int32_t* col, const float* val, const LayerShape& layer, int adjoint,
                     void* out, size_t bytes) {
  const LayerShape s = adjoint ? adjoint_shape(layer) : layer;
  GCNB_REQUIRE(out && val && s.M >= 4 && (s.M & 3) == 0 && csr_rows_valid(rowptr, col, s.M, s.nnz),
               "gcnb_cheb_image_build: needs host CSR arrays of a graph with M %% 4 == 0");
  std::vector<BlockList> bl;
  block_lists(rowptr, col, val, s.M, &bl);
  std::vector<int> order, steps;
  group_blocks(bl, &order, &steps);
  long long ent = 0;
  for (int st : steps) ent += (long long)(st / 2) * kImgPair;
  DeviceInfo di;
  plan_device(&di);
  const UmmaFwdPlan pl = plan_umma_fwd(s, di.sm_count, di.smem_optin, ent, adjoint != 0);
  GCNB_REQUIRE(pl.ok, "gcnb_cheb_image_build: no image-based kernel for this shape");
  GCNB_REQUIRE(bytes == pl.img_bytes, "gcnb_cheb_image_build: buffer has %zu bytes, the image needs %zu", bytes, pl.img_bytes);
  const ImgGeom ge = img_geom(s.M);
  unsigned char* img = static_cast<unsigned char*>(out);
  memset(img, 0, bytes);
  uint32_t* hdr = reinterpret_cast<uint32_t*>(img);
  hdr[0] = kImgMagic;
  hdr[1] = img_signature(s, pl);
  hdr[2] = (uint32_t)bytes;
  hdr[3] = (uint32_t)ge.ng;
  uint32_t* grp = reinterpret_cast<uint32_t*>(img + ge.grp_off);
  uint16_t* blk = reinterpret_cast<uint16_t*>(img + ge.blk_off);
  int log2p = 0;
  while ((1 << log2p) < s.p) ++log2p;
  auto code16 = [](int row) { return (uint16_t)(gather_code(row) >> 4); };  // rows < 2048 (256 KB of descriptors)
  auto code_of = [&](int v) { return code16((v & (s.p - 1)) * pl.BQ + (v >> log2p)); };
  const uint16_t zero_code = code16(s.p * pl.BQ);
  size_t at = ge.ent_off;
  for (int g = 0; g < ge.ng; ++g) {
    grp[g * 2] = (uint32_t)at;
    grp[g * 2 + 1] = (uint32_t)steps[g];
    for (int q = 0; q < 4; ++q) blk[g * 4 + q] = g * 4 + q < ge.nb ? (uint16_t)order[g * 4 + q] : (uint16_t)0xffff;
    for (int j = 0; j < steps[g]; ++j) {
      unsigned char* pair = img + at + (size_t)(j / 2) * kImgPair;
      float* w = reinterpret_cast<float*>(pair + (j & 1) * 64);
      uint16_t* codes = reinterpret_cast<uint16_t*>(pair + 128);
      for (int q = 0; q < 4; ++q) {
        uint16_t code = zero_code;
        if (g * 4 + q < ge.nb) {
          const BlockList& b = bl[order[g * 4 + q]];
          if (j < (int)b.cols.size()) {
            code = code_of(b.cols[j]);
            for (int i = 0; i < 4; ++i) w[q * 4 + i] = b.w[(size_t)j * 4 + i];
          }
        }
        codes[q * 2 + (j & 1)] = code;
      }
    }
    at += (size_t)(steps[g] / 2) * kImgPair;
  }
  return GCNB_OK;
}

struct UmmaAdjoint {
  const float* dy;
  const float* y;
  const uint8_t* argmax;
  int p, relu, dy_is_mean;
  bool raw;             // the RAW instances: output rows of any width, sent to raw row perm[m] (perm nullable)
  const int32_t* perm;
  int M_in;
};

struct UmmaStack {  // a stack of identical layers run back to back on a tile (UmmaFwdParams::nlayers)
  int nlayers;
  const float* const* W;
  const float* const* bias;
  const void* const* tap_images;  // nullable; entries nullable (device pointers, 16-byte aligned)
};

static int umma_launch(const float* x, const int32_t* perm, int M_in, const gcnb_csr& L, const float* W, const float* bias,
                       float* y, uint8_t* argmax, float* y_mean, float* xstack, const LayerShape& s, int bias_mode, int relu,
                       const UmmaAdjoint* adj, cudaStream_t st, const UmmaStack* stack = nullptr) {
  DeviceInfo di;
  int rc = device_info(&di);
  if (rc) return rc;
  const bool img = L.image != nullptr;
  if (img) {
    const size_t fixed = img_geom(s.M).ent_off;
    GCNB_REQUIRE((s.M & 3) == 0 && L.image_bytes >= fixed && (L.image_bytes & 15) == 0 &&
                     (reinterpret_cast<uintptr_t>(L.image) & 15) == 0,
                 "operator image: bad size or alignment");
  }
  const bool raw = adj != nullptr && adj->raw;
  const UmmaFwdPlan pl = img ? plan_umma_fwd(s, di.sm_count, di.smem_optin, (long long)(L.image_bytes - img_geom(s.M).ent_off), raw)
                             : plan_umma_fwd(s, di.sm_count, di.smem_optin, -1, raw);
  if (!pl.ok) {
    set_error(img ? "the operator image does not belong to this layer shape" : "tcgen05 forward does not support this shape");
    return GCNB_ERR_INVALID;
  }
  UmmaFwdParams P{};
  P.x = x; P.perm = perm; P.M_in = M_in;
  P.rowptr = L.rowptr; P.col = L.col; P.val = L.val; P.nnz = L.nnz;
  P.W = W; P.bias = bias; P.y = y; P.argmax = argmax; P.y_mean = y_mean; P.xstack = xstack;
  P.B = s.B; P.M = s.M; P.Fin = s.Fin; P.Fout = s.Fout; P.K = s.K; P.p = s.p; P.bias_mode = bias_mode; P.relu = relu;
  P.log2p = 0;
  while ((1 << P.log2p) < s.p) ++P.log2p;
  P.nlayers = 1;
  P.Wl[0] = W;
  P.biasl[0] = bias;
  if (stack) {
    GCNB_REQUIRE(img && !adj && stack->nlayers >= 1 && stack->nlayers <= 8 && s.p == 1 && s.Fin == 32 && s.Fout == 32 &&
                     xstack == nullptr && y_mean == nullptr,
                 "layer stack: needs an operator image, p = 1, Fin = Fout = 32, 1..8 layers, inference outputs only");
    P.nlayers = stack->nlayers;
    P.tap_bytes = (int)(2 * (size_t)s.K * pl.FP * 32 * 4 + (size_t)s.K * pl.FP * 32 * 2);
    for (int l = 0; l < stack->nlayers; ++l) {
      P.Wl[l] = stack->W[l];
      P.biasl[l] = stack->bias ? stack->bias[l] : nullptr;
      P.tapimg[l] = stack->tap_images ? static_cast<const unsigned char*>(stack->tap_images[l]) : nullptr;
      GCNB_REQUIRE((reinterpret_cast<uintptr_t>(P.tapimg[l]) & 15) == 0, "layer stack: tap image %d is not 16-byte aligned", l);
    }
    GCNB_REQUIRE(pl.off_wl == pl.off_wh + (int)((size_t)s.K * pl.FP * 32 * 4) && pl.off_wb == pl.off_wl + (pl.off_wl - pl.off_wh) &&
                     (pl.off_wh & 15) == 0, "layer stack: tap arrays are not contiguous");
    P.W = P.Wl[0];
    P.bias = P.biasl[stack->nlayers - 1];
  }
  if (adj) {
    P.adj = 1;
    P.adj_dy = adj->dy; P.adj_y = adj->y; P.adj_arg = adj->argmax;
    P.adj_relu = adj->relu; P.adj_mean = adj->dy_is_mean;
    P.adj_log2p = 0;
    while ((1 << P.adj_log2p) < adj->p) ++P.adj_log2p;
    P.adj_Mo = s.M >> P.adj_log2p;
    if (raw) {  // the prologue's source-row table becomes the destination-row table of the epilogue
      P.perm = adj->perm;
      P.M_in = adj->M_in;
    }
  }
  P.NS = pl.NS; P.S = pl.NS * pl.G; P.Q = pl.Q; P.BQ = pl.BQ; P.T = pl.T; P.NG = pl.NG; P.nlo = pl.nlo; P.nacc = pl.nacc;
  P.acc_cols = pl.acc_cols; P.tmem_cols = pl.tmem_cols; P.slab_rows = pl.slab_rows;
  P.ntiles = ceil_div(s.B, P.S);
  P.off_lo = pl.off_lo; P.off_wh = pl.off_wh; P.off_wl = pl.off_wl; P.off_wb = pl.off_wb; P.off_ent = pl.off_ent;
  P.off_grow = pl.off_grow; P.off_grho = pl.off_grho; P.off_gslot = pl.off_gslot; P.off_glen = pl.off_glen;
  P.off_src = pl.off_src; P.off_rlen = pl.off_rlen; P.off_sorted = pl.off_sorted; P.off_bias = pl.off_bias;
  P.off_bar = pl.off_bar; P.off_rp = pl.off_rp;
  if (img) {
    const ImgGeom ge = img_geom(s.M);
    P.image = static_cast<const unsigned char*>(L.image);
    P.img_bytes = (int)pl.img_bytes;
    P.img_sig = img_signature(s, pl);
    P.n_groups = ge.ng;
    P.off_img = pl.off_img; P.off_grp = pl.off_img + (int)ge.grp_off; P.off_blk = pl.off_img + (int)ge.blk_off;
    // bulk copies need 16-byte aligned windows; the staged tile lies inside one state buffer, clear of its zero row
    const size_t wbytes = (size_t)M_in * s.Fin * 4;
    P.stage = !adj && (reinterpret_cast<uintptr_t>(x) & 15) == 0 && (wbytes & 15) == 0 &&
              (size_t)P.S * wbytes <= (size_t)s.p * pl.BQ * 128;
  }
#ifdef GCNB_TRACE
  P.debug = std::getenv("GCNB_UMMA_DEBUG") ? std::atoi(std::getenv("GCNB_UMMA_DEBUG")) : 0;
#endif
  const int grid = std::min(P.ntiles, di.sm_count);
#define GCNB_UMMA_CASE(fp, mi, im, stk, rw)                                                                             \
  if (pl.FP == fp && pl.MAXI == mi && img == im && (P.nlayers > 1) == stk && raw == rw) {                               \
    GCNB_CUDA(cudaFuncSetAttribute(k_cheb_fwd_umma<fp, mi, im, stk, rw>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.smem)); \
    k_cheb_fwd_umma<fp, mi, im, stk, rw><<<grid, kThreads, pl.smem, st>>>(P);                                          \
  }
  GCNB_UMMA_CASE(16, 3, false, false, false) GCNB_UMMA_CASE(16, 5, false, false, false)
  GCNB_UMMA_CASE(32, 3, false, false, false) GCNB_UMMA_CASE(32, 5, false, false, false)
  GCNB_UMMA_CASE(16, 1, true, false, false) GCNB_UMMA_CASE(32, 1, true, false, false)
  GCNB_UMMA_CASE(32, 1, true, true, false)
  GCNB_UMMA_CASE(16, 3, false, false, true) GCNB_UMMA_CASE(16, 5, false, false, true)
  GCNB_UMMA_CASE(32, 3, false, false, true) GCNB_UMMA_CASE(32, 5, false, false, true)
  GCNB_UMMA_CASE(16, 1, true, false, true) GCNB_UMMA_CASE(32, 1, true, false, true)
#undef GCNB_UMMA_CASE
  GCNB_LAUNCH_CHECK("k_cheb_fwd_umma");
  return GCNB_OK;
}

int umma_cheb_fwd(const float* x, const int32_t* perm, int M_in, const gcnb_csr& L, const float* W, const float* bias,
                  float* y, uint8_t* argmax, float* y_mean, float* xstack, const LayerShape& s, int bias_mode, int relu,
                  cudaStream_t st) {
  return umma_launch(x, perm, M_in, L, W, bias, y, argmax, y_mean, xstack, s, bias_mode, relu, nullptr, st);
}

// A stack of `nlayers` identical layers (same operator, p = 1, 32 -> 32 filters, same K / bias mode / ReLU) in ONE launch:
// activations stay in shared memory / TMEM between the layers (the production network of model.py:271-274 is six such
// layers).  Needs the operator image of the layer shape.
bool umma_stack_supported(const LayerShape& s, const gcnb_csr& L) {
  if (L.image == nullptr || s.p != 1 || s.Fin != 32 || s.Fout != 32 || (s.M & 3)) return false;
  if (L.image_bytes < img_geom(s.M).ent_off) return false;
  DeviceInfo di;
  plan_device(&di);
  return plan_umma_fwd(s, di.sm_count, di.smem_optin, (long long)(L.image_bytes - img_geom(s.M).ent_off)).ok;
}

// ---- pre-split tap images (host side) ----------------------------------------------------------------------------
// The kernel's tap split, bit for bit: cvt.rna.tf32.f32 = round to nearest, ties away from zero, to a 10-bit mantissa;
// the bf16 image is round-to-nearest-even of the fp32 weight.
static inline uint32_t f2u(float f) { uint32_t u; memcpy(&u, &f, 4); return u; }
static inline float u2f(uint32_t u) { float f; memcpy(&f, &u, 4); return f; }
static inline float host_tf32_rna(float x) { return u2f((f2u(x) + 0x1000u) & 0xffffe000u); }
static inline uint16_t host_bf16_rn(float x) {
  const uint32_t u = f2u(x);
  return (uint16_t)((u + 0x7fffu + ((u >> 16) & 1u)) >> 16);
}

size_t cheb_tap_image_bytes(int Fin, int Fout, int K) {
  if (Fin <= 8 || Fin > 32 || Fout < 4 || Fout > 32 || (Fout & 3) || K < 1) return 0;
  const size_t FP = Fin <= 16 ? 16 : 32;
  return 2 * (size_t)K * FP * 32 * 4 + (size_t)K * FP * 32 * 2;
}

int cheb_tap_image_build(const float* W, int Fin, int Fout, int K, void* out, size_t bytes) {
  GCNB_REQUIRE(W && out && bytes != 0 && bytes == cheb_tap_image_bytes(Fin, Fout, K),
               "gcnb_cheb_tap_image_build: bad arguments or buffer size");
  const int FP = Fin <= 16 ? 16 : 32;
  const size_t taps = (size_t)K * FP * 32 * 4;
  unsigned char* img = static_cast<unsigned char*>(out);
  memset(img, 0, bytes);
  for (int kk = 0; kk < K * FP; ++kk) {
    const int k = kk / FP, f = kk - k * FP;
    for (int o = 0; o < 32; ++o) {
      const float w = (f < Fin && o < Fout) ? W[((size_t)f * K + k) * Fout + o] : 0.f;
      const float hi = host_tf32_rna(w), lo = host_tf32_rna(w - hi);
      memcpy(img + tap_off_tf32(kk, o), &hi, 4);
      memcpy(img + taps + tap_off_tf32(kk, o), &lo, 4);
      const uint16_t b = host_bf16_rn(w);
      memcpy(img + 2 * taps + tap_off_bf16(kk, o), &b, 2);
    }
  }
  return GCNB_OK;
}

int umma_cheb_stack_fwd(const float* x, const gcnb_csr& L, const float* const* W, const float* const* bias,
                        const void* const* tap_images, float* y, int nlayers, const LayerShape& s, int bias_mode, int relu,
                        cudaStream_t st) {
  UmmaStack stk{nlayers, W, bias, tap_images};
  return umma_launch(x, nullptr, s.M, L, W[0], bias ? bias[nlayers - 1] : nullptr, y, nullptr, nullptr, nullptr, s, bias_mode,
                     relu, nullptr, st, &stk);
}

// The layer's input gradient through the forward kernel: operator L~^T, taps W_k^T, input dZ (see UmmaFwdParams::adj).
bool umma_adj_supported(const LayerShape& s) {
  if ((s.Fout & 3) || (s.Fin & 3) || s.M % s.p != 0 || s.p > 255) return false;
  return umma_fwd_supported(adjoint_shape(s));
}

int umma_cheb_adj(const float* dy, int dy_is_mean, const float* y, const uint8_t* argmax, const gcnb_csr& Lt, const float* W,
                  float* dx, const LayerShape& s, int relu, cudaStream_t st) {
  UmmaAdjoint a{dy, y, argmax, s.p, relu, dy_is_mean, false, nullptr, s.M};
  return umma_launch(nullptr, nullptr, s.M, Lt, W, nullptr, dx, nullptr, nullptr, nullptr, adjoint_shape(s), GCNB_BIAS_NONE, 0,
                     &a, st);
}

// The same for any input width Fin in [4, 32] (the RAW instances); the layer's Fout must still be a multiple of 4 (dZ is
// rebuilt from dy / y / arg-max with 16-byte loads).
bool umma_adj_raw_supported(const LayerShape& s) {
  if ((s.Fout & 3) || s.M % s.p != 0 || s.p > 255) return false;
  DeviceInfo di;
  plan_device(&di);
  return plan_umma_fwd(adjoint_shape(s), di.sm_count, di.smem_optin, -1, true).ok;
}

int umma_adj_describe(const LayerShape& s, char* out, size_t n) {
  DeviceInfo di;
  plan_device(&di);
  const UmmaFwdPlan pl = plan_umma_fwd(adjoint_shape(s), di.sm_count, di.smem_optin, -1, true);
  if (!pl.ok) return 0;
  return snprintf(out, n, "k_cheb_fwd_umma<FP=%d, RAW> on L~^T, MMA N=%d, %d windows/tile, %zu B smem, %d tiles", pl.FP,
                  s.Fin <= 16 ? 16 : 32, pl.NS * pl.G, pl.smem, ceil_div(s.B, pl.NS * pl.G));
}

int umma_cheb_adj_raw(const float* dy, int dy_is_mean, const float* y, const uint8_t* argmax, const gcnb_csr& Lt,
                      const float* W, float* dx, const int32_t* perm, int M_in, const LayerShape& s, int relu, cudaStream_t st) {
  UmmaAdjoint a{dy, y, argmax, s.p, relu, dy_is_mean, true, perm, M_in};
  return umma_launch(nullptr, nullptr, s.M, Lt, W, nullptr, dx, nullptr, nullptr, nullptr, adjoint_shape(s), GCNB_BIAS_NONE, 0,
                     &a, st);
}

}  // namespace gcnb

#ifdef GCNB_TRACE
extern "C" __attribute__((visibility("default"))) int gcnb_debug_read_trace(long long* out) {
  return (int)cudaMemcpyFromSymbol(out, gcnb::g_trace, sizeof(long long) * 4 * 512);
}
#endif
