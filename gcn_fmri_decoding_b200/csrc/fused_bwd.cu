// Fused ChebyNet backward for graphs that fit in shared memory (what tf.gradients builds for
// chebyshev5 + b1relu/b2relu + mpool1, models_gcn.py:298-303; SURVEY.md A.2).
//
// Per tile of S windows, one CTA
//   1. rebuilds dZ (MaxPoolGrad o ReluGrad of dy, from y and the arg-max bytes) in shared memory,
//   2. recomputes the Chebyshev basis X_k = T_k(L~) x order by order (same sparse step as the forward) and
//      contracts it against dZ on the tensor cores: dW_k[f][o] += sum_rows X_k[row][f] dZ[row][o]
//      (3xTF32 mma.sync; X_k^T is the A operand straight out of the slab),
//   3. if dx is wanted, forms G_k = dZ W_k^T on the tensor cores and runs the adjoint recursion in
//      Clenshaw form with the transposed operator:  b_k = G_k + 2 L~^T b_{k+1} - b_{k+2},
//      dx = G_0 + L~^T b_1 - b_2  (K-1 sparse steps, no G stack).
// Nothing but x, y, arg-max and dy is read from HBM and only dx is written; dW is reduced without float
// atomics: warps -> CTA through a shared-memory scratch (fixed order), CTAs -> a small second kernel.
// The bias gradient is a separate two-stage column sum over the pooled tensors (also fixed order).
#include <algorithm>
#include <cmath>

#include "fused_common.cuh"

namespace gcnb {

struct BwdParams {
  const float* x;
  const int32_t* perm;
  int M_in;
  const float* y;
  const uint8_t* argmax;
  const float* dy;
  const int32_t *rowptr, *col;
  const float* val;
  const int32_t *rowptr_t, *col_t;
  const float* val_t;
  int nnz;
  const float* W;
  float* dx;       // nullable
  float* dw_part;  // [grid][K][chunks][256]
  float* db_part;  // [grid][FoP] per-filter bias-gradient partials (nullable)
  int B, Fin, Fout, K, p, log2p, relu;
  int skip_dw;     // the weight/bias gradients come from the saved basis (stack_dw.cu): only dx is computed here
  int dy_is_mean;  // dy is [B][M/p]: the gradient of the mean over filters (every filter gets dy/Fout)
  TileGeom g;      // FP/KS/RS describe the X slabs
  int FoP, RSz;    // padded Fout, dZ slab stride
  int ntiles;
  int nchunks;     // MT*NT/2 accumulator chunks of 256 floats
  int off_opT, off_wfragT, off_dws, off_scratch, off_dz, off_slab;
};

// MT = FP/16 (1 or 2) m-tiles over the input features, NT = FoP/8 n-tiles over the filters.
template <int MT, int NT, int SLOTS>
__global__ void __launch_bounds__(896, 1) k_cheb_bwd_fused(const BwdParams P) {
  extern __shared__ __align__(16) unsigned char smem[];
  const TileGeom& G = P.g;
  OperatorSmem opL, opT;
  opL.carve(smem, G.Mpad, P.nnz);
  opT.carve(smem + P.off_opT, G.Mpad, P.nnz);
  float4* wfragT = reinterpret_cast<float4*>(smem + P.off_wfragT);
  float* dWs = reinterpret_cast<float*>(smem + P.off_dws);
  float* scratch = reinterpret_cast<float*>(smem + P.off_scratch);
  float* dZ = reinterpret_cast<float*>(smem + P.off_dz);
  unsigned char* slabA = smem + P.off_slab;
  unsigned char* slabB = slabA + (size_t)G.Mpad * G.RS * 4;

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int g = lane >> 2, t = lane & 3;
  const int rw = warp % G.RW, sg = warp / G.RW;
  const int RS = G.RS, FP = G.FP, RSz = P.RSz, FoP = P.FoP;
  const int nwarps = blockDim.x >> 5;
  const bool need_dx = P.dx != nullptr;
  constexpr int NTF = MT * 2;  // n-tiles over the input features in the G contraction
  constexpr int NCH = MT * NT / 2;

  // ---- once per CTA ---------------------------------------------------------------------------------------------
  if (!P.skip_dw) build_operator(P.rowptr, P.col, P.val, G.M, G.Mpad, P.nnz, RS, opL);
  if (need_dx && P.K > 1) build_operator(P.rowptr_t, P.col_t, P.val_t, G.M, G.Mpad, P.nnz, RS, opT);
  if (need_dx) {
    // B fragments of W_k^T (k8 = filters o, n8 = input features f), TF32 hi/lo
    const int KSo = FoP / 8;
    for (int idx = tid; idx < P.K * KSo * NTF * 32; idx += blockDim.x) {
      const int ln = idx & 31, ntf = (idx >> 5) % NTF, ks = (idx / (32 * NTF)) % KSo, k = idx / (32 * NTF * KSo);
      const int gg = ln >> 2, tt = ln & 3;
      const int f = ntf * 8 + gg, o0 = ks * 8 + tt, o1 = o0 + 4;
      float w0 = 0.f, w1 = 0.f;
      if (f < P.Fin) {
        if (o0 < P.Fout) w0 = __ldg(P.W + ((long long)f * P.K + k) * P.Fout + o0);
        if (o1 < P.Fout) w1 = __ldg(P.W + ((long long)f * P.K + k) * P.Fout + o1);
      }
      uint32_t h0, l0, h1, l1;
      split_tf32(w0, h0, l0);
      split_tf32(w1, h1, l1);
      wfragT[idx] = make_float4(__uint_as_float(h0), __uint_as_float(h1), __uint_as_float(l0), __uint_as_float(l1));
    }
  }
  for (int i = tid; i < P.K * NCH * 256; i += blockDim.x) dWs[i] = 0.f;

  const int col_byte = sg * G.WS * FP * 4;
  const int Mo = G.M >> P.log2p;
  const int fp_shift = FP == 8 ? 3 : (FP == 16 ? 4 : 5);
  const int lrow = lane >> fp_shift, lf = lane & (FP - 1), rows_per_instr = 32 >> fp_shift;
  const int per_sample = P.M_in * P.Fin;

  float dbacc = 0.f;  // this thread's filter (o = tid % FoP is the same in every iteration: FoP | blockDim)

  for (int tile = blockIdx.x; tile < P.ntiles; tile += gridDim.x) {
    const int b0 = tile * G.S;
    __syncthreads();
    // ---- x -> slab A;  dZ slab from (dy, y, arg-max) ---------------------------------------------------------
    for (int s = 0; s < (P.skip_dw ? 0 : G.S); ++s) {
      const int b = b0 + s;
      const float* xb = P.x + (long long)b * per_sample;
      for (int m = warp * rows_per_instr + lrow; m < G.Mpad; m += nwarps * rows_per_instr) {
        float v = 0.f;
        if (b < P.B && m < G.M && lf < P.Fin) {
          const int src = P.perm ? __ldg(P.perm + m) : m;
          if (src < P.M_in) v = __ldg(xb + (long long)src * P.Fin + lf);
        }
        reinterpret_cast<float*>(slabA)[m * RS + s * FP + lf] = v;
      }
    }
    {
      // pooled elements (s, j, o) of the tile, o fastest (coalesced); padded filters and rows are zeroed
      const int MoP = G.Mpad >> P.log2p;
      const int fo_shift = FoP == 16 ? 4 : 5;
      const int o = tid & (FoP - 1);
      for (int rj = tid >> fo_shift; rj < G.S * MoP; rj += blockDim.x >> fo_shift) {
        const int s = rj / MoP, j = rj - s * MoP;
        const int b = b0 + s;
        float gval = 0.f;
        int am = 0;
        if (b < P.B && j < Mo && o < P.Fout) {
          const long long gi = ((long long)b * Mo + j) * P.Fout + o;
          gval = P.dy_is_mean ? __ldg(P.dy + (long long)b * Mo + j) / (float)P.Fout : __ldg(P.dy + gi);
          if (P.relu && !(__ldg(P.y + gi) > 0.f)) gval = 0.f;
          if (P.argmax != nullptr && P.p > 1) am = __ldg(P.argmax + gi);
        }
        dbacc += gval;
        float* dst = dZ + (size_t)(j << P.log2p) * RSz + s * FoP + o;
        for (int i = 0; i < P.p; ++i) dst[(size_t)i * RSz] = (i == am) ? gval : 0.f;
      }
    }
    __syncthreads();

    // ---- phase A: X_k order by order, dW_k += X_k^T dZ ---------------------------------------------------------
    for (int k = 0; k < (P.skip_dw ? 0 : P.K); ++k) {
      unsigned char* cur = (k & 1) ? slabB : slabA;
      if (k > 0) {
        const unsigned char* src = (k & 1) ? slabA : slabB;
        spmm_dispatch(G.LPR, opL, src, cur, G.Mpad, col_byte, rw, G.RW, k == 1 ? 1.f : 2.f, k > 1);
        __syncthreads();
      }
      float acc[MT][NT][4];
#pragma unroll
      for (int m = 0; m < MT; ++m)
#pragma unroll
        for (int n = 0; n < NT; ++n)
#pragma unroll
          for (int c = 0; c < 4; ++c) acc[m][n][c] = 0.f;
      const float* curf = reinterpret_cast<const float*>(cur);
#pragma unroll
      for (int a = 0; a < SLOTS; ++a) {
        const int tt = a / G.WS, s = a - tt * G.WS;
        const int rt = rw + tt * G.RW;
        if (!(a < G.TPW * G.WS && rt < G.RT)) continue;
        const int scol = (sg * G.WS + s);
#pragma unroll
        for (int h2 = 0; h2 < 2; ++h2) {
          const int r = rt * 16 + h2 * 8 + t;  // rows r and r+4 of this 8-row step
          uint32_t bh[NT][2], bl[NT][2];
          const float* zr = dZ + (size_t)r * RSz + scol * FoP + g;
#pragma unroll
          for (int n = 0; n < NT; ++n) {
            split_trunc(zr[n * 8], bh[n][0], bl[n][0]);
            split_trunc(zr[n * 8 + 4 * RSz], bh[n][1], bl[n][1]);
          }
          const float* xr = curf + (size_t)r * RS + scol * FP + g;
#pragma unroll
          for (int m = 0; m < MT; ++m) {
            uint32_t ah[4], al[4];
            const bool hi_ok = (m * 16 + g + 8) < FP;  // FP = 8: features 8..15 do not exist
            split_trunc(xr[m * 16], ah[0], al[0]);
            split_trunc(hi_ok ? xr[m * 16 + 8] : 0.f, ah[1], al[1]);
            split_trunc(xr[m * 16 + 4 * RS], ah[2], al[2]);
            split_trunc(hi_ok ? xr[m * 16 + 8 + 4 * RS] : 0.f, ah[3], al[3]);
#pragma unroll
            for (int n = 0; n < NT; ++n) mma_3xtf32(acc[m][n], ah, al, bh[n][0], bh[n][1], bl[n][0], bl[n][1]);
          }
        }
      }
      // ---- warps -> CTA: fixed-order reduction through the scratch, two n-tiles (256 floats) per round --------
#pragma unroll
      for (int m = 0; m < MT; ++m) {
#pragma unroll
        for (int np = 0; np < NT / 2; ++np) {
          float* mine = scratch + (size_t)warp * 256 + lane;
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            mine[c * 32] = acc[m][2 * np][c];
            mine[(4 + c) * 32] = acc[m][2 * np + 1][c];
          }
          __syncthreads();
          for (int e = tid; e < 256; e += blockDim.x) {
            // fixed association, four independent chains (the loads are independent, only the adds chain)
            float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
            int w = 0;
            for (; w + 4 <= nwarps; w += 4) {
              s0 += scratch[w * 256 + e];
              s1 += scratch[(w + 1) * 256 + e];
              s2 += scratch[(w + 2) * 256 + e];
              s3 += scratch[(w + 3) * 256 + e];
            }
            for (; w < nwarps; ++w) s0 += scratch[w * 256 + e];
            dWs[((size_t)k * NCH + m * (NT / 2) + np) * 256 + e] += (s0 + s1) + (s2 + s3);
          }
          __syncthreads();
        }
      }
    }

    // ---- phase B: dx by the Clenshaw form of the adjoint recursion ---------------------------------------------
    if (need_dx) {
      const int KSo = FoP / 8;
      for (int k = P.K - 1; k >= 0; --k) {
        const int step = P.K - 1 - k;                       // 0, 1, 2, ...
        unsigned char* cur = (step & 1) ? slabB : slabA;    // b_k lands here (it holds b_{k+2})
        if (step > 0) {
          const unsigned char* src = (step & 1) ? slabA : slabB;  // b_{k+1}
          spmm_dispatch(G.LPR, opT, src, cur, G.Mpad, col_byte, rw, G.RW, k == 0 ? 1.f : 2.f, step > 1);
        }
        // G_k = dZ W_k^T for the warp's own row tiles (independent of the sparse step above)
        float gacc[SLOTS][NTF][4];
#pragma unroll
        for (int a = 0; a < SLOTS; ++a)
#pragma unroll
          for (int n = 0; n < NTF; ++n)
#pragma unroll
            for (int c = 0; c < 4; ++c) gacc[a][n][c] = 0.f;
        const float4* wk = wfragT + (size_t)k * KSo * NTF * 32 + lane;
        for (int ks = 0; ks < KSo; ++ks) {
          uint32_t ah[SLOTS][4], al[SLOTS][4];
#pragma unroll
          for (int a = 0; a < SLOTS; ++a) {
            const int tt = a / G.WS, s = a - tt * G.WS;
            const int rt = rw + tt * G.RW;
            if (a < G.TPW * G.WS && rt < G.RT) {
              const float* base = dZ + (size_t)(rt * 16 + g) * RSz + (sg * G.WS + s) * FoP + ks * 8 + t;
              split_trunc(base[0], ah[a][0], al[a][0]);
              split_trunc(base[8 * RSz], ah[a][1], al[a][1]);
              split_trunc(base[4], ah[a][2], al[a][2]);
              split_trunc(base[8 * RSz + 4], ah[a][3], al[a][3]);
            } else {
#pragma unroll
              for (int c = 0; c < 4; ++c) ah[a][c] = al[a][c] = 0u;
            }
          }
#pragma unroll
          for (int n = 0; n < NTF; ++n) {
            const float4 w = wk[(ks * NTF + n) * 32];
#pragma unroll
            for (int a = 0; a < SLOTS; ++a)
              mma_3xtf32(gacc[a][n], ah[a], al[a], __float_as_uint(w.x), __float_as_uint(w.y), __float_as_uint(w.z),
                         __float_as_uint(w.w));
          }
        }
        group_barrier(sg, G.RW * 32);  // sparse step complete for every row of this sample group's columns
        float* curf = reinterpret_cast<float*>(cur);
#pragma unroll
        for (int a = 0; a < SLOTS; ++a) {
          const int tt = a / G.WS, s = a - tt * G.WS;
          const int rt = rw + tt * G.RW;
          if (!(a < G.TPW * G.WS && rt < G.RT)) continue;
#pragma unroll
          for (int n = 0; n < NTF; ++n) {
            if (n * 8 >= FP) continue;
#pragma unroll
            for (int h = 0; h < 2; ++h) {
              float2* pz = reinterpret_cast<float2*>(curf + (size_t)(rt * 16 + g + 8 * h) * RS + (sg * G.WS + s) * FP +
                                                     n * 8 + 2 * t);
              float2 v = make_float2(gacc[a][n][2 * h], gacc[a][n][2 * h + 1]);
              if (step > 0) {
                const float2 o = *pz;
                v.x += o.x;
                v.y += o.y;
              }
              *pz = v;
            }
          }
        }
        group_barrier(sg, G.RW * 32);
      }
      __syncthreads();
      // dx rows of the tile: the slab that received b_0
      const float* fin = reinterpret_cast<const float*>(((P.K - 1) & 1) ? slabB : slabA);
      for (int s = 0; s < G.S; ++s) {
        const int b = b0 + s;
        if (b >= P.B) break;
        float* dxb = P.dx + (long long)b * G.M * P.Fin;
        for (int m = warp * rows_per_instr + lrow; m < G.M; m += nwarps * rows_per_instr)
          if (lf < P.Fin) dxb[(long long)m * P.Fin + lf] = fin[m * RS + s * FP + lf];
      }
    }
  }
  __syncthreads();
  if (P.skip_dw) return;
  float* out = P.dw_part + (size_t)blockIdx.x * P.K * NCH * 256;
  for (int i = tid; i < P.K * NCH * 256; i += blockDim.x) out[i] = dWs[i];
  if (P.db_part != nullptr) {  // per-filter bias gradient of this CTA: threads -> filters in fixed order
    scratch[tid] = dbacc;
    __syncthreads();
    if (tid < FoP) {
      float sum = 0.f;
      for (int i = tid; i < (int)blockDim.x; i += FoP) sum += scratch[i];
      P.db_part[(size_t)blockIdx.x * FoP + tid] = sum;
    }
  }
}

// dW[(f*K + k)*Fout + o] = sum over CTAs of the chunked partials (and, in the trailing columns, the per-filter
// bias-gradient partials).  A CTA owns 32 consecutive elements: lane = element, so every load of a warp is one
// coalesced 128-byte line; its 8 warps split the CTAs' partials (many independent loads in flight per thread) and
// are combined through shared memory in warp order -- a fixed summation order, bit-reproducible.
__global__ void __launch_bounds__(256) k_dw_from_partials(const float* __restrict__ part, float* __restrict__ dW,
                                                           int nblocks, int K, int MT, int NT, int Fin, int Fout,
                                                           const float* __restrict__ db_part, float* __restrict__ db,
                                                           int FoP) {
  __shared__ float red[8][32];
  const int NCH = MT * NT / 2;
  const int total = K * NCH * 256;
  const int ntot = total + (db_part != nullptr ? Fout : 0);
  const int lane = threadIdx.x & 31, wp = threadIdx.x >> 5;
  const int w = blockIdx.x * 32 + lane;
  float s = 0.f;
  if (w < ntot) {
    const float* src = w < total ? part + w : db_part + (w - total);
    const size_t stride = w < total ? (size_t)total : (size_t)FoP;
    const int per = (nblocks + 7) >> 3, b0 = wp * per, b1 = min(nblocks, b0 + per);
    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
    int b = b0;
#pragma unroll 4
    for (; b + 3 < b1; b += 4) {
      a0 += src[(size_t)b * stride];
      a1 += src[(size_t)(b + 1) * stride];
      a2 += src[(size_t)(b + 2) * stride];
      a3 += src[(size_t)(b + 3) * stride];
    }
    for (; b < b1; ++b) a0 += src[(size_t)b * stride];
    s = (a0 + a1) + (a2 + a3);
  }
  red[wp][lane] = s;
  __syncthreads();
  if (wp != 0 || w >= ntot) return;
  s = red[0][lane];
#pragma unroll
  for (int i = 1; i < 8; ++i) s += red[i][lane];
  if (w < total) {
    const int e = w & 255, chunk = (w >> 8) % NCH, k = w / (256 * NCH);
    const int m = chunk / (NT / 2), np = chunk % (NT / 2);
    const int reg = e >> 5, ln = e & 31, gg = ln >> 2, tt = ln & 3;
    const int n = 2 * np + (reg >> 2), c = reg & 3;
    const int f = m * 16 + gg + ((c & 2) ? 8 : 0), o = n * 8 + 2 * tt + (c & 1);
    if (f < Fin && o < Fout) dW[((size_t)f * K + k) * Fout + o] = s;
  } else {
    db[w - total] = s;
  }
}

// bias gradient, stage 1: part[chunk][m][o] = sum over the samples of the chunk of dZ[b][m][o]
__global__ void k_db_partial(const float* __restrict__ dy, const float* __restrict__ y, const uint8_t* __restrict__ argmax,
                             float* __restrict__ part, int B, int M, int Fout, int p, int log2p, int relu, int bchunk,
                             int dy_is_mean) {
  const int Mo = M >> log2p;
  const int e = blockIdx.x * blockDim.x + threadIdx.x;  // pooled element (j, o)
  if (e >= Mo * Fout) return;
  const int o = e % Fout, j = e / Fout;
  const int blo = blockIdx.y * bchunk, bhi = min(B, blo + bchunk);
  float acc[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) acc[i] = 0.f;
  for (int b = blo; b < bhi; ++b) {
    const long long gi = ((long long)b * Mo + j) * Fout + o;
    float g = dy_is_mean ? __ldg(dy + (long long)b * Mo + j) / (float)Fout : __ldg(dy + gi);
    if (relu && !(__ldg(y + gi) > 0.f)) g = 0.f;
    const int am = (argmax != nullptr && p > 1) ? __ldg(argmax + gi) : 0;
#pragma unroll
    for (int i = 0; i < 16; ++i) acc[i] += (i == am) ? g : 0.f;
  }
  float* dst = part + ((size_t)blockIdx.y * M + ((size_t)j << log2p)) * Fout + o;
#pragma unroll
  for (int i = 0; i < 16; ++i)
    if (i < p) dst[(size_t)i * Fout] = acc[i];
}

// stage 2: PER_VERTEX: db[m][o] = sum_chunks part;  PER_FILTER: db[o] = sum_chunks sum_m part (one warp per filter,
// lanes stride over (chunk, m), fixed-order shuffle tree)
__global__ void k_db_final(const float* __restrict__ part, float* __restrict__ db, int nchunks, int M, int Fout,
                           int per_vertex) {
  if (per_vertex) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= M * Fout) return;
    float s = 0.f;
    for (int c = 0; c < nchunks; ++c) s += part[(size_t)c * M * Fout + i];
    db[i] = s;
  } else {
    const int o = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (o >= Fout) return;
    float s = 0.f;
    for (int r = lane; r < nchunks * M; r += 32) s += part[(size_t)r * Fout + o];
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) s += __shfl_xor_sync(0xffffffffu, s, d);
    if (lane == 0) db[o] = s;
  }
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
static const size_t kSmemBudgetBwd = 225 * 1024;
static const int kDbChunks = 64;

struct BwdPlan {
  bool ok;
  TileGeom g;
  int MT, NT, SLOTS, FoP, RSz, nchunks;
  size_t smem;
  int off_opT, off_wfragT, off_dws, off_scratch, off_dz, off_slab;
};

static BwdPlan plan_bwd(const LayerShape& s, bool need_dx) {
  BwdPlan pl;
  pl.ok = false;
  TileGeom& g = pl.g;
  if (s.Fin < 1 || s.Fin > 32 || s.Fout < 1 || s.Fout > 32) return pl;
  if (s.p > 16 || s.M % s.p != 0) return pl;
  g.M = s.M;
  g.Mpad = round_up(s.M, 16);
  g.RT = g.Mpad / 16;
  g.FP = s.Fin <= 8 ? 8 : (s.Fin <= 16 ? 16 : 32);
  g.KS = g.FP / 8;
  pl.MT = g.FP <= 16 ? 1 : 2;
  pl.FoP = s.Fout <= 16 ? 16 : 32;
  pl.NT = pl.FoP / 8;
  pl.nchunks = pl.MT * pl.NT / 2;
  const size_t op_bytes = operator_smem_bytes(g.Mpad, s.nnz);
  const size_t wfragT = need_dx ? (size_t)s.K * (pl.FoP / 8) * (pl.MT * 2) * 32 * 16 : 0;
  const size_t dws = (size_t)s.K * pl.nchunks * 256 * 4;
  double best = -1;
  for (int S = 1; S <= 8; S *= 2) {
    if (S > s.B && S > 1) continue;
    for (int ws = 1; ws <= S; ws *= 2) {
      const int cw = ws * g.FP;
      if (cw > 128) continue;
      const int sgn = S / ws;
      int rwn = std::min(g.RT, 28 / sgn);
      if (rwn < 1) continue;
      const int tpw = ceil_div(g.RT, rwn);
      rwn = ceil_div(g.RT, tpw);
      const int slots = tpw * ws;
      if (slots > 4) continue;
      const int SL = slots <= 1 ? 1 : (slots <= 2 ? 2 : 4);
      // registers: phase A holds MT*NT accumulators, phase B SLOTS*MT*2; keep both <= 8 fragments
      // the instance table below has no <MT=2, *, SLOTS=4> kernel: reject it whether or not dx is wanted, so that
      // fused_bwd_supported() implies an existing instance
      if (pl.MT * pl.NT > 8 || SL * pl.MT * 2 > 8) continue;
      const int nw = rwn * sgn;
      // slab strides: RS/8 odd keeps the transposed fragment loads of the dW contraction conflict free
      int RS = S * g.FP + 8;
      if ((RS / 8) % 2 == 0) RS += 8;
      if (S * g.FP == 16) RS = 16;  // 64-byte rows: alternate bank halves in the sparse step (measured best)
      int RSz = S * pl.FoP + 8;
      if ((RSz / 8) % 2 == 0) RSz += 8;
      const size_t need = op_bytes * ((need_dx && s.K > 1) ? 2 : 1) + wfragT + dws + (size_t)nw * 256 * 4 +
                          (size_t)g.Mpad * RSz * 4 + 2 * (size_t)g.Mpad * RS * 4 + 64;
      if (need > kSmemBudgetBwd) continue;
      const double cw32 = cw / 32.0;
      const double wf = (1.0 + cw32) / cw32;
      const double occ = std::min(1.0, nw / 12.0);
      const int tiles = ceil_div(s.B, S);
      const double eff = tiles / (std::ceil(tiles / 148.0) * 148.0);
      const double amort = 1.0 - 0.15 / S;  // per-tile fixed costs (barriers, reductions) amortise with S
      const double score = occ * std::max(eff, 0.05) * amort / wf;
      if (score > best) {
        best = score;
        g.WS = ws; g.SG = sgn; g.S = S; g.RS = RS; g.RW = rwn; g.TPW = tpw; g.nwarps = nw; g.LPR = cw / 4;
        pl.SLOTS = SL; pl.RSz = RSz; pl.smem = need;
      }
    }
  }
  if (best < 0) return pl;
  size_t off = op_bytes;
  pl.off_opT = (int)off;
  if (need_dx && s.K > 1) off += op_bytes;
  pl.off_wfragT = (int)off; off += wfragT;
  pl.off_dws = (int)off; off += dws;
  pl.off_scratch = (int)off; off += (size_t)g.nwarps * 256 * 4;
  pl.off_dz = (int)off; off += (size_t)g.Mpad * pl.RSz * 4;
  off = align_up(off, 16);
  pl.off_slab = (int)off; off += 2 * (size_t)g.Mpad * g.RS * 4;
  pl.smem = off;
  pl.ok = pl.smem <= kSmemBudgetBwd + 64;
  return pl;
}

bool fused_bwd_supported(const LayerShape& s, bool need_dx) { return plan_bwd(s, need_dx).ok; }

int launch_dw_from_partials(const float* part, float* dW, int nblocks, int K, int MT, int NT, int Fin, int Fout,
                            const float* db_part, float* db, int FoP, cudaStream_t st) {
  const int total = K * (MT * NT / 2) * 256;
  const int elems = total + (db_part != nullptr ? Fout : 0);
  k_dw_from_partials<<<ceil_div(elems, 32), 256, 0, st>>>(part, dW, nblocks, K, MT, NT, Fin, Fout, db_part, db, FoP);
  GCNB_LAUNCH_CHECK("k_dw_from_partials");
  return GCNB_OK;
}

size_t db_vertex_workspace(const LayerShape& s) { return align_up((size_t)kDbChunks * s.M * s.Fout * 4, 256) + 256; }

// per-vertex bias gradient (b2relu): two-stage column sum over the pooled tensors
int launch_db_vertex(const float* dy, const float* y, const uint8_t* argmax, float* db, const LayerShape& s, int relu,
                     int dy_is_mean, Workspace& ws, cudaStream_t st) {
  float* dbp = ws.take<float>((size_t)kDbChunks * s.M * s.Fout);
  if (!dbp) {
    set_error("workspace too small for the bias gradient");
    return GCNB_ERR_WORKSPACE;
  }
  int log2p = 0;
  while ((1 << log2p) < s.p) ++log2p;
  const int Mo = s.M / s.p;
  const int bchunk = ceil_div(s.B, kDbChunks);
  const int nch = ceil_div(s.B, bchunk);
  dim3 grid_db(ceil_div(Mo * s.Fout, 128), nch);
  k_db_partial<<<grid_db, 128, 0, st>>>(dy, y, argmax, dbp, s.B, s.M, s.Fout, s.p, log2p, relu, bchunk, dy_is_mean);
  GCNB_LAUNCH_CHECK("k_db_partial");
  k_db_final<<<ceil_div(s.M * s.Fout, 128), 128, 0, st>>>(dbp, db, nch, s.M, s.Fout, 1);
  GCNB_LAUNCH_CHECK("k_db_final");
  return GCNB_OK;
}

size_t fused_cheb_workspace(const LayerShape& s, bool backward, bool need_dx) {
  if (!backward) return 256;
  const BwdPlan pl = plan_bwd(s, need_dx);
  if (!pl.ok) return 0;
  const size_t part = (size_t)148 * 2 * (s.K * pl.nchunks * 256 + 32) * 4;  // up to 296 CTAs (+ bias partials)
  return align_up(part, 256) + db_vertex_workspace(s) + 512;
}

template <int MT, int NT, int SLOTS>
static int launch_bwd(const BwdParams& P, const BwdPlan& pl, int grid, cudaStream_t st) {
  auto kern = k_cheb_bwd_fused<MT, NT, SLOTS>;
  GCNB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.smem));
  kern<<<grid, pl.g.nwarps * 32, pl.smem, st>>>(P);
  GCNB_LAUNCH_CHECK("k_cheb_bwd_fused");
  return GCNB_OK;
}

int fused_cheb_bwd(const float* x, const int32_t* perm, int M_in, const float* y, const uint8_t* argmax, const float* dy,
                   const gcnb_csr& L, const gcnb_csr* Lt, const float* W, float* dx, float* dW, float* db,
                   const LayerShape& s, int bias_mode, int relu, int dy_is_mean, bool skip_dw, Workspace& ws,
                   cudaStream_t st) {
  const bool need_dx = dx != nullptr;
  const BwdPlan pl = plan_bwd(s, need_dx);
  if (!pl.ok) {
    set_error("fused backward does not support this shape");
    return GCNB_ERR_INVALID;
  }
  DeviceInfo di;
  int rc = device_info(&di);
  if (rc) return rc;
  const int ntiles = ceil_div(s.B, pl.g.S);
  const int grid = std::min(ntiles, std::min(di.sm_count, 296));
  float* part = ws.take<float>((size_t)grid * s.K * pl.nchunks * 256);
  float* dbf = ws.take<float>((size_t)grid * 32);
  if (!part || !dbf) {
    set_error("workspace too small for the fused backward path");
    return GCNB_ERR_WORKSPACE;
  }
  BwdParams P;
  P.x = x; P.perm = perm; P.M_in = M_in; P.y = y; P.argmax = argmax; P.dy = dy;
  P.rowptr = L.rowptr; P.col = L.col; P.val = L.val; P.nnz = L.nnz;
  P.rowptr_t = Lt ? Lt->rowptr : nullptr; P.col_t = Lt ? Lt->col : nullptr; P.val_t = Lt ? Lt->val : nullptr;
  const bool db_fused = bias_mode == GCNB_BIAS_PER_FILTER && db != nullptr;
  P.W = W; P.dx = dx; P.dw_part = part; P.db_part = db_fused ? dbf : nullptr;
  P.B = s.B; P.Fin = s.Fin; P.Fout = s.Fout; P.K = s.K; P.p = s.p; P.relu = relu; P.dy_is_mean = dy_is_mean;
  P.skip_dw = skip_dw ? 1 : 0;
  P.log2p = 0;
  while ((1 << P.log2p) < s.p) ++P.log2p;
  P.g = pl.g; P.FoP = pl.FoP; P.RSz = pl.RSz; P.ntiles = ntiles; P.nchunks = pl.nchunks;
  P.off_opT = pl.off_opT; P.off_wfragT = pl.off_wfragT; P.off_dws = pl.off_dws; P.off_scratch = pl.off_scratch;
  P.off_dz = pl.off_dz; P.off_slab = pl.off_slab;
  rc = GCNB_ERR_INVALID;
#define GCNB_BWD_CASE(mt, nt, sl) \
  if (pl.MT == mt && pl.NT == nt && pl.SLOTS == sl) rc = launch_bwd<mt, nt, sl>(P, pl, grid, st);
  GCNB_BWD_CASE(1, 2, 1) GCNB_BWD_CASE(1, 2, 2) GCNB_BWD_CASE(1, 2, 4)
  GCNB_BWD_CASE(1, 4, 1) GCNB_BWD_CASE(1, 4, 2) GCNB_BWD_CASE(1, 4, 4)
  GCNB_BWD_CASE(2, 2, 1) GCNB_BWD_CASE(2, 2, 2)
  GCNB_BWD_CASE(2, 4, 1) GCNB_BWD_CASE(2, 4, 2)
#undef GCNB_BWD_CASE
  if (rc) {
    if (rc == GCNB_ERR_INVALID) set_error("fused backward: no kernel instance for MT=%d NT=%d SLOTS=%d", pl.MT, pl.NT, pl.SLOTS);
    return rc;
  }
  if (skip_dw) return GCNB_OK;
  rc = launch_dw_from_partials(part, dW, grid, s.K, pl.MT, pl.NT, s.Fin, s.Fout, P.db_part, db, pl.FoP, st);
  if (rc) return rc;
  if (bias_mode == GCNB_BIAS_PER_VERTEX && db != nullptr) return launch_db_vertex(dy, y, argmax, db, s, relu, dy_is_mean, ws, st);
  return GCNB_OK;
}

}  // namespace gcnb
