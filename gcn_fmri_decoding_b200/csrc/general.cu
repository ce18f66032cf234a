// General (HBM-resident) path of the ChebyNet layer and the stand-alone pieces.
//
// Used when the rescaled Laplacian plus a tile of samples does not fit in shared memory
// (vertex-level graphs, BASELINE config 5) and as the shape-agnostic fallback of the fused
// kernels.  State lives in HBM/L2 in a vertex-major layout  Xn[m][b*F + f]  -- one contiguous
// row of B*F floats per vertex -- so that the sparse recursion gathers whole coalesced rows.
// (The reference picks the same [M, Fin*N] layout for its SpMM, models_gcn.py:598-599, but then
// pays two full transposes and K concats; here the layout change is one pass in and one out.)
//
// Kernels: to/from vertex-major (with the Graclus permutation gather fused in), CSR SpMM
// recursion step, row-tiled contractions for z = X W, G = dZ W^T and dW = X^T dZ, the
// bias/ReLU/max-pool epilogue and its adjoint, bias-gradient reductions.
#include <algorithm>

#include "common.cuh"

namespace gcnb {

// ------------------------------------------------------------------------------------------------
// layout changes
// ------------------------------------------------------------------------------------------------
// Xn[m][b*F + f] = x[b][perm ? perm[m] : m][f]   (0 for fake vertices, coarsening.py:260-264)
__global__ void k_to_node_major(const float* __restrict__ x, const int32_t* __restrict__ perm,
                                float* __restrict__ Xn, int B, int M, int M_in, int F) {
  const long long C = (long long)B * F;
  for (int m = blockIdx.y; m < M; m += gridDim.y) {
    const int src = perm ? perm[m] : m;
    for (long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x; c < C; c += (long long)gridDim.x * blockDim.x) {
      const int b = (int)(c / F);
      const int f = (int)(c - (long long)b * F);
      float v = 0.f;
      if (src < M_in) v = __ldg(x + ((long long)b * M_in + src) * F + f);
      Xn[(long long)m * C + c] = v;
    }
  }
}

// x[b][m][f] = Xn[m][b*F + f]
__global__ void k_from_node_major(const float* __restrict__ Xn, float* __restrict__ x, int B, int M, int F) {
  const long long C = (long long)B * F;
  for (int m = blockIdx.y; m < M; m += gridDim.y) {
    for (long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x; c < C; c += (long long)gridDim.x * blockDim.x) {
      const int b = (int)(c / F);
      const int f = (int)(c - (long long)b * F);
      x[((long long)b * M + m) * F + f] = Xn[(long long)m * C + c];
    }
  }
}

// Tiled versions of the two layout changes (and of the p == 1 epilogue adjoint): a CTA moves a tile of kTileM
// vertices x TB samples through shared memory so that BOTH sides are read / written in long contiguous runs
// (TM*F floats per sample on the sample-major side, TB*F floats per vertex on the vertex-major side) instead of
// F-float snippets on one of them.
//   MODE 0: Xn[m][b*ld + f] = x[b][perm ? perm[m] : m][f]      (0 for fake vertices)
//   MODE 1: x[b][m][f]      = Xn[m][b*ld + f]
//   MODE 2: dZn[m][b*ld + o] = relu ? (y[b][m][o] > 0 ? dy[b][m][o] : 0) : dy[b][m][o]        (p == 1)
constexpr int kTileM = 16;

template <int MODE>
__global__ void __launch_bounds__(256) k_tile_swap(const float* __restrict__ src, const float* __restrict__ src2,
                                                   const int32_t* __restrict__ perm, float* __restrict__ dst, int B, int M,
                                                   int M_in, int F, int ld, int TB, int relu) {
  extern __shared__ float tile[];  // [kTileM][TB*F]
  const int m0 = blockIdx.x * kTileM, b0 = blockIdx.y * TB;
  const int tm = min(kTileM, M - m0), tb = min(TB, B - b0);
  const int row = TB * F;
  if (MODE == 1) {
    // vertex-major in: per vertex a run of tb*F floats (rows are ld apart per sample; ld == F here)
    for (int i = threadIdx.x; i < tm * tb * F; i += 256) {
      const int m = i / (tb * F), c = i - m * (tb * F);
      tile[m * row + c] = src[((long long)(m0 + m) * B + b0) * ld + c];
    }
    __syncthreads();
    for (int i = threadIdx.x; i < tb * tm * F; i += 256) {
      const int b = i / (tm * F), j = i - b * (tm * F);
      const int m = j / F, f = j - m * F;
      dst[((long long)(b0 + b) * M + m0) * F + j] = tile[m * row + b * F + f];
    }
  } else {
    for (int i = threadIdx.x; i < tb * tm * F; i += 256) {
      const int b = i / (tm * F), j = i - b * (tm * F);
      const int m = j / F, f = j - m * F;
      float v;
      if (MODE == 0) {
        const int sm = perm ? perm[m0 + m] : m0 + m;
        v = sm < M_in ? src[((long long)(b0 + b) * M_in + sm) * F + f] : 0.f;
      } else {
        const long long o = ((long long)(b0 + b) * M + m0) * F + j;
        v = src[o];
        if (relu && !(src2[o] > 0.f)) v = 0.f;
      }
      tile[m * row + b * F + f] = v;
    }
    __syncthreads();
    if (ld == F) {
      for (int i = threadIdx.x; i < tm * tb * F; i += 256) {
        const int m = i / (tb * F), c = i - m * (tb * F);
        dst[((long long)(m0 + m) * B + b0) * F + c] = tile[m * row + c];
      }
    } else {
      for (int i = threadIdx.x; i < tm * tb * F; i += 256) {
        const int m = i / (tb * F), c = i - m * (tb * F);
        const int b = c / F, f = c - b * F;
        dst[((long long)(m0 + m) * B + b0 + b) * ld + f] = tile[m * row + c];
      }
    }
  }
}

// samples per tile so that the tile fits the 48 KB static shared-memory window; 0 = use the untiled kernels
static int tile_samples(int B, int F) {
  const int cap = 48 * 1024 / (kTileM * F * 4);
  return cap >= 4 ? std::min(std::min(B, 32), cap) : 0;
}

int launch_to_node_major(const float* x, const int32_t* perm, float* X0, int B, int M, int M_in, int F,
                         cudaStream_t st) {
  const int TB = tile_samples(B, F);
  if (TB > 0) {
    dim3 grid((unsigned)ceil_div(M, kTileM), (unsigned)ceil_div(B, TB));
    k_tile_swap<0><<<grid, 256, (size_t)kTileM * TB * F * 4, st>>>(x, nullptr, perm, X0, B, M, M_in, F, F, TB, 0);
    GCNB_LAUNCH_CHECK("k_tile_swap<0>");
    return GCNB_OK;
  }
  long long C = (long long)B * F;
  dim3 grid((unsigned)std::min<long long>(ceil_div_ll(C, 256), 1024), (unsigned)std::min(M, 65535));
  k_to_node_major<<<grid, 256, 0, st>>>(x, perm, X0, B, M, M_in, F);
  GCNB_LAUNCH_CHECK("k_to_node_major");
  return GCNB_OK;
}

int launch_from_node_major(const float* Xn, float* x, int B, int M, int F, cudaStream_t st) {
  const int TB = tile_samples(B, F);
  if (TB > 0) {
    dim3 grid((unsigned)ceil_div(M, kTileM), (unsigned)ceil_div(B, TB));
    k_tile_swap<1><<<grid, 256, (size_t)kTileM * TB * F * 4, st>>>(Xn, nullptr, nullptr, x, B, M, M, F, F, TB, 0);
    GCNB_LAUNCH_CHECK("k_tile_swap<1>");
    return GCNB_OK;
  }
  long long C = (long long)B * F;
  dim3 grid((unsigned)std::min<long long>(ceil_div_ll(C, 256), 1024), (unsigned)std::min(M, 65535));
  k_from_node_major<<<grid, 256, 0, st>>>(Xn, x, B, M, F);
  GCNB_LAUNCH_CHECK("k_from_node_major");
  return GCNB_OK;
}

// ------------------------------------------------------------------------------------------------
// sparse recursion step:  out[m][:] = alpha * sum_j val_j * src[col_j][:] + beta * add[m][:] + beta2 * add2[m][:]
//   forward  X_k = 2 L~ X_{k-1} - X_{k-2}                 (alpha=2 (1 for k=1), beta=-1, no add2)
//   adjoint  b_k = G_k + 2 L~^T b_{k+1} - b_{k+2}         (Clenshaw; add = G_k aliases out, add2 = b_{k+2})
// One block row per vertex, threads along the B*F columns, VEC floats per thread.
// ------------------------------------------------------------------------------------------------
template <int VEC>
__global__ void __launch_bounds__(128) k_spmm_step(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col,
                                                   const float* __restrict__ val, const float* __restrict__ src,
                                                   const float* add, const float* add2, float* out, int M,
                                                   long long C, float alpha, float beta, float beta2) {
  const long long CV = C / VEC;
  for (int m = blockIdx.y; m < M; m += gridDim.y) {
    const int beg = rowptr[m], end = rowptr[m + 1];
    for (long long cv = (long long)blockIdx.x * blockDim.x + threadIdx.x; cv < CV; cv += (long long)gridDim.x * blockDim.x) {
      float acc[VEC];
#pragma unroll
      for (int i = 0; i < VEC; ++i) acc[i] = 0.f;
      for (int j = beg; j < end; ++j) {
        const float v = __ldg(val + j);
        const float* p = src + (long long)__ldg(col + j) * C + cv * VEC;
        if (VEC == 4) {
          const float4 t = *reinterpret_cast<const float4*>(p);
          acc[0] = fmaf(v, t.x, acc[0]);
          acc[1 % VEC] = fmaf(v, t.y, acc[1 % VEC]);
          acc[2 % VEC] = fmaf(v, t.z, acc[2 % VEC]);
          acc[3 % VEC] = fmaf(v, t.w, acc[3 % VEC]);
        } else {
          acc[0] = fmaf(v, *p, acc[0]);
        }
      }
      const long long o = (long long)m * C + cv * VEC;
      if (VEC == 4) {
        float4 r = make_float4(alpha * acc[0], alpha * acc[1 % VEC], alpha * acc[2 % VEC], alpha * acc[3 % VEC]);
        if (add != nullptr) {
          const float4 a = *reinterpret_cast<const float4*>(add + o);
          r.x = fmaf(beta, a.x, r.x);
          r.y = fmaf(beta, a.y, r.y);
          r.z = fmaf(beta, a.z, r.z);
          r.w = fmaf(beta, a.w, r.w);
        }
        if (add2 != nullptr) {
          const float4 a = *reinterpret_cast<const float4*>(add2 + o);
          r.x = fmaf(beta2, a.x, r.x);
          r.y = fmaf(beta2, a.y, r.y);
          r.z = fmaf(beta2, a.z, r.z);
          r.w = fmaf(beta2, a.w, r.w);
        }
        *reinterpret_cast<float4*>(out + o) = r;
      } else {
        float r = alpha * acc[0];
        if (add != nullptr) r = fmaf(beta, add[o], r);
        if (add2 != nullptr) r = fmaf(beta2, add2[o], r);
        out[o] = r;
      }
    }
  }
}

static int launch_spmm_step(const gcnb_csr& L, const float* src, const float* add, const float* add2, float* out,
                            long long C, float alpha, float beta, float beta2, cudaStream_t st) {
  if (spmm_tma_supported(L, C, src, add, add2, out)) return spmm_tma(L, src, add, add2, out, C, alpha, beta, beta2, st);
  const bool vec = (C % 4 == 0) && ((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(out) |
                                     reinterpret_cast<uintptr_t>(add) | reinterpret_cast<uintptr_t>(add2)) % 16 == 0);
  const long long CV = vec ? C / 4 : C;
  dim3 grid((unsigned)std::min<long long>(ceil_div_ll(CV, 128), 4096), (unsigned)std::min(L.M, 65535));
  if (vec)
    k_spmm_step<4><<<grid, 128, 0, st>>>(L.rowptr, L.col, L.val, src, add, add2, out, L.M, C, alpha, beta, beta2);
  else
    k_spmm_step<1><<<grid, 128, 0, st>>>(L.rowptr, L.col, L.val, src, add, add2, out, L.M, C, alpha, beta, beta2);
  GCNB_LAUNCH_CHECK("k_spmm_step");
  return GCNB_OK;
}

// ------------------------------------------------------------------------------------------------
// row-tiled contraction (FFMA):
//   C[z][r][n] = sum_{q<nq} sum_{kk<Kd} A[q*a_q + r*lda + kk] * Bm[z*b_z + q*b_q + kk*sbk + n*sbn]
// 64 rows x 32 columns per block, 256 threads, 8 rows per thread, A tile read as broadcast float4.
//   z = X W          : nq=K, A=X stack (lda=Fin), B=W  (sbk=K*Fout, sbn=1, b_q=Fout)
//   G_k = dZ W_k^T   : z=k,  A=dZ (lda=Fout),     B=W  (sbk=1, sbn=K*Fout, b_z=Fout)
// ------------------------------------------------------------------------------------------------
struct RowGemm {
  const float* A;
  long long a_q;
  int lda;
  const float* Bm;
  long long b_z, b_q, sbk, sbn;
  float* C;
  long long c_z;
  int ldc;
  long long R;
  int N, Kd, nq;
};

__global__ void __launch_bounds__(256) k_rowgemm(RowGemm g) {
  __shared__ __align__(16) float As[64][36];
  __shared__ float Bs[32][33];
  const int tid = threadIdx.x, lane = tid & 31, ty = tid >> 5;
  const long long r0 = (long long)blockIdx.x * 64;
  const int n0 = blockIdx.y * 32;
  const int z = blockIdx.z;
  float acc[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) acc[i] = 0.f;
  for (int q = 0; q < g.nq; ++q) {
    const float* Aq = g.A + (long long)q * g.a_q;
    const float* Bq = g.Bm + (long long)z * g.b_z + (long long)q * g.b_q;
    for (int k0 = 0; k0 < g.Kd; k0 += 32) {
      for (int idx = tid; idx < 64 * 32; idx += 256) {
        const int row = idx >> 5, j = idx & 31;
        float v = 0.f;
        if (r0 + row < g.R && k0 + j < g.Kd) v = __ldg(Aq + (r0 + row) * g.lda + k0 + j);
        As[row][j] = v;
      }
      for (int idx = tid; idx < 32 * 32; idx += 256) {
        // idx -> (kk, n); walk the contiguous axis of B with consecutive threads
        int kk, n;
        if (g.sbn == 1) { kk = idx >> 5; n = idx & 31; } else { n = idx >> 5; kk = idx & 31; }
        float v = 0.f;
        if (k0 + kk < g.Kd && n0 + n < g.N) v = __ldg(Bq + (long long)(k0 + kk) * g.sbk + (long long)(n0 + n) * g.sbn);
        Bs[kk][n] = v;
      }
      __syncthreads();
#pragma unroll
      for (int kk = 0; kk < 32; kk += 4) {
        const float b0 = Bs[kk][lane], b1 = Bs[kk + 1][lane], b2 = Bs[kk + 2][lane], b3 = Bs[kk + 3][lane];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float4 a = *reinterpret_cast<const float4*>(&As[ty * 8 + i][kk]);
          acc[i] = fmaf(a.x, b0, acc[i]);
          acc[i] = fmaf(a.y, b1, acc[i]);
          acc[i] = fmaf(a.z, b2, acc[i]);
          acc[i] = fmaf(a.w, b3, acc[i]);
        }
      }
      __syncthreads();
    }
  }
  if (n0 + lane < g.N) {
    float* Cz = g.C + (long long)z * g.c_z;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const long long r = r0 + ty * 8 + i;
      if (r < g.R) Cz[r * g.ldc + n0 + lane] = acc[i];
    }
  }
}

static int launch_rowgemm(const RowGemm& g, int nz, cudaStream_t st) {
  dim3 grid((unsigned)ceil_div_ll(g.R, 64), (unsigned)ceil_div(g.N, 32), (unsigned)nz);
  k_rowgemm<<<grid, 256, 0, st>>>(g);
  GCNB_LAUNCH_CHECK("k_rowgemm");
  return GCNB_OK;
}

// ------------------------------------------------------------------------------------------------
// weight gradient:  part[k][chunk][f][o] = sum_{r in chunk} X_k[r][f] * dZ[r][o]
// then dW[f*K+k][o] = sum_chunk part  (two-stage, deterministic -- no float atomics)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_dw_partial(const float* __restrict__ Xs, long long slab,
                                                    const float* __restrict__ dZ, int ldz, float* __restrict__ part,
                                                    long long R, int Fin, int Fout, int rows_per_chunk, int nchunks) {
  __shared__ __align__(16) float Xt[32][36];
  __shared__ float Dt[32][33];
  const int tid = threadIdx.x, lane = tid & 31, ty = tid >> 5;
  const int chunk = blockIdx.x, k = blockIdx.y;
  const int nfo = (Fout + 31) / 32;
  const int f0 = (blockIdx.z / nfo) * 32, o0 = (blockIdx.z % nfo) * 32;
  const float* Xk = Xs + (long long)k * slab;
  const long long rbeg = (long long)chunk * rows_per_chunk;
  const long long rend = rbeg + rows_per_chunk < R ? rbeg + rows_per_chunk : R;
  float acc[4] = {0.f, 0.f, 0.f, 0.f};
  for (long long r0 = rbeg; r0 < rend; r0 += 32) {
    for (int idx = tid; idx < 32 * 32; idx += 256) {
      const int rr = idx >> 5, j = idx & 31;
      const long long r = r0 + rr;
      Xt[rr][j] = (r < rend && f0 + j < Fin) ? __ldg(Xk + r * Fin + f0 + j) : 0.f;
      Dt[rr][j] = (r < rend && o0 + j < Fout) ? __ldg(dZ + r * ldz + o0 + j) : 0.f;
    }
    __syncthreads();
#pragma unroll 8
    for (int rr = 0; rr < 32; ++rr) {
      const float d = Dt[rr][lane];
      const float4 xv = *reinterpret_cast<const float4*>(&Xt[rr][4 * ty]);
      acc[0] = fmaf(xv.x, d, acc[0]);
      acc[1] = fmaf(xv.y, d, acc[1]);
      acc[2] = fmaf(xv.z, d, acc[2]);
      acc[3] = fmaf(xv.w, d, acc[3]);
    }
    __syncthreads();
  }
  if (o0 + lane < Fout) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int f = f0 + 4 * ty + i;
      if (f < Fin) part[(((long long)k * nchunks + chunk) * Fin + f) * Fout + o0 + lane] = acc[i];
    }
  }
}

__global__ void k_dw_reduce(const float* __restrict__ part, float* __restrict__ dW, int K, int Fin, int Fout,
                            int nchunks) {
  const int total = K * Fin * Fout;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int o = i % Fout, f = (i / Fout) % Fin, k = i / (Fout * Fin);
    float s = 0.f;
    for (int c = 0; c < nchunks; ++c) s += part[(((long long)k * nchunks + c) * Fin + f) * Fout + o];
    dW[((long long)f * K + k) * Fout + o] = s;
  }
}

// ------------------------------------------------------------------------------------------------
// epilogue on the vertex-major pre-activation Zn[m][b*F + o]:
//   a = relu(z + bias);  y[b][j][o] = max over the SAME-padded window of p vertices; first max wins.
// ------------------------------------------------------------------------------------------------
__global__ void k_epilogue(const float* __restrict__ Zn, const float* __restrict__ bias, float* __restrict__ y,
                           uint8_t* __restrict__ argmax, int B, int M, int F, int p, int bias_mode, int relu) {
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
      float v = Zn[((long long)m * B + b) * F + o];
      if (bias_mode == GCNB_BIAS_PER_FILTER) v += bias[o];
      else if (bias_mode == GCNB_BIAS_PER_VERTEX) v += bias[(long long)m * F + o];
      if (relu) v = fmaxf(v, 0.f);
      if (v > best) { best = v; bi = w; }  // strict: the first maximum keeps the slot
    }
    y[i] = best;
    if (argmax) argmax[i] = (uint8_t)bi;
  }
}

int launch_epilogue(const float* Zn, const float* bias, float* y, uint8_t* argmax, int B, int M, int F, int p,
                    int bias_mode, int relu, cudaStream_t st) {
  const long long total = (long long)B * ceil_div(M, p) * F;
  k_epilogue<<<(unsigned)std::min<long long>(ceil_div_ll(total, 256), 1 << 20), 256, 0, st>>>(Zn, bias, y, argmax, B, M,
                                                                                            F, p, bias_mode, relu);
  GCNB_LAUNCH_CHECK("k_epilogue");
  return GCNB_OK;
}

// adjoint of the epilogue: dZn[m][b*F+o] = (m is the window's arg-max) ? dy * [y>0] : 0
__global__ void k_dz(const float* __restrict__ dy, const float* __restrict__ y, const uint8_t* __restrict__ argmax,
                     float* __restrict__ dZn, int ldz, int B, int M, int F, int p, int relu) {
  const int Mo = (M + p - 1) / p;
  const int before = (Mo * p - M) / 2;
  const long long total = (long long)B * Mo * F;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int o = (int)(i % F);
    const int j = (int)((i / F) % Mo);
    const int b = (int)(i / ((long long)F * Mo));
    float g = dy[i];
    if (relu && !(y[i] > 0.f)) g = 0.f;
    const int am = (argmax && p > 1) ? argmax[i] : 0;
    for (int w = 0; w < p; ++w) {
      const int m = j * p - before + w;
      if (m < 0 || m >= M) continue;
      dZn[((long long)m * B + b) * ldz + o] = (w == am) ? g : 0.f;
    }
  }
}

int launch_dz(const float* dy, const float* y, const uint8_t* argmax, float* dZn, int ldz, int B, int M, int F, int p,
              int relu, cudaStream_t st) {
  const int TB = tile_samples(B, F);
  if (p == 1 && TB > 0 && M <= 65535 * kTileM) {
    dim3 grid((unsigned)ceil_div(M, kTileM), (unsigned)ceil_div(B, TB));
    k_tile_swap<2><<<grid, 256, (size_t)kTileM * TB * F * 4, st>>>(dy, y, nullptr, dZn, B, M, M, F, ldz, TB, relu);
    GCNB_LAUNCH_CHECK("k_tile_swap<2>");
    return GCNB_OK;
  }
  const long long total = (long long)B * ceil_div(M, p) * F;
  k_dz<<<(unsigned)std::min<long long>(ceil_div_ll(total, 256), 1 << 20), 256, 0, st>>>(dy, y, argmax, dZn, ldz, B, M,
                                                                                      F, p, relu);
  GCNB_LAUNCH_CHECK("k_dz");
  return GCNB_OK;
}

// db2[m][o] = sum_b dZn[m][b*ldz+o]   (one block per vertex; fixed summation order)
__global__ void __launch_bounds__(256) k_db_vertex(const float* __restrict__ dZn, int ldz, float* __restrict__ db2, int B,
                                                   int F) {
  __shared__ float red[256];
  const int m = blockIdx.x;
  const float* row = dZn + (long long)m * B * ldz;
  for (int o0 = 0; o0 < F; o0 += 32) {
    // 8 groups of 32 lanes stride over b, then a fixed-order tree over the 8 groups
    const int lane = threadIdx.x & 31, grp = threadIdx.x >> 5;
    float s = 0.f;
    if (o0 + lane < F)
      for (int b = grp; b < B; b += 8) s += row[(long long)b * ldz + o0 + lane];
    red[threadIdx.x] = s;
    __syncthreads();
    if (grp == 0 && o0 + lane < F) {
      float t = 0.f;
#pragma unroll
      for (int g2 = 0; g2 < 8; ++g2) t += red[g2 * 32 + lane];
      db2[(long long)m * F + o0 + lane] = t;
    }
    __syncthreads();
  }
}

// db[o] = sum_m db2[m][o] in two fixed-order stages: kDbFilterChunks partial sums over vertex ranges, then their sum
constexpr int kDbFilterChunks = 64;

__global__ void __launch_bounds__(256) k_db_filter_partial(const float* __restrict__ db2, float* __restrict__ part, int M,
                                                           int F) {
  __shared__ float red[256];
  const int lane = threadIdx.x & 31, grp = threadIdx.x >> 5;
  const int o = blockIdx.x * 32 + lane;
  const int per = (M + kDbFilterChunks - 1) / kDbFilterChunks;
  const int m0 = blockIdx.y * per, m1 = min(M, m0 + per);
  float s = 0.f;
  if (o < F)
    for (int m = m0 + grp; m < m1; m += 8) s += db2[(long long)m * F + o];
  red[threadIdx.x] = s;
  __syncthreads();
  if (grp == 0 && o < F) {
    float t = 0.f;
#pragma unroll
    for (int g2 = 0; g2 < 8; ++g2) t += red[g2 * 32 + lane];
    part[blockIdx.y * F + o] = t;
  }
}

__global__ void k_db_filter_final(const float* __restrict__ part, float* __restrict__ db, int F) {
  const int o = blockIdx.x * blockDim.x + threadIdx.x;
  if (o >= F) return;
  float t = 0.f;
  for (int c = 0; c < kDbFilterChunks; ++c) t += part[c * F + o];
  db[o] = t;
}

// scratch: M*F floats (per-vertex sums) followed by kDbFilterChunks*F floats
size_t db_scratch_floats(int M, int F) { return (size_t)M * F + (size_t)kDbFilterChunks * F; }

int launch_db(const float* dZn, int ldz, float* db, float* scratch, int B, int M, int F, int bias_mode, cudaStream_t st) {
  if (bias_mode == GCNB_BIAS_NONE || db == nullptr) return GCNB_OK;
  float* db2 = bias_mode == GCNB_BIAS_PER_VERTEX ? db : scratch;
  k_db_vertex<<<M, 256, 0, st>>>(dZn, ldz, db2, B, F);
  GCNB_LAUNCH_CHECK("k_db_vertex");
  if (bias_mode == GCNB_BIAS_PER_FILTER) {
    float* part = scratch + (size_t)M * F;
    k_db_filter_partial<<<dim3(ceil_div(F, 32), kDbFilterChunks), 256, 0, st>>>(db2, part, M, F);
    GCNB_LAUNCH_CHECK("k_db_filter_partial");
    k_db_filter_final<<<ceil_div(F, 128), 128, 0, st>>>(part, db, F);
    GCNB_LAUNCH_CHECK("k_db_filter_final");
  }
  return GCNB_OK;
}

// ------------------------------------------------------------------------------------------------
// the general layer: forward and backward drivers
// ------------------------------------------------------------------------------------------------
static int dw_chunking(long long R, int* rows_per_chunk) {
  long long rpc = std::max<long long>(2048, ceil_div_ll(R, 256));
  rpc = (rpc + 31) / 32 * 32;
  *rows_per_chunk = (int)rpc;
  return (int)ceil_div_ll(R, rpc);
}

size_t general_cheb_workspace(const LayerShape& s, bool backward, bool need_dx) {
  const size_t slab = (size_t)s.M * s.B * s.Fin;
  const size_t zn = (size_t)s.M * s.B * node_mma_ldz(s.Fout);  // dZn rows may be padded for the tensor-core kernels
  size_t n = 0;
  auto add = [&](size_t floats) { n = align_up(n, 256) + floats * sizeof(float); };
  add(slab * s.K);  // X stack (forward) / recomputed stack (backward)
  add(zn);          // Zn or dZn
  if (backward) {
    int rpc;
    const int nch = std::max(dw_chunking((long long)s.M * s.B, &rpc), node_dw_blocks(s));
    add((size_t)s.K * nch * s.Fin * s.Fout);  // dW partials
    add(db_scratch_floats(s.M, s.Fout));      // db scratch
    if (need_dx) add(slab * s.K);             // G stack
  }
  return align_up(n, 256) + 256;
}

static int build_stack(float* Xs, const gcnb_csr& L, long long slab, long long C, int K, cudaStream_t st) {
  for (int k = 1; k < K; ++k) {
    const float* prev = Xs + (long long)(k - 1) * slab;
    const float* prev2 = k >= 2 ? Xs + (long long)(k - 2) * slab : nullptr;
    int rc = launch_spmm_step(L, prev, prev2, nullptr, Xs + (long long)k * slab, C, k == 1 ? 1.f : 2.f, -1.f, 0.f, st);
    if (rc) return rc;
  }
  return GCNB_OK;
}

int general_cheb_fwd(const float* x, const int32_t* perm, int M_in, const gcnb_csr& L, const float* W,
                     const float* bias, float* y, uint8_t* argmax, float* xstack, const LayerShape& s, int bias_mode,
                     int relu, Workspace& ws, cudaStream_t st) {
  const long long C = (long long)s.B * s.Fin;
  const long long slab = (long long)s.M * C;
  // the Chebyshev stack is built in the caller's buffer when it wants to keep it for the backward pass
  float* Xs = xstack ? xstack : ws.take<float>((size_t)slab * s.K);
  float* Zn = ws.take<float>((size_t)s.M * s.B * node_mma_ldz(s.Fout));
  if (!Xs || !Zn) {
    set_error("workspace too small for the general forward path");
    return GCNB_ERR_WORKSPACE;
  }
  int rc = launch_to_node_major(x, perm, Xs, s.B, s.M, M_in, s.Fin, st);
  if (rc) return rc;
  rc = build_stack(Xs, L, slab, C, s.K, st);
  if (rc) return rc;
  if (node_contract_supported(s)) {
    // tensor-core contraction streaming the stack through TMA; without pooling the bias/ReLU epilogue is fused
    // and y is written once, straight in the caller's [B, M, Fout] layout
    if (s.p == 1) {
      rc = node_contract(Xs, slab, W, bias, y, s, bias_mode, relu, 1, st);
      if (rc) return rc;
      if (argmax) GCNB_CUDA(cudaMemsetAsync(argmax, 0, (size_t)s.B * s.M * s.Fout, st));
      return GCNB_OK;
    }
    rc = node_contract(Xs, slab, W, nullptr, Zn, s, GCNB_BIAS_NONE, 0, 0, st);
    if (rc) return rc;
    return launch_epilogue(Zn, bias, y, argmax, s.B, s.M, s.Fout, s.p, bias_mode, relu, st);
  }
  RowGemm g;
  g.A = Xs; g.a_q = slab; g.lda = s.Fin;
  g.Bm = W; g.b_z = 0; g.b_q = s.Fout; g.sbk = (long long)s.K * s.Fout; g.sbn = 1;
  g.C = Zn; g.c_z = 0; g.ldc = s.Fout;
  g.R = (long long)s.M * s.B; g.N = s.Fout; g.Kd = s.Fin; g.nq = s.K;
  rc = launch_rowgemm(g, 1, st);
  if (rc) return rc;
  return launch_epilogue(Zn, bias, y, argmax, s.B, s.M, s.Fout, s.p, bias_mode, relu, st);
}

// seeds G_k = dZ W_k^T for every k, then the Clenshaw form of the adjoint recursion, in place on the seeds:
//   b_k = G_k + 2 L~^T b_{k+1} - b_{k+2}  (k = K-2 .. 1, b_{K-1} = G_{K-1}),   dx = G_0 + L~^T b_1 - b_2
// Gs ends with dx (vertex-major) in slab 0 and b_1 .. b_{K-1} in slabs 1 .. K-1.  Lt may be NULL when K = 1.
static int adjoint_states(const float* dZn, int ldz, const float* W, const gcnb_csr* Lt, float* Gs, bool mma_g,
                          const LayerShape& s, cudaStream_t st) {
  const long long C = (long long)s.B * s.Fin;
  const long long slab = (long long)s.M * C;
  int rc;
  if (mma_g) {
    rc = node_dz_wt(dZn, W, Gs, slab, s, st);
    if (rc) return rc;
  } else {
    RowGemm g;
    g.A = dZn; g.a_q = 0; g.lda = ldz;
    g.Bm = W; g.b_z = s.Fout; g.b_q = 0; g.sbk = 1; g.sbn = (long long)s.K * s.Fout;
    g.C = Gs; g.c_z = slab; g.ldc = s.Fin;
    g.R = (long long)s.M * s.B; g.N = s.Fin; g.Kd = s.Fout; g.nq = 1;
    rc = launch_rowgemm(g, s.K, st);
    if (rc) return rc;
  }
  for (int k = s.K - 2; k >= 0; --k) {
    float* bk = Gs + (long long)k * slab;
    const float* bk1 = Gs + (long long)(k + 1) * slab;
    const float* bk2 = k + 2 <= s.K - 1 ? Gs + (long long)(k + 2) * slab : nullptr;
    rc = launch_spmm_step(*Lt, bk1, bk, bk2, bk, C, k == 0 ? 1.f : 2.f, 1.f, -1.f, st);
    if (rc) return rc;
  }
  return GCNB_OK;
}

int general_cheb_bwd(const float* x, const int32_t* perm, int M_in, const float* y, const uint8_t* argmax, const float* dy, const gcnb_csr& L,
                     const gcnb_csr* Lt, const float* W, float* dx, float* dW, float* db, const float* xstack,
                     const LayerShape& s, int bias_mode, int relu, Workspace& ws, cudaStream_t st) {
  const long long C = (long long)s.B * s.Fin;
  const long long slab = (long long)s.M * C;
  const long long R = (long long)s.M * s.B;
  const bool mma_dw = node_dw_supported(s);
  const bool mma_g = dx != nullptr && node_dz_wt_supported(s);
  const int ldz = (mma_dw || mma_g) ? node_mma_ldz(s.Fout) : s.Fout;
  int rpc;
  const int nch = mma_dw ? node_dw_blocks(s) : dw_chunking(R, &rpc);
  float* Xw = xstack ? nullptr : ws.take<float>((size_t)slab * s.K);
  const float* Xs = xstack ? xstack : Xw;
  float* dZn = ws.take<float>((size_t)R * node_mma_ldz(s.Fout));
  float* part = ws.take<float>((size_t)s.K * std::max(nch, node_dw_blocks(s)) * s.Fin * s.Fout);
  float* dbs = ws.take<float>(db_scratch_floats(s.M, s.Fout));
  float* Gs = dx ? ws.take<float>((size_t)slab * s.K) : nullptr;
  if (!Xs || !dZn || !part || !dbs || (dx && !Gs)) {
    set_error("workspace too small for the general backward path");
    return GCNB_ERR_WORKSPACE;
  }
  int rc = launch_dz(dy, y, argmax, dZn, ldz, s.B, s.M, s.Fout, s.p, relu, st);
  if (rc) return rc;
  rc = launch_db(dZn, ldz, db, dbs, s.B, s.M, s.Fout, bias_mode, st);
  if (rc) return rc;
  if (xstack == nullptr) {
    // recompute the Chebyshev stack from x (nothing but x, y and argmax was kept from the forward)
    rc = launch_to_node_major(x, perm, Xw, s.B, s.M, M_in, s.Fin, st);
    if (rc) return rc;
    rc = build_stack(Xw, L, slab, C, s.K, st);
    if (rc) return rc;
  }
  if (mma_dw) {
    rc = node_dw(Xs, slab, dZn, part, s, st);
    if (rc) return rc;
  } else {
    dim3 grid((unsigned)nch, (unsigned)s.K, (unsigned)(ceil_div(s.Fin, 32) * ceil_div(s.Fout, 32)));
    k_dw_partial<<<grid, 256, 0, st>>>(Xs, slab, dZn, ldz, part, R, s.Fin, s.Fout, rpc, nch);
    GCNB_LAUNCH_CHECK("k_dw_partial");
  }
  {
    const int total = s.K * s.Fin * s.Fout;
    k_dw_reduce<<<ceil_div(total, 256), 256, 0, st>>>(part, dW, s.K, s.Fin, s.Fout, nch);
    GCNB_LAUNCH_CHECK("k_dw_reduce");
  }
  if (dx == nullptr) return GCNB_OK;
  if (Lt == nullptr && s.K > 1) {
    set_error("dx requested but the transposed operator Lt is NULL");
    return GCNB_ERR_INVALID;
  }
  rc = adjoint_states(dZn, ldz, W, Lt, Gs, mma_g, s, st);
  if (rc) return rc;
  return launch_from_node_major(Gs, dx, s.B, s.M, s.Fin, st);
}

// ------------------------------------------------------------------------------------------------
// gradient w.r.t. the operator (edge saliency): the basis X_k and the Clenshaw states b_k of general_cheb_bwd, then
// dL~ = sum_k c_k b_k X_{k-1}^T sampled on L~'s pattern and diagonal (k_sddmm_tma, sddmm_tma.cu).  No dW, no db.
// ------------------------------------------------------------------------------------------------
size_t general_cheb_dL_workspace(const LayerShape& s) {
  const size_t slab = (size_t)s.M * s.B * s.Fin;
  size_t n = 0;
  auto add = [&](size_t floats) { n = align_up(n, 256) + floats * sizeof(float); };
  add(slab * s.K + 4);                          // X stack (+16 bytes read past the end by the gathers)
  add((size_t)s.M * s.B * node_mma_ldz(s.Fout));  // dZn
  add(slab * s.K + 4);                          // G stack -> Clenshaw states
  return align_up(n, 256) + 256;
}

int general_cheb_dL(const float* x, const int32_t* perm, int M_in, const float* y, const uint8_t* argmax, const float* dy,
                    const gcnb_csr& L, const gcnb_csr* Lt, const float* W, float* dval, float* ddiag, int accumulate,
                    float* dx, const LayerShape& s, int relu, Workspace& ws, cudaStream_t st) {
  const long long C = (long long)s.B * s.Fin;
  const long long slab = (long long)s.M * C;
  const long long R = (long long)s.M * s.B;
  // the same kernels, layouts and summation orders as general_cheb_bwd with dx, so that dx agrees bit for bit
  const bool mma_g = node_dz_wt_supported(s);
  const int ldz = (node_dw_supported(s) || mma_g) ? node_mma_ldz(s.Fout) : s.Fout;
  float* Xs = ws.take<float>((size_t)slab * s.K + 4);
  float* dZn = ws.take<float>((size_t)R * node_mma_ldz(s.Fout));
  float* Gs = ws.take<float>((size_t)slab * s.K + 4);
  if (!Xs || !dZn || !Gs) {
    set_error("workspace too small for the operator gradient");
    return GCNB_ERR_WORKSPACE;
  }
  if (Lt == nullptr && s.K > 1) {
    set_error("the operator gradient needs the transposed operator Lt");
    return GCNB_ERR_INVALID;
  }
  int rc = launch_dz(dy, y, argmax, dZn, ldz, s.B, s.M, s.Fout, s.p, relu, st);
  if (rc) return rc;
  rc = launch_to_node_major(x, perm, Xs, s.B, s.M, M_in, s.Fin, st);
  if (rc) return rc;
  rc = build_stack(Xs, L, slab, C, s.K, st);
  if (rc) return rc;
  rc = adjoint_states(dZn, ldz, W, Lt, Gs, mma_g, s, st);
  if (rc) return rc;
  if (s.K > 1) {
    rc = sddmm_tma(L, Xs, Gs, dval, ddiag, accumulate, s, st);
    if (rc) return rc;
  } else if (!accumulate) {  // a K = 1 layer applies no operator: its gradient is zero
    GCNB_CUDA(cudaMemsetAsync(dval, 0, (size_t)s.B * L.nnz * sizeof(float), st));
    GCNB_CUDA(cudaMemsetAsync(ddiag, 0, (size_t)s.B * s.M * sizeof(float), st));
  }
  return dx ? launch_from_node_major(Gs, dx, s.B, s.M, s.Fin, st) : GCNB_OK;
}

}  // namespace gcnb
