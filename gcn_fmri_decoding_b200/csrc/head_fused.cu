// The classifier head of the training step as ONE persistent cooperative kernel (SURVEY.md 8f row 1):
//   forward  (models_gcn.py:650-656, :674-681, :253-259)
//     h1 = dropout(relu(a0 W1 + b1)) ; h2 = dropout(relu(h1 W2 + b2)) ; logits = h2 W3 + b3
//     loss = mean_b (logsumexp(logits_b) - logits_b[label_b]) ; d3 = (softmax - onehot) / B
//   backward (what tf.gradients builds, :298-303)
//     gW3 = h2^T d3, gb3 = colsum d3, d2 = (d3 W3^T) . mask2
//     gW2 = h1^T d2, gb2 = colsum d2, d1 = (d2 W2^T) . mask1
//     gW1 = a0^T d1, gb1 = colsum d1, d0 = d1 W1^T          (d0 = gradient of the mean over filters, fed to conv2 bwd)
// a0 [B x d0] is the mean over the filters of the last conv layer (models_gcn.py:673), written by its epilogue.
//
// The head is ~0.6 GFLOP in seven dependent GEMM stages: at B = 512 it is launch- and latency-bound, not
// throughput-bound (round 1: 13 launches, 97 us).  Here one CTA per SM stays resident and walks six phases separated
// by grid barriers; every phase deals its 64x64 output tiles (K split where a phase has too few tiles) over all
// CTAs.  Plain fp32 FFMA (4x4 register tiles out of shared memory): exact fp32 products, no split passes, and the
// whole head needs ~8 us of FFMA issue.  All reductions run in a fixed order: results are bit-reproducible.
#include <cooperative_groups.h>

#include <algorithm>

#include "common.cuh"

namespace cg = cooperative_groups;

namespace gcnb {

#ifdef GCNB_TRACE
__device__ long long g_head_trace[32];
__device__ long long g_head_cta[160][16];  // every CTA's own clock at every trace point (per-SM clocks: use differences)
#define HTRACE(i) do { if (threadIdx.x == 0) { const long long c_ = clock64(); if (blockIdx.x == 0) g_head_trace[i] = c_; if (blockIdx.x < 160) g_head_cta[blockIdx.x][i] = c_; } } while (0)
#else
#define HTRACE(i) do { } while (0)
#endif

constexpr int HT = 256;         // threads per CTA
constexpr int TM = 64, TN = 64, TK = 32;
constexpr int TS = TM + 9;      // shared tile row stride (floats), 9 mod 32: the transposing stores of k-contiguous operands
                                // (32 lanes = 32 k, one column) hit 32 banks, the mma fragment loads (4 k x 8 columns) nearly so
constexpr int CTS = TM + 4;     // row stride of the accumulator hand-over tile (16-byte aligned rows)
constexpr int SK2 = 4;          // K split of h1 W2 (too few output tiles otherwise)
constexpr int SKW = 2;          // K (= batch) split of h1^T d2
constexpr int SKC = 128;        // k chunk of the narrow products
constexpr int SK3 = 8;          // batch split of h2^T d3 (16 column blocks alone would leave 130 CTAs waiting)
constexpr int SK1 = 4;          // batch split of a0^T d1 and K split of d1 W1^T

__host__ __device__ static inline int ceil_div_d(int a, int b) { return (a + b - 1) / b; }

struct TileSmem {
  float a[TK][TS];
  float b[TK][TS];
};

// Strided 2-D view of an operand in global memory: element (i, j) = p[i * si + j * sj].
struct View {
  const float* p;
  long long si, sj;
  __device__ __forceinline__ float at(int i, int j) const { return p[i * si + j * sj]; }
};

// One 64x64 output tile of op(A) op(B) over k in [k0, k1): acc[i][j] of thread (ty, tx) = C[m0 + 4 ty + i][n0 + 4 tx + j].
// Operands are strided views of global memory; AK / BK say which index is contiguous (so that the cooperative tile
// loads coalesce): AK: A(m, k) = A[m * lda + k], else A[k * lda + m];  BK: B(k, n) = B[n * ldb + k], else B[k * ldb + n].
// All per-element address arithmetic is hoisted out of the chunk loop (one pointer, one validity bit per element);
// the next chunk's 16 loads are in flight while the current one is multiplied.  Plain (coherent) loads: some operands
// were written earlier in this kernel.  The chunk loop runs on the tensor cores (3xTF32 mma.sync; the FFMA version it
// replaces was issue bound at 512 FFMA per thread and chunk).
__device__ __forceinline__ void split_hl(float v, uint32_t& hi, uint32_t& lo) {
  hi = __float_as_uint(v) & 0xffffe000u;            // what the tensor core keeps of an fp32 operand
  lo = __float_as_uint(v - __uint_as_float(hi));    // exact remainder
}
__device__ __forceinline__ void mma8(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};\n"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

template <bool AK, bool BK>
__device__ __forceinline__ void tile_gemm(TileSmem& sm, const float* A, int lda, const float* Bp,
                                          int ldb, int M, int N, int m0, int n0, int k0, int k1, float (&acc)[4][4]) {
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int lane = tid & 31, wid = tid >> 5, g8 = lane >> 2, t4 = lane & 3;
  const int mw = (wid & 3) * 16, nw = (wid >> 2) * 32;
  float c[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) c[i][j] = 0.f;
  // element i of this thread: A: (k = ak0 + i*AKS, m = am0 + i*AMS), B likewise
  const int ak0 = AK ? (tid & 31) : (tid >> 6), am0 = AK ? (tid >> 5) : (tid & 63);
  const int bk0 = BK ? (tid & 31) : (tid >> 6), bn0 = BK ? (tid >> 5) : (tid & 63);
  constexpr int AKS = AK ? 0 : 4, AMS = AK ? 8 : 0, BKS = BK ? 0 : 4, BNS = BK ? 8 : 0;
  const float* pa = AK ? A + (long long)(m0 + am0) * lda + ak0 : A + (long long)ak0 * lda + (m0 + am0);
  const float* pb = BK ? Bp + (long long)(n0 + bn0) * ldb + bk0 : Bp + (long long)bk0 * ldb + (n0 + bn0);
  const long long sa = AK ? (long long)AMS * lda : (long long)AKS * lda, sb = BK ? (long long)BNS * ldb : (long long)BKS * ldb;
  const long long ka = AK ? 1 : lda, kb = BK ? 1 : ldb;  // address step per unit of k
  uint32_t va = 0, vb = 0;                               // row / column validity of the 8 elements
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    va |= (m0 + am0 + i * AMS < M ? 1u : 0u) << i;
    vb |= (n0 + bn0 + i * BNS < N ? 1u : 0u) << i;
  }
  // two chunks of loads in flight (a tile is one CTA's whole phase: the chain of chunk loads is its critical path)
  float ra[8], rb[8], ra2[8], rb2[8];
  auto fetch = [&](int kc, float (&qa)[8], float (&qb)[8]) {
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      qa[i] = ((va >> i) & 1u) && kc + ak0 + i * AKS < k1 ? pa[kc * ka + i * sa] : 0.f;
      qb[i] = ((vb >> i) & 1u) && kc + bk0 + i * BKS < k1 ? pb[kc * kb + i * sb] : 0.f;
    }
  };
  fetch(k0, ra, rb);
  fetch(k0 + TK, ra2, rb2);  // (all zeros past k1)
  for (int kc = k0; kc < k1; kc += TK) {
    __syncthreads();  // the previous chunk has been consumed
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      sm.a[ak0 + i * AKS][am0 + i * AMS] = ra[i];
      sm.b[bk0 + i * BKS][bn0 + i * BNS] = rb[i];
    }
    __syncthreads();
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      ra[i] = ra2[i];
      rb[i] = rb2[i];
    }
    if (kc + 2 * TK < k1) fetch(kc + 2 * TK, ra2, rb2);
    // 3xTF32 on the tensor cores (mma.sync m16n8k8): warp w owns rows 16 (w & 3) .., columns 32 (w >> 2) .. of the tile.
    // Both operands are split by truncation (hi = top 19 bits, lo = exact remainder): the dropped lo*lo term and the
    // truncation of lo are ~2^-20 relative -- fp32-level products at a sixth of the FFMA issue slots.
#pragma unroll
    for (int ks = 0; ks < TK / 8; ++ks) {
      const int kb = ks * 8;
      uint32_t ah[4], al[4];
      split_hl(sm.a[kb + t4][mw + g8], ah[0], al[0]);
      split_hl(sm.a[kb + t4][mw + g8 + 8], ah[1], al[1]);
      split_hl(sm.a[kb + t4 + 4][mw + g8], ah[2], al[2]);
      split_hl(sm.a[kb + t4 + 4][mw + g8 + 8], ah[3], al[3]);
#pragma unroll
      for (int nt = 0; nt < 4; ++nt) {
        uint32_t bh0, bl0, bh1, bl1;
        split_hl(sm.b[kb + t4][nw + nt * 8 + g8], bh0, bl0);
        split_hl(sm.b[kb + t4 + 4][nw + nt * 8 + g8], bh1, bl1);
        mma8(c[nt], al, bh0, bh1);
        mma8(c[nt], ah, bl0, bl1);
        mma8(c[nt], ah, bh0, bh1);
      }
    }
  }
  __syncthreads();
  // accumulator fragments -> the 4 x 4 register tiles the phase epilogues are written for, through the tile buffer
  float(*ct)[CTS] = reinterpret_cast<float(*)[CTS]>(&sm);  // [TM][CTS] over the (contiguous) a and b tiles
  static_assert(sizeof(float) * TM * CTS <= sizeof(TileSmem), "hand-over tile must fit");
#pragma unroll
  for (int nt = 0; nt < 4; ++nt) {
    *reinterpret_cast<float2*>(&ct[mw + g8][nw + nt * 8 + 2 * t4]) = make_float2(c[nt][0], c[nt][1]);
    *reinterpret_cast<float2*>(&ct[mw + g8 + 8][nw + nt * 8 + 2 * t4]) = make_float2(c[nt][2], c[nt][3]);
  }
  __syncthreads();
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float4 v = *reinterpret_cast<const float4*>(&ct[ty * 4 + i][tx * 4]);
    acc[i][0] = v.x; acc[i][1] = v.y; acc[i][2] = v.z; acc[i][3] = v.w;
  }
  __syncthreads();
}

// Narrow products: out[j * soj + c * soc] = sum_k X(k, j) * Y(k, c) for j < Jv <= 16 and c < CY <= 32, k < Kd.
// Both operands are staged through shared memory in chunks of SKC k (cooperative loads, next chunk in flight while
// the current one is multiplied).  Thread (kq, jq, cg) owns a 4 x 2 block of outputs (j = 4 jq .., c = cg, cg + 16)
// for the k of its quarter (k = kq mod 4): one LDS.128 + two LDS per eight FMAs -- the first version, one output pair
// per thread, was bound by shared-memory wavefronts.  The four k-quarters are combined in a fixed order through
// shared memory at the end: bit-reproducible.  kfast: k is the contiguous index of both operands in memory (loads
// then run along k), else j / c are.  One copy of the code for its three users.
constexpr int SXS = 20;  // row stride of the staged X chunk (floats): 16-byte aligned rows
__device__ __noinline__ void skinny16(float* sm /* >= SKC*SXS + SKC*33 floats */, View X, int Jv, View Y, int CY, int Kd,
                                      bool kfast, float* out, long long soj, long long soc) {
  float(*xs)[SXS] = reinterpret_cast<float(*)[SXS]>(sm);
  float(*ys)[33] = reinterpret_cast<float(*)[33]>(sm + SKC * SXS);
  const int tid = threadIdx.x, kq = tid >> 6, jq = tid & 3, cg = (tid >> 2) & 15;
  constexpr int NX = SKC * 16 / HT, NY = SKC * 32 / HT;
  float rx[NX], ry[NY];
  auto fetch = [&](int k0) {
#pragma unroll
    for (int i = 0; i < NX; ++i) {
      const int e = i * HT + tid;
      const int kk = kfast ? (e & (SKC - 1)) : (e >> 4), j = kfast ? (e / SKC) : (e & 15);
      rx[i] = (k0 + kk < Kd && j < Jv) ? X.at(k0 + kk, j) : 0.f;
    }
#pragma unroll
    for (int i = 0; i < NY; ++i) {
      const int e = i * HT + tid;
      const int kk = kfast ? (e & (SKC - 1)) : (e >> 5), c = kfast ? (e / SKC) : (e & 31);
      ry[i] = (k0 + kk < Kd && c < CY) ? Y.at(k0 + kk, c) : 0.f;
    }
  };
  float acc[4][2];
#pragma unroll
  for (int i = 0; i < 4; ++i) acc[i][0] = acc[i][1] = 0.f;
  fetch(0);
  for (int k0 = 0; k0 < Kd; k0 += SKC) {
    __syncthreads();
#pragma unroll
    for (int i = 0; i < NX; ++i) {
      const int e = i * HT + tid;
      const int kk = kfast ? (e & (SKC - 1)) : (e >> 4), j = kfast ? (e / SKC) : (e & 15);
      xs[kk][j] = rx[i];
    }
#pragma unroll
    for (int i = 0; i < NY; ++i) {
      const int e = i * HT + tid;
      const int kk = kfast ? (e & (SKC - 1)) : (e >> 5), c = kfast ? (e / SKC) : (e & 31);
      ys[kk][c] = ry[i];
    }
    __syncthreads();
    if (k0 + SKC < Kd) fetch(k0 + SKC);
#pragma unroll 8
    for (int k = kq; k < SKC; k += 4) {
      const float4 x = *reinterpret_cast<const float4*>(&xs[k][jq * 4]);
      const float y0 = ys[k][cg], y1 = ys[k][cg + 16];
      acc[0][0] = fmaf(x.x, y0, acc[0][0]); acc[0][1] = fmaf(x.x, y1, acc[0][1]);
      acc[1][0] = fmaf(x.y, y0, acc[1][0]); acc[1][1] = fmaf(x.y, y1, acc[1][1]);
      acc[2][0] = fmaf(x.z, y0, acc[2][0]); acc[2][1] = fmaf(x.z, y1, acc[2][1]);
      acc[3][0] = fmaf(x.w, y0, acc[3][0]); acc[3][1] = fmaf(x.w, y1, acc[3][1]);
    }
  }
  __syncthreads();
  float* red = sm;  // [4 k-quarters][16 j][32 c]
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    red[(kq * 16 + jq * 4 + i) * 32 + cg] = acc[i][0];
    red[(kq * 16 + jq * 4 + i) * 32 + cg + 16] = acc[i][1];
  }
  __syncthreads();
  for (int o = tid; o < 16 * 32; o += HT) {
    const int j = o >> 5, c = o & 31;
    const float v = ((red[o] + red[512 + o]) + red[1024 + o]) + red[1536 + o];
    if (j < Jv && c < CY) out[j * soj + c * soc] = v;
  }
  __syncthreads();
}

// out[c] = sum_r X[r][c] for 32 columns c0..c0+31: 8 row slices x 32 columns, fixed-order combine.
__device__ __noinline__ void colsum32(float* red /* [8][32] */, const float* X, int ld, int cols, int c0, int R,
                                      float* __restrict__ out) {
  const int tid = threadIdx.x, cl = tid & 31, rs = tid >> 5;
  const int c = c0 + cl;
  float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
  if (c < cols) {
    int r = rs;
    for (; r + 24 < R; r += 32) {
      s0 += X[(long long)r * ld + c];
      s1 += X[(long long)(r + 8) * ld + c];
      s2 += X[(long long)(r + 16) * ld + c];
      s3 += X[(long long)(r + 24) * ld + c];
    }
    for (; r < R; r += 8) s0 += X[(long long)r * ld + c];
  }
  __syncthreads();
  red[rs * 32 + cl] = (s0 + s1) + (s2 + s3);
  __syncthreads();
  if (tid < 32 && c < cols) {
    float s = 0.f;
#pragma unroll
    for (int q = 0; q < 8; ++q) s += red[q * 32 + cl];
    out[c] = s;
  }
  __syncthreads();
}


__global__ void __launch_bounds__(HT, 1) k_head_step(const HeadParams P) {
  cg::grid_group grid = cg::this_grid();
  HTRACE(0);
  // one shared buffer, three views: the GEMM tiles, the staging of the narrow products, rows of h2 (+ W3)
  __shared__ __align__(16) float smem_f[16 * 16 * 33];
  static_assert(sizeof(TileSmem) <= sizeof(float) * 16 * 16 * 33, "tile view must fit");
  static_assert(SKC * SXS + SKC * 33 <= 16 * 16 * 33, "narrow-product staging must fit");
  TileSmem& sm = *reinterpret_cast<TileSmem*>(smem_f);
  float* red = smem_f;
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int nb = gridDim.x, bid = blockIdx.x;
  float acc[4][4];
  const int B = P.B, n0 = P.n0, n1 = P.n1, n2 = P.n2, C = P.C;
  const uint32_t key1 = dropout_key(P.seed1, P.state), key2 = dropout_key(P.seed2, P.state);
  const uint32_t thresh = dropout_threshold(P.keep);
  const int tmB = ceil_div_d(B, TM), tn1 = ceil_div_d(n1, TN), tn2 = ceil_div_d(n2, TN), tm1 = ceil_div_d(n1, TM);

  // ---- F1: h1 = dropout(relu(a0 W1 + b1)) ---------------------------------------------------------------------
  for (int u = bid; u < tmB * tn1; u += nb) {
    const int m0 = (u / tn1) * TM, c0 = (u % tn1) * TN;
    tile_gemm<true, false>(sm, P.a0, n0, P.W1, n1, B, n1, m0, c0, 0, n0, acc);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int m = m0 + ty * 4 + i;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int n = c0 + tx * 4 + j;
        if (m < B && n < n1) {
          float v = fmaxf(acc[i][j] + __ldg(P.b1 + n), 0.f);
          if (P.keep < 1.f) v = dropout_keeps((uint32_t)((long long)m * n1 + n), key1, thresh) ? v * P.inv_keep : 0.f;
          P.h1[(long long)m * n1 + n] = v;
        }
      }
    }
  }
  HTRACE(1);
  grid.sync();
  HTRACE(2);

  // ---- F2: partial sums of h1 W2, K split SK2 ways ---------------------------------------------------------------
  {
    const int kper = ceil_div_d(ceil_div_d(n1, SK2), TK) * TK;
    for (int u = bid; u < tmB * tn2 * SK2; u += nb) {
      const int sp = u % SK2, t = u / SK2;
      const int m0 = (t / tn2) * TM, c0 = (t % tn2) * TN;
      const int k0 = sp * kper, k1 = min(n1, k0 + kper);
      tile_gemm<true, false>(sm, P.h1, n1, P.W2, n2, B, n2, m0, c0, k0, k1, acc);
      float* dst = P.part2 + (long long)sp * B * n2;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int m = m0 + ty * 4 + i;
        const int n = c0 + tx * 4;
        if (m < B) {
          if (n + 3 < n2 && (n2 & 3) == 0) {
            *reinterpret_cast<float4*>(dst + (long long)m * n2 + n) = make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
          } else {
#pragma unroll
            for (int j = 0; j < 4; ++j)
              if (n + j < n2) dst[(long long)m * n2 + n + j] = acc[i][j];
          }
        }
      }
    }
  }
  HTRACE(3);
  grid.sync();
  HTRACE(4);

  // ---- F3: per row: h2 = dropout(relu(sum of partials + b2)), logits, cross-entropy, d3 ------------------------
  {
    const int warp = tid >> 5, lane = tid & 31;
    // Four rows at a time, two warps per row: hidden units summed from the partials, logits, cross-entropy.
    // Shared memory: four row buffers [hidden units | logits], then the logits weights when they fit (22 KB at 256 x 22).
    const int o_lg = (n2 + 31) & ~31;
    float* w3s = smem_f + 4 * (o_lg + 32);
    const bool w3_smem = (size_t)4 * (o_lg + 32) + (size_t)n2 * C <= (size_t)(16 * 16 * 33);
    const int q = warp >> 1, half = warp & 1, t64 = half * 32 + lane;  // row slot, thread index inside the warp pair
    if (w3_smem && bid * 4 < B) {
      for (int i0 = 0; i0 < n2 * C; i0 += HT * 8) {
        float v[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) v[u] = i0 + u * HT + tid < n2 * C ? __ldg(P.W3 + i0 + u * HT + tid) : 0.f;
#pragma unroll
        for (int u = 0; u < 8; ++u)
          if (i0 + u * HT + tid < n2 * C) w3s[i0 + u * HT + tid] = v[u];
      }
    }
    __syncthreads();
    for (int rb = bid * 4; rb < B; rb += nb * 4) {
      const int r = rb + q;
      float* hr = smem_f + q * (o_lg + 32);
      float* lgr = hr + o_lg;
      if (r < B) {
        for (int n = t64; n < n2; n += 64) {
          float v = __ldg(P.b2 + n);
#pragma unroll
          for (int sp = 0; sp < SK2; ++sp) v += P.part2[((long long)sp * B + r) * n2 + n];
          v = fmaxf(v, 0.f);
          if (P.keep < 1.f) v = dropout_keeps((uint32_t)((long long)r * n2 + n), key2, thresh) ? v * P.inv_keep : 0.f;
          hr[n] = v;
          P.h2[(long long)r * n2 + n] = v;
        }
      }
      __syncthreads();
      if (r < B) {
        for (int c = half; c < C; c += 2) {
          float sacc = 0.f;
          if (w3_smem) {
            for (int k = lane; k < n2; k += 32) sacc = fmaf(hr[k], w3s[k * C + c], sacc);
          } else {
            for (int k = lane; k < n2; k += 32) sacc = fmaf(hr[k], __ldg(P.W3 + (long long)k * C + c), sacc);
          }
#pragma unroll
          for (int d = 16; d > 0; d >>= 1) sacc += __shfl_xor_sync(0xffffffffu, sacc, d);
          if (lane == 0) {
            sacc += __ldg(P.b3 + c);
            lgr[c] = sacc;
            P.logits[(long long)r * C + c] = sacc;
          }
        }
      }
      __syncthreads();
      if (r < B && half == 0) {
        float mx = -INFINITY;
        for (int c = lane; c < C; c += 32) mx = fmaxf(mx, lgr[c]);
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, d));
        float se = 0.f;
        for (int c = lane; c < C; c += 32) se += expf(lgr[c] - mx);
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) se += __shfl_xor_sync(0xffffffffu, se, d);
        const float lse = mx + logf(se);
        const long long lab = P.labels[r];
        const bool ok = lab >= 0 && lab < C;  // a label outside [0, C) contributes no loss and no gradient
        const float scale = 1.f / (float)B;
        for (int c = lane; c < C; c += 32)
          P.d3[(long long)r * C + c] = ok ? (expf(lgr[c] - lse) - (c == (int)lab ? 1.f : 0.f)) * scale : 0.f;
        if (lane == 0) P.loss_rows[r] = ok ? lse - lgr[(int)lab] : 0.f;
      }
      __syncthreads();
    }
  }
  HTRACE(5);
  grid.sync();
  HTRACE(6);

  // ---- B1: gW3, gb3, d2 = (d3 W3^T) . mask2 ; mean loss ----------------------------------------------------------
  {
    const int uW3 = ceil_div_d(n2, 16) * SK3, uD2 = ceil_div_d(B * n2, HT * 4);
    for (int u = bid; u < uW3 + 1 + uD2; u += nb) {
      if (u < uW3) {
        // partial of gW3[j][c] = sum_r h2[r][j] d3[r][c] over one slice of the batch, 16 columns j
        const int j0 = (u / SK3) * 16, sp = u % SK3;
        const int rper = ceil_div_d(B, SK3), r0 = sp * rper, r1 = min(B, r0 + rper);
        skinny16(red, View{P.h2 + (long long)r0 * n2 + j0, n2, 1}, min(16, n2 - j0), View{P.d3 + (long long)r0 * C, C, 1}, C,
                 max(r1 - r0, 0), false, P.part3 + (long long)sp * n2 * C + (long long)j0 * C, C, 1);
      } else if (u == uW3) {
        colsum32(red, P.d3, C, C, 0, B, P.gb3);
        float s = 0.f;  // mean loss, fixed order
        for (int i = tid; i < B; i += HT) s += P.loss_rows[i];
        __syncthreads();
        red[tid] = s;
        __syncthreads();
        for (int d = HT / 2; d > 0; d >>= 1) {
          if (tid < d) red[tid] += red[tid + d];
          __syncthreads();
        }
        if (tid == 0) P.loss[0] = red[0] / (float)B;
        __syncthreads();
      } else {
        // d2[r][n] = mask2 * sum_c d3[r][c] W3[n][c]: both C-long rows in registers before the first FMA
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int o = ((u - uW3 - 1) * 4 + i) * HT + tid;
          if (o < B * n2) {
            const int r = o / n2, n = o - r * n2;
            float sacc = 0.f;
            if (P.h2[o] > 0.f) {
              const float* dr = P.d3 + (long long)r * C;
              const float* wr = P.W3 + (long long)n * C;
              float dv[32], wv[32];
#pragma unroll
              for (int c = 0; c < 32; ++c) {
                dv[c] = c < C ? dr[c] : 0.f;
                wv[c] = c < C ? __ldg(wr + c) : 0.f;
              }
#pragma unroll
              for (int c = 0; c < 32; ++c) sacc = fmaf(dv[c], wv[c], sacc);
              sacc *= P.inv_keep;
            }
            P.d2[o] = sacc;
          }
        }
      }
    }
  }
  HTRACE(7);
  grid.sync();
  HTRACE(8);
  if (bid == 0 && tid == 0 && P.state != nullptr && P.tick) {
    const float p1 = P.state[0] * P.beta1, p2 = P.state[1] * P.beta2;
    P.state[0] = p1;
    P.state[1] = p2;
    P.state[2] = P.lr * sqrtf(1.f - p2) / (1.f - p1);
    P.state[3] += 1.f;
  }

  // ---- B2: partial gW2 = h1^T d2 (batch split SKW ways), d1 = (d2 W2^T) . mask1, gb2 -----------------------------
  {
    const int uW = tm1 * tn2 * SKW, uD = tmB * tn1, uB = ceil_div_d(n2, 32), uR3 = ceil_div_d(n2 * C, HT * 4);
    const int bper = ceil_div_d(ceil_div_d(B, SKW), TK) * TK;
    for (int u = bid; u < uW + uD + uB + uR3; u += nb) {
      if (u >= uW + uD + uB) {  // gW3 = sum of the batch-slice partials of B1 (fixed order)
        float v[4][SK3];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int o = ((u - uW - uD - uB) * 4 + i) * HT + tid;
#pragma unroll
          for (int q = 0; q < SK3; ++q) v[i][q] = o < n2 * C ? P.part3[(long long)q * n2 * C + o] : 0.f;
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int o = ((u - uW - uD - uB) * 4 + i) * HT + tid;
          float sacc = v[i][0];
#pragma unroll
          for (int q = 1; q < SK3; ++q) sacc += v[i][q];
          if (o < n2 * C) P.gW3[o] = sacc;
        }
        continue;
      }
      if (u < uW) {
        const int sp = u % SKW, t = u / SKW;
        const int m0 = (t / tn2) * TM, c0 = (t % tn2) * TN;
        const int k0 = sp * bper, k1 = min(B, k0 + bper);
        tile_gemm<false, false>(sm, P.h1, n1, P.d2, n2, n1, n2, m0, c0, k0, k1, acc);
        float* dst = P.partW2 + (long long)sp * n1 * n2;
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const int m = m0 + ty * 4 + i, n = c0 + tx * 4 + j;
            if (m < n1 && n < n2) dst[(long long)m * n2 + n] = acc[i][j];
          }
      } else if (u < uW + uD) {
        const int t = u - uW;
        const int m0 = (t / tn1) * TM, c0 = (t % tn1) * TN;
        tile_gemm<true, true>(sm, P.d2, n2, P.W2, n2, B, n1, m0, c0, 0, n2, acc);
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const int m = m0 + ty * 4 + i, n = c0 + tx * 4 + j;
            if (m < B && n < n1)
              P.d1[(long long)m * n1 + n] = P.h1[(long long)m * n1 + n] > 0.f ? acc[i][j] * P.inv_keep : 0.f;
          }
      } else {
        colsum32(red, P.d2, n2, n2, (u - uW - uD) * 32, B, P.gb2);
      }
    }
  }
  HTRACE(9);
  grid.sync();
  HTRACE(10);

  // ---- B3: gW2 = sum of partials, gb1, slice partials of gW1 = a0^T d1 and of d0 = d1 W1^T ---------------------------
  {
    const int uS = ceil_div_d(n1 * n2, HT * 8), uW1 = ceil_div_d(n1, 16) * SK1, uB1 = ceil_div_d(n1, 32),
              uD0 = ceil_div_d(B, 16) * SK1;
    for (int u = bid; u < uS + uW1 + uB1 + uD0; u += nb) {
      if (u < uS) {
        float v[8][SKW];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const long long o = ((long long)u * 8 + i) * HT + tid;
#pragma unroll
          for (int q = 0; q < SKW; ++q) v[i][q] = o < (long long)n1 * n2 ? P.partW2[(long long)q * n1 * n2 + o] : 0.f;
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const long long o = ((long long)u * 8 + i) * HT + tid;
          float sacc = v[i][0];
#pragma unroll
          for (int q = 1; q < SKW; ++q) sacc += v[i][q];
          if (o < (long long)n1 * n2) P.gW2[o] = sacc;
        }
      } else if (u < uS + uW1) {
        // partial of gW1[m][n] = sum_r a0[r][m] d1[r][n] over one slice of the batch, 16 columns n
        const int t = u - uS, j0 = (t / SK1) * 16, sp = t % SK1;
        const int rper = ceil_div_d(B, SK1), r0 = sp * rper, r1 = min(B, r0 + rper);
        skinny16(red, View{P.d1 + (long long)r0 * n1 + j0, n1, 1}, min(16, n1 - j0), View{P.a0 + (long long)r0 * n0, n0, 1}, n0,
                 max(r1 - r0, 0), false, P.part1 + (long long)sp * n0 * n1 + j0, 1, n1);
      } else if (u < uS + uW1 + uB1) {
        colsum32(red, P.d1, n1, n1, (u - uS - uW1) * 32, B, P.gb1);
      } else {
        // partial of d0[r][m] = sum_k d1[r][k] W1[m][k] over one slice of k, 16 rows r
        const int t = u - uS - uW1 - uB1, r0 = (t / SK1) * 16, sp = t % SK1;
        const int kper = ceil_div_d(n1, SK1), k0 = sp * kper, k1 = min(n1, k0 + kper);
        skinny16(red, View{P.d1 + (long long)r0 * n1 + k0, 1, n1}, min(16, B - r0), View{P.W1 + k0, 1, n1}, n0, max(k1 - k0, 0),
                 true, P.part0 + (long long)sp * B * n0 + (long long)r0 * n0, n0, 1);
      }
    }
  }
  HTRACE(11);
  grid.sync();
  HTRACE(12);

  // ---- B4: gW1 and d0 = sums of their slice partials (fixed order) ---------------------------------------------------
  {
    const int nW = n0 * n1, nD = B * n0;
    for (int o = bid * HT + tid; o < nW + nD; o += nb * HT) {
      const float* src = o < nW ? P.part1 + o : P.part0 + (o - nW);
      const long long stride = o < nW ? nW : nD;
      float v[SK1];
#pragma unroll
      for (int q = 0; q < SK1; ++q) v[q] = src[q * stride];
      float sacc = v[0];
#pragma unroll
      for (int q = 1; q < SK1; ++q) sacc += v[q];
      if (o < nW) P.gW1[o] = sacc; else P.d0[o - nW] = sacc;
    }
  }
  HTRACE(13);
}


// ---------------------------------------------------------------------------------------------------------------
size_t head_step_workspace(int B, int n0, int n1, int n2, int C) {
  size_t f = (size_t)B * n1 * 2 /*h1, d1*/ + (size_t)B * n2 * 2 /*h2, d2*/ + (size_t)B * C /*d3*/ +
             (size_t)SK2 * B * n2 /*part2*/ + (size_t)SKW * n1 * n2 /*partW2*/ + (size_t)B /*loss rows*/ +
             (size_t)SK3 * n2 * C /*part3*/ + (size_t)SK1 * n0 * n1 /*part1*/ + (size_t)SK1 * B * n0 /*part0*/;
  return f * sizeof(float) + 16 * 256;
}

bool head_step_supported(int B, int n0, int n1, int n2, int C) {
  return B >= 1 && n0 >= 1 && n0 <= 32 && C >= 1 && C <= 32 && n1 >= 1 && n2 >= 1 && n2 <= 2048;
}

int head_step(const HeadParams& P0, Workspace& ws, cudaStream_t st) {
  HeadParams P = P0;
  const int B = P.B, n1 = P.n1, n2 = P.n2, C = P.C;
  P.h1 = ws.take<float>((size_t)B * n1);
  P.d1 = ws.take<float>((size_t)B * n1);
  P.h2 = ws.take<float>((size_t)B * n2);
  P.d2 = ws.take<float>((size_t)B * n2);
  P.d3 = ws.take<float>((size_t)B * C);
  P.part2 = ws.take<float>((size_t)SK2 * B * n2);
  P.partW2 = ws.take<float>((size_t)SKW * n1 * n2);
  P.loss_rows = ws.take<float>((size_t)B);
  P.part3 = ws.take<float>((size_t)SK3 * n2 * C);
  P.part1 = ws.take<float>((size_t)SK1 * P.n0 * n1);
  P.part0 = ws.take<float>((size_t)SK1 * B * P.n0);
  if (!P.loss_rows || !P.part3 || !P.part1 || !P.part0) {
    set_error("gcnb_head_step_f32: workspace too small");
    return GCNB_ERR_WORKSPACE;
  }
  DeviceInfo di;
  int rc = device_info(&di);
  if (rc) return rc;
  int per_sm = 0;
  GCNB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_head_step, HT, 0));
  if (per_sm < 1) {
    set_error("gcnb_head_step_f32: the kernel does not fit on an SM");
    return GCNB_ERR_CUDA;
  }
  // one CTA per SM: every phase has at most ~150 work units, and two units on one SM while another SM idles lose
  // more than the extra warps hide (measured: 83 us with two CTAs per SM, 67 us with one)
  const int grid = di.sm_count;
  void* args[] = {(void*)&P};
  GCNB_CUDA(cudaLaunchCooperativeKernel((const void*)k_head_step, dim3(grid), dim3(HT), args, 0, st));
  GCNB_LAUNCH_CHECK("k_head_step");
  return GCNB_OK;
}

}  // namespace gcnb

using namespace gcnb;

extern "C" {

size_t gcnb_head_step_workspace_bytes(int B, int n0, int n1, int n2, int C) {
  return head_step_supported(B, n0, n1, n2, C) ? head_step_workspace(B, n0, n1, n2, C) : 0;
}

int gcnb_head_step_f32(const float* a0, const int64_t* labels, const float* W1, const float* b1, const float* W2,
                       const float* b2, const float* W3, const float* b3, float* logits, float* loss, float* gW1,
                       float* gb1, float* gW2, float* gb2, float* gW3, float* gb3, float* d0, int B, int n0, int n1,
                       int n2, int C, float keep, unsigned seed1, unsigned seed2, float* adam_state, float lr,
                       float beta1, float beta2, int tick, void* workspace, size_t workspace_bytes,
                       gcnb_stream_t stream) {
  GCNB_REQUIRE(head_step_supported(B, n0, n1, n2, C),
               "gcnb_head_step_f32: unsupported sizes B=%d widths %d-%d-%d-%d (needs n0 <= 32, C <= 32, n2 <= 2048)", B, n0,
               n1, n2, C);
  GCNB_REQUIRE(a0 && labels && W1 && b1 && W2 && b2 && W3 && b3 && logits && loss && gW1 && gb1 && gW2 && gb2 && gW3 &&
                   gb3 && d0,
               "gcnb_head_step_f32: NULL argument");
  GCNB_REQUIRE(keep > 0.f && keep <= 1.f, "gcnb_head_step_f32: keep probability must be in (0, 1] (got %g)", (double)keep);
  HeadParams P{};
  P.a0 = a0; P.labels = reinterpret_cast<const long long*>(labels);
  P.W1 = W1; P.b1 = b1; P.W2 = W2; P.b2 = b2; P.W3 = W3; P.b3 = b3;
  P.logits = logits; P.loss = loss;
  P.gW1 = gW1; P.gb1 = gb1; P.gW2 = gW2; P.gb2 = gb2; P.gW3 = gW3; P.gb3 = gb3; P.d0 = d0;
  P.B = B; P.n0 = n0; P.n1 = n1; P.n2 = n2; P.C = C;
  P.keep = keep; P.inv_keep = 1.f / keep; P.seed1 = seed1; P.seed2 = seed2;
  P.state = adam_state; P.lr = lr; P.beta1 = beta1; P.beta2 = beta2; P.tick = tick;
  Workspace ws(workspace, workspace_bytes);
  return head_step(P, ws, static_cast<cudaStream_t>(stream));
}

}  // extern "C"

#ifdef GCNB_TRACE
extern "C" __attribute__((visibility("default"))) int gcnb_debug_read_head_cta(long long* out) {
  return (int)cudaMemcpyFromSymbol(out, gcnb::g_head_cta, sizeof(long long) * 160 * 16);
}
extern "C" __attribute__((visibility("default"))) int gcnb_debug_read_head_trace(long long* out) {
  return (int)cudaMemcpyFromSymbol(out, gcnb::g_head_trace, sizeof(long long) * 32);
}
#endif
