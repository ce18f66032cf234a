// Fused ChebyNet forward for graphs that fit in shared memory:
//   (perm gather) -> T_k(L~) recursion -> contraction with the taps -> bias -> ReLU -> max-pool
// in ONE kernel: x is read from HBM once, y (and the arg-max bytes) written once; the K-stack, the
// layout transposes and the pre-pool activation of the reference (models_gcn.py:598-617, 619-639)
// never exist in memory.  See fused_common.cuh for the CTA layout.
#include <algorithm>
#include <cmath>

#include "fused_common.cuh"

namespace gcnb {

struct FwdParams {
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
  float* xstack;  // nullable: X_k for all k as [K][B][M][FP] (training: lets the weight gradient skip the recursion)
  float* y_mean;  // nullable: mean over the filters of the pooled output, [B][M/p] (models_gcn.py:673 fused)
  uint8_t* argmax;
  int B, Fin, Fout, K, p, bias_mode, relu;
  TileGeom g;
  int ntiles;
  int off_wfrag, off_slab;  // byte offsets into dynamic smem (operator image at 0)
  int off_stage;            // raw staging buffer for the TMA bulk prefetch of the next tile (0 = none)
  int off_misc;             // int src_row[Mpad] (gather table, -1 = zero row) followed by float bias_f[64]
  int log2p;
};

// register-heavy instances (many accumulator fragments) run with at most 16 warps
template <int NT, int SLOTS>
__global__ void __launch_bounds__((SLOTS * NT > 8) ? 512 : 896, 1) k_cheb_fwd_fused(const FwdParams P) {
  extern __shared__ __align__(16) unsigned char smem[];
  const TileGeom& G = P.g;
  OperatorSmem op;
  op.carve(smem, G.Mpad, P.nnz);
  float4* wfrag = reinterpret_cast<float4*>(smem + P.off_wfrag);
  unsigned char* slabA = smem + P.off_slab;
  unsigned char* slabB = slabA + (size_t)G.Mpad * G.RS * 4;

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int g = lane >> 2, t = lane & 3;
  const int rw = warp % G.RW, sg = warp / G.RW;
  const int RS = G.RS, FP = G.FP, KS = G.KS;

  // ---- TMA bulk prefetch of the tile's raw windows (contiguous in HBM) into a staging buffer ----------
  const bool staged = P.off_stage != 0;
  float* stage = reinterpret_cast<float*>(smem + P.off_stage);
  uint64_t* mbar = reinterpret_cast<uint64_t*>(smem + P.off_stage - 16);
  const int per_sample = P.M_in * P.Fin;
  uint32_t phase = 0;
  if (staged && tid == 0) {
    mbar_init(mbar, 1);
    const int nb = min(G.S, P.B - (int)blockIdx.x * G.S);
    const uint32_t bytes = (uint32_t)nb * per_sample * 4u;
    mbar_expect_tx(mbar, bytes);
    bulk_g2s(stage, P.x + (long long)blockIdx.x * G.S * per_sample, bytes, mbar);
  }

  // ---- once per CTA: operator image and the filter taps as TF32 hi/lo B-fragments --------------------
  build_operator(P.rowptr, P.col, P.val, G.M, G.Mpad, P.nnz, RS, op);
  for (int idx = tid; idx < P.K * KS * NT * 32; idx += blockDim.x) {
    const int ln = idx & 31, nt = (idx >> 5) % NT, ks = (idx / (32 * NT)) % KS, k = idx / (32 * NT * KS);
    const int gg = ln >> 2, tt = ln & 3;
    const int o = nt * 8 + gg, f0 = ks * 8 + tt, f1 = f0 + 4;
    float w0 = 0.f, w1 = 0.f;
    if (o < P.Fout) {
      if (f0 < P.Fin) w0 = __ldg(P.W + ((long long)f0 * P.K + k) * P.Fout + o);
      if (f1 < P.Fin) w1 = __ldg(P.W + ((long long)f1 * P.K + k) * P.Fout + o);
    }
    uint32_t h0, l0, h1, l1;
    split_tf32(w0, h0, l0);
    split_tf32(w1, h1, l1);
    wfrag[idx] = make_float4(__uint_as_float(h0), __uint_as_float(h1), __uint_as_float(l0), __uint_as_float(l1));
  }

  int* src_row = reinterpret_cast<int*>(smem + P.off_misc);
  float* bias_f = reinterpret_cast<float*>(src_row + G.Mpad);
  for (int m = tid; m < G.Mpad; m += blockDim.x) {
    int src = -1;
    if (m < G.M) {
      src = P.perm ? __ldg(P.perm + m) : m;
      if (src >= P.M_in) src = -1;  // fake vertex: stays zero (coarsening.py:260-264)
    }
    src_row[m] = src;
  }
  for (int o = tid; o < 64; o += blockDim.x)
    bias_f[o] = (P.bias_mode == GCNB_BIAS_PER_FILTER && o < P.Fout) ? __ldg(P.bias + o) : 0.f;

  const int col_byte = sg * G.WS * FP * 4;  // first column of this warp's sample group
  const int Mo = G.M / P.p;
  // loader geometry: FP is a power of two; 32/FP rows per warp instruction
  const int fp_shift = FP == 8 ? 3 : (FP == 16 ? 4 : 5);
  const int lrow = lane >> fp_shift, lf = lane & (FP - 1), rows_per_instr = 32 >> fp_shift;
  const int nwarps = blockDim.x >> 5;

  for (int tile = blockIdx.x; tile < P.ntiles; tile += gridDim.x) {
    const int b0 = tile * G.S;
    __syncthreads();  // previous tile fully consumed (also orders the one-time setup above)
    // ---- x (gathered through perm) into slab A: column s*FP + f of row m ------------------------------
    if (staged) mbar_wait(mbar, phase);  // the bulk copy of this tile has landed
    for (int s = 0; s < G.S; ++s) {
      const int b = b0 + s;
      const float* xb = staged ? stage + s * per_sample : P.x + (long long)b * per_sample;
      for (int m = warp * rows_per_instr + lrow; m < G.Mpad; m += nwarps * rows_per_instr) {
        float v = 0.f;
        const int src = src_row[m];
        if (b < P.B && src >= 0 && lf < P.Fin) v = staged ? xb[src * P.Fin + lf] : __ldg(xb + (long long)src * P.Fin + lf);
        reinterpret_cast<float*>(slabA)[m * RS + s * FP + lf] = v;
      }
    }
    __syncthreads();
    if (staged) {  // staging buffer is free again: fetch the next tile while this one is computed
      phase ^= 1;
      const int nt_ = tile + gridDim.x;
      if (tid == 0 && nt_ < P.ntiles) {
        const int nb = min(G.S, P.B - nt_ * G.S);
        const uint32_t bytes = (uint32_t)nb * per_sample * 4u;
        mbar_expect_tx(mbar, bytes);
        bulk_g2s(stage, P.x + (long long)nt_ * G.S * per_sample, bytes, mbar);
      }
    }

    float acc[SLOTS][NT][4];
#pragma unroll
    for (int a = 0; a < SLOTS; ++a)
#pragma unroll
      for (int n = 0; n < NT; ++n)
#pragma unroll
        for (int c = 0; c < 4; ++c) acc[a][n][c] = 0.f;

    // Contraction of the warp's own row tiles of X_k (in slab `cur`) with the taps of order k.
    auto contract = [&](int k, const unsigned char* cur) {
      const float4* wk = wfrag + (size_t)k * KS * NT * 32 + lane;
      const float* curf = reinterpret_cast<const float*>(cur) + g * RS + sg * G.WS * FP + t;
      for (int ks = 0; ks < KS; ++ks) {
        uint32_t ah[SLOTS][4], al[SLOTS][4];
#pragma unroll
        for (int a = 0; a < SLOTS; ++a) {
          const int tt = a / G.WS, s = a - tt * G.WS;
          const int rt = rw + tt * G.RW;
          if (a < G.TPW * G.WS && rt < G.RT) {
            const float* base = curf + rt * 16 * RS + s * FP + ks * 8;
            split_trunc(base[0], ah[a][0], al[a][0]);
            split_trunc(base[8 * RS], ah[a][1], al[a][1]);
            split_trunc(base[4], ah[a][2], al[a][2]);
            split_trunc(base[8 * RS + 4], ah[a][3], al[a][3]);
          } else {
#pragma unroll
            for (int c = 0; c < 4; ++c) ah[a][c] = al[a][c] = 0u;
          }
        }
#pragma unroll
        for (int n = 0; n < NT; ++n) {
          const float4 w = wk[(ks * NT + n) * 32];
          const uint32_t bh0 = __float_as_uint(w.x), bh1 = __float_as_uint(w.y);
          const uint32_t bl0 = __float_as_uint(w.z), bl1 = __float_as_uint(w.w);
#pragma unroll
          for (int a = 0; a < SLOTS; ++a) mma_3xtf32(acc[a][n], ah[a], al[a], bh0, bh1, bl0, bl1);
        }
      }
    };

    // Optional: keep the basis for the backward pass.  X_k sits untouched in its slab during step k+1, so each warp
    // streams its share of rows out at the start of that step (no extra barrier).
    auto spill = [&](int k, const unsigned char* slab) {  // each sample group streams out its own columns
      if (P.xstack == nullptr) return;
      const int q4 = FP >> 2;  // float4 per (row, sample)
      const int per_row = G.WS * q4;
      const int gthreads = G.RW * 32, gtid = tid - sg * gthreads;
      for (int idx = gtid; idx < G.M * per_row; idx += gthreads) {
        const int m = idx / per_row, rem = idx - m * per_row;
        const int s = sg * G.WS + rem / q4, q = rem % q4;
        const int b = b0 + s;
        if (b >= P.B) continue;
        const float4 v = *reinterpret_cast<const float4*>(slab + ((size_t)m * RS + s * FP + 4 * q) * 4);
        *reinterpret_cast<float4*>(P.xstack + (((size_t)k * P.B + b) * G.M + m) * FP + 4 * q) = v;
      }
    };

    // Step k: the sparse step that produces X_k (shared-memory / FFMA pipes) and the contraction of X_{k-1} (tensor
    // pipe) are independent -- both only read X_{k-1}.  Odd warps run them in one order, even warps in the other,
    // so at any time about half of the CTA feeds each pipe.  One barrier per order.
    for (int k = 1; k < P.K; ++k) {
      unsigned char* cur = (k & 1) ? slabB : slabA;         // receives X_k (holds X_{k-2})
      const unsigned char* prev = (k & 1) ? slabA : slabB;  // X_{k-1}
      spill(k - 1, prev);
      if (warp & 1) contract(k - 1, prev);
      spmm_dispatch(G.LPR, op, prev, cur, G.Mpad, col_byte, rw, G.RW, k == 1 ? 1.f : 2.f, k > 1);
      if (!(warp & 1)) contract(k - 1, prev);
      group_barrier(sg, G.RW * 32);  // X_k complete for this sample group's columns
    }
    spill(P.K - 1, ((P.K - 1) & 1) ? slabB : slabA);
    contract(P.K - 1, ((P.K - 1) & 1) ? slabB : slabA);

    // ---- epilogue: bias, ReLU, max-pool over p consecutive vertices (first maximum wins), store -------------
    // The accumulator fragments of one (row tile, sample) go through the warp's own 16 rows of the slab that is
    // no longer needed (X_{K-2}); then lane = filter: p values per pooled row are read back conflict free, the
    // pooled row is stored as one coalesced 128-byte line (arg-max bytes: 32 bytes).  Only __syncwarp is needed.
    {
      float* fs = reinterpret_cast<float*>(((P.K - 1) & 1) ? slabA : slabB);
#pragma unroll
      for (int a = 0; a < SLOTS; ++a) {
        const int tt = a / G.WS, s = a - tt * G.WS;
        const int rt = rw + tt * G.RW;
        const int b = b0 + sg * G.WS + s;
        const bool live = (a < G.TPW * G.WS) && rt < G.RT && b < P.B;  // warp-uniform
        if (!live) continue;
        // own 16 rows, own column range (warps of other sample groups share the rows): CW = WS*FP >= 32 columns
        float* tile_s = fs + (size_t)rt * 16 * RS + sg * G.WS * FP;
#pragma unroll
        for (int c0 = 0; c0 < NT; c0 += 4) {  // 32 filters at a time
          __syncwarp();
#pragma unroll
          for (int n = c0; n < c0 + 4 && n < NT; ++n) {
            *reinterpret_cast<float2*>(tile_s + g * RS + (n - c0) * 8 + 2 * t) = make_float2(acc[a][n][0], acc[a][n][1]);
            *reinterpret_cast<float2*>(tile_s + (g + 8) * RS + (n - c0) * 8 + 2 * t) = make_float2(acc[a][n][2], acc[a][n][3]);
          }
          __syncwarp();
          const int o = c0 * 8 + lane;
          const bool valid = o < P.Fout && lane < (NT - c0) * 8;
          const float bf = valid ? bias_f[o] : 0.f;
          for (int j = 0; j < (16 >> P.log2p); ++j) {
            const int r0 = rt * 16 + (j << P.log2p);
            if (r0 >= G.M) break;  // warp-uniform
            float best = -INFINITY;
            int bi = 0;
            if (valid) {
              for (int i = 0; i < P.p; ++i) {
                float v = tile_s[((j << P.log2p) + i) * RS + lane] + bf;
                if (P.bias_mode == GCNB_BIAS_PER_VERTEX) v += __ldg(P.bias + (long long)(r0 + i) * P.Fout + o);
                if (P.relu) v = fmaxf(v, 0.f);
                if (v > best) {  // strict: the first maximum keeps the slot
                  best = v;
                  bi = i;
                }
              }
              const long long oidx = ((long long)b * Mo + (r0 >> P.log2p)) * P.Fout + o;
              P.y[oidx] = best;
              if (P.argmax) P.argmax[oidx] = (uint8_t)bi;
            }
            if (P.y_mean != nullptr) {  // Fout <= 32 (one chunk): fixed-order shuffle tree over the filters
              float sm = valid ? best : 0.f;
#pragma unroll
              for (int d = 16; d > 0; d >>= 1) sm += __shfl_xor_sync(0xffffffffu, sm, d);
              if (lane == 0) P.y_mean[(long long)b * Mo + (r0 >> P.log2p)] = sm / (float)P.Fout;
            }
          }
        }
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// host side: geometry, eligibility, launch
// ------------------------------------------------------------------------------------------------
static const size_t kSmemBudget = 225 * 1024;

struct FwdPlan {
  bool ok;
  TileGeom g;
  int NT, SLOTS;
  size_t smem;
  int off_wfrag, off_slab, off_stage, off_misc;
  bool staged;
};

// M_in: vertices of the raw input (differs from M when the permutation gather is fused in).
static FwdPlan plan_fwd(const LayerShape& s, int M_in, bool x_aligned16) {
  FwdPlan pl;
  pl.ok = false;
  pl.staged = false;
  TileGeom& g = pl.g;
  if (s.Fin < 1 || s.Fin > 32 || s.Fout < 1 || s.Fout > 64) return pl;
  if (s.p > 16 || s.M % s.p != 0) return pl;
  g.M = s.M;
  g.Mpad = round_up(s.M, 16);
  g.RT = g.Mpad / 16;
  g.FP = s.Fin <= 8 ? 8 : (s.Fin <= 16 ? 16 : 32);
  g.KS = g.FP / 8;
  pl.NT = s.Fout <= 16 ? 2 : (s.Fout <= 32 ? 4 : 8);
  const size_t misc = (size_t)g.Mpad * 4 + 64 * 4;
  const size_t fixed = operator_smem_bytes(g.Mpad, s.nnz) + (size_t)s.K * g.KS * pl.NT * 32 * 16 + misc;
  // Candidates: WS samples per warp (CW = WS*FP columns in {32,64,128}) x SG sample groups.
  // Prefer the configuration with the fewest shared-memory wavefronts per nonzero (large CW), subject to
  // registers (SLOTS*NT accumulator fragments), warps (<= 28, or <= 16 for heavy instances) and smem.
  double best_score = -1;
  for (int ws = 32 / g.FP; ws * g.FP <= 128; ws *= 2) {
    for (int sgn = 1; sgn <= 8; ++sgn) {
      const int S = ws * sgn;
      if (S > s.B && !(ws == 32 / g.FP && sgn == 1)) continue;
      const int RS = S * g.FP + 4;
      size_t need = fixed + 2 * (size_t)g.Mpad * RS * 4;
      if (need > kSmemBudget) continue;
      // staging buffer for the bulk prefetch: only when a window is a multiple of 16 bytes and it fits
      const size_t stage_bytes = 16 + (size_t)S * M_in * s.Fin * 4;
      const bool can_stage = x_aligned16 && ((long long)M_in * s.Fin) % 4 == 0 && need + stage_bytes <= kSmemBudget;
      if (can_stage) need += stage_bytes;
      for (int heavy = 0; heavy < 2; ++heavy) {
        const int maxw = heavy ? 16 : 28;
        int rwn = std::min(g.RT, maxw / sgn);
        if (rwn < 1) continue;
        const int tpw = ceil_div(g.RT, rwn);
        rwn = ceil_div(g.RT, tpw);
        const int slots = tpw * ws;
        const int SL = slots <= 1 ? 1 : (slots <= 2 ? 2 : 4);
        if (slots > 4) continue;
        if (!heavy && SL * pl.NT > 8) continue;
        if (heavy && SL * pl.NT > 16) continue;
        const int nw = rwn * sgn;
        // wavefronts per nonzero per 32 columns: (1 entry + CW/32 data) / (CW/32); fewer is better;
        // penalise low warp counts (latency hiding) and wasted tile rounds over the SMs
        const double cw32 = ws * g.FP / 32.0;
        const double wf = (1.0 + cw32) / cw32;
        const double occ = std::min(1.0, nw / 12.0);
        const int tiles = ceil_div(s.B, S);
        const double rounds = std::ceil(tiles / 148.0);
        const double eff = tiles / (rounds * 148.0);
        const double score = occ * std::max(eff, 0.05) / wf * (can_stage ? 1.0 : 0.85);
        if (score > best_score) {
          best_score = score;
          g.WS = ws; g.SG = sgn; g.S = S; g.RS = RS; g.RW = rwn; g.TPW = tpw; g.nwarps = nw;
          g.LPR = ws * g.FP / 4;
          pl.SLOTS = SL;
          pl.smem = need;
          pl.staged = can_stage;
        }
        break;  // the light variant fits: do not consider the heavy one for the same (ws, sgn)
      }
    }
  }
  if (best_score < 0) return pl;
  pl.off_wfrag = (int)operator_smem_bytes(g.Mpad, s.nnz);
  pl.off_misc = pl.off_wfrag + s.K * g.KS * pl.NT * 32 * 16;
  pl.off_slab = pl.off_misc + (int)misc;
  pl.off_stage = pl.staged ? pl.off_slab + 2 * g.Mpad * g.RS * 4 + 16 : 0;
  pl.ok = true;
  return pl;
}

bool fused_fwd_supported(const LayerShape& s) { return plan_fwd(s, s.M, false).ok; }

template <int NT, int SLOTS>
static int launch_fwd(const FwdParams& P, const FwdPlan& pl, cudaStream_t st) {
  auto kern = k_cheb_fwd_fused<NT, SLOTS>;
  GCNB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.smem));
  DeviceInfo di;
  int rc = device_info(&di);
  if (rc) return rc;
  const int grid = std::min(P.ntiles, di.sm_count);
  kern<<<grid, pl.g.nwarps * 32, pl.smem, st>>>(P);
  GCNB_LAUNCH_CHECK("k_cheb_fwd_fused");
  return GCNB_OK;
}

int fused_cheb_fwd(const float* x, const int32_t* perm, int M_in, const gcnb_csr& L, const float* W,
                   const float* bias, float* y, uint8_t* argmax, float* y_mean, float* xstack, const LayerShape& s,
                   int bias_mode, int relu, Workspace& ws, cudaStream_t st) {
  (void)ws;
  const FwdPlan pl = plan_fwd(s, M_in, (reinterpret_cast<uintptr_t>(x) & 15) == 0);
  if (!pl.ok) {
    set_error("fused forward does not support this shape");
    return GCNB_ERR_INVALID;
  }
  FwdParams P;
  P.x = x; P.perm = perm; P.M_in = M_in;
  P.rowptr = L.rowptr; P.col = L.col; P.val = L.val; P.nnz = L.nnz;
  P.W = W; P.bias = bias; P.y = y; P.argmax = argmax; P.y_mean = s.Fout <= 32 ? y_mean : nullptr;
  P.xstack = xstack;
  P.B = s.B; P.Fin = s.Fin; P.Fout = s.Fout; P.K = s.K; P.p = s.p; P.bias_mode = bias_mode; P.relu = relu;
  P.g = pl.g;
  P.ntiles = ceil_div(s.B, pl.g.S);
  P.off_wfrag = pl.off_wfrag; P.off_slab = pl.off_slab; P.off_stage = pl.off_stage; P.off_misc = pl.off_misc;
  P.log2p = 0;
  while ((1 << P.log2p) < s.p) ++P.log2p;
#define GCNB_FWD_CASE(nt, sl) \
  if (pl.NT == nt && pl.SLOTS == sl) return launch_fwd<nt, sl>(P, pl, st);
  GCNB_FWD_CASE(2, 1) GCNB_FWD_CASE(2, 2) GCNB_FWD_CASE(2, 4)
  GCNB_FWD_CASE(4, 1) GCNB_FWD_CASE(4, 2) GCNB_FWD_CASE(4, 4)
  GCNB_FWD_CASE(8, 1) GCNB_FWD_CASE(8, 2)
#undef GCNB_FWD_CASE
  set_error("fused forward: no kernel instance for NT=%d SLOTS=%d", pl.NT, pl.SLOTS);
  return GCNB_ERR_INVALID;
}

}  // namespace gcnb
