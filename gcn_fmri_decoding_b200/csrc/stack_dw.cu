// Weight / bias gradient of the ChebyNet layer from a saved Chebyshev basis (training, first layer).
//
// When the forward pass kept X_k for all k (`xstack`, [K][B*M][FP]), the weight gradient
//     dW[f*K+k][o] = sum_{rows} X_k[row][f] * dZ[row][o],        rows = (sample, vertex)
// needs no recursion at all: it is one tall-skinny GEMM with the rows as the reduction dimension, streamed once from
// HBM.  That trades K*|x| bytes of extra traffic (cheap at 6+ TB/s) for the shared-memory-bound recomputation of the
// basis (measured 3x slower for the 400-vertex layer).  Each CTA walks chunks of 128 rows: the X tiles arrive by
// cp.async into a double buffer, dZ (MaxPoolGrad o ReluGrad of dy) is rebuilt per chunk from the pooled tensors, the
// contraction runs on the tensor cores (3xTF32 mma.sync, accumulators live in registers for the whole kernel), and
// the result is reduced warps -> CTA -> k_dw_from_partials in a fixed order (no float atomics).
#include <algorithm>

#include "fused_common.cuh"

namespace gcnb {


struct StackDwParams {
  const float* xstack;
  const float* y;
  const uint8_t* argmax;
  const float* dy;
  float* dw_part;
  float* db_part;  // nullable
  long long R;     // B*M rows
  int B, M, Mo, Fout, FoP, FP, p, log2p, relu, dy_is_mean;
  int CR, SX, SZ, nchunks;
  int NS;  // TMA stages for the X tiles
};

__device__ __forceinline__ void cp_async16(void* dst, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}

template <int K, int MT, int NT>
// light instances (<= 20 accumulator fragments) run two CTAs per SM: one CTA's loads hide behind the other's MMAs
__global__ void __launch_bounds__(256, (K * MT * NT > 20) ? 1 : 2) k_dw_from_stack(const StackDwParams P) {
  extern __shared__ __align__(16) unsigned char smem[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int g = lane >> 2, t = lane & 3;
  const int CR = P.CR, SX = P.SX, SZ = P.SZ, FP = P.FP, NS = P.NS;
  // smem: NS stages of K dense X tiles [CR][FP] (filled by TMA bulk copies), two dZ tiles [CR][SZ], NS mbarriers
  // stage = K dense X tiles [CR][FP] + the raw pooled rows of the chunk (dy, y, arg-max), all filled by TMA bulk copies
  const int cpr = CR >> P.log2p;  // pooled rows per chunk
  const size_t xbytes = (size_t)K * CR * SX * 4;
  const size_t rawf = (size_t)cpr * P.Fout * 4;                      // dy / y tile (dy: cpr floats in mean form)
  const size_t rawa = ((size_t)cpr * P.Fout + 15) / 16 * 16;         // arg-max tile
  const size_t sbytes = xbytes + 2 * rawf + rawa;                    // multiple of 16
  float* Zs = reinterpret_cast<float*>(smem + NS * sbytes);          // expanded dZ tile [CR][SZ]
  uint64_t* mbar = reinterpret_cast<uint64_t*>(smem + NS * sbytes + (size_t)CR * SZ * 4);
  constexpr int NCH = MT * NT / 2;

  float acc[K][MT][NT][4];
#pragma unroll
  for (int k = 0; k < K; ++k)
#pragma unroll
    for (int m = 0; m < MT; ++m)
#pragma unroll
      for (int n = 0; n < NT; ++n)
#pragma unroll
        for (int c = 0; c < 4; ++c) acc[k][m][n][c] = 0.f;
  float dbacc = 0.f;  // column o = tid % FoP of dZ (FoP divides 256)

  if (tid == 0)
    for (int s = 0; s < NS; ++s) mbar_init(mbar + s, 1);
  __syncthreads();

  const long long npr = P.R >> P.log2p;
  const bool has_am = P.argmax != nullptr && P.p > 1;
  // bulk copies per chunk: for every order k the rows of a chunk are contiguous in HBM, and so are its pooled rows
  auto issue = [&](int chunk, int stage) {
    const long long r0 = (long long)chunk * CR;
    const int rows = (int)min((long long)CR, P.R - r0);
    unsigned char* st = smem + (size_t)stage * sbytes;
    float* xs = reinterpret_cast<float*>(st);
    if (rows < CR)  // tail chunk: rows past the end must read as zero (their dZ rows are zero, but 0 * garbage may be NaN)
      for (int i = tid; i < K * (CR - rows) * FP; i += 256) {
        const int k = i / ((CR - rows) * FP), rem = i - k * (CR - rows) * FP;
        xs[(size_t)k * CR * FP + rows * FP + rem] = 0.f;
      }
    const long long pr0 = r0 >> P.log2p;
    const int prs = (int)min((long long)cpr, npr - pr0);
    const uint32_t xb = (uint32_t)rows * FP * 4u;
    const uint32_t fb = (uint32_t)prs * P.Fout * 4u, db = P.dy_is_mean ? (uint32_t)prs * 4u : fb;
    const uint32_t ab = has_am ? (uint32_t)prs * P.Fout : 0u;
    const float* dsrc = P.dy + (P.dy_is_mean ? pr0 : pr0 * P.Fout);
    // pieces whose size is not a multiple of 16 bytes (only possible in the last chunk) are copied by the threads
    const bool d_bulk = (db & 15u) == 0, f_bulk = (fb & 15u) == 0, a_bulk = (ab & 15u) == 0;
    if (!d_bulk)
      for (int i = tid; i < (int)(db >> 2); i += 256) reinterpret_cast<float*>(st + xbytes)[i] = __ldg(dsrc + i);
    if (P.relu && !f_bulk)
      for (int i = tid; i < (int)(fb >> 2); i += 256) reinterpret_cast<float*>(st + xbytes + rawf)[i] = __ldg(P.y + pr0 * P.Fout + i);
    if (has_am && !a_bulk)
      for (int i = tid; i < (int)ab; i += 256) (st + xbytes + 2 * rawf)[i] = __ldg(P.argmax + pr0 * P.Fout + i);
    if (tid == 0) {
      mbar_expect_tx(mbar + stage, xb * K + (d_bulk ? db : 0u) + ((P.relu && f_bulk) ? fb : 0u) + ((has_am && a_bulk) ? ab : 0u));
      for (int k = 0; k < K; ++k) bulk_g2s(xs + (size_t)k * CR * FP, P.xstack + ((size_t)k * P.R + r0) * FP, xb, mbar + stage);
      if (d_bulk && db) bulk_g2s(st + xbytes, dsrc, db, mbar + stage);
      if (P.relu && f_bulk && fb) bulk_g2s(st + xbytes + rawf, P.y + pr0 * P.Fout, fb, mbar + stage);
      if (has_am && a_bulk && ab) bulk_g2s(st + xbytes + 2 * rawf, P.argmax + pr0 * P.Fout, ab, mbar + stage);
    }
  };

  // dZ tile of the chunk from its raw pooled rows (shared -> shared): MaxPoolGrad o ReluGrad of dy
  const int fo_shift = P.FoP == 16 ? 4 : 5;
  const int zo = tid & (P.FoP - 1);
  auto expand_z = [&](int chunk, int stage) {
    const unsigned char* st = smem + (size_t)stage * sbytes;
    const float* rdy = reinterpret_cast<const float*>(st + xbytes);
    const float* ry = reinterpret_cast<const float*>(st + xbytes + rawf);
    const unsigned char* ram = st + xbytes + 2 * rawf;
    const long long pr0 = ((long long)chunk * CR) >> P.log2p;
    for (int j = tid >> fo_shift; j < cpr; j += 256 >> fo_shift) {
      float v = 0.f;
      int am = 0;
      if (pr0 + j < npr && zo < P.Fout) {
        const int gi = j * P.Fout + zo;
        v = P.dy_is_mean ? rdy[j] / (float)P.Fout : rdy[gi];
        if (P.relu && !(ry[gi] > 0.f)) v = 0.f;
        if (has_am) am = ram[gi];
      }
      dbacc += v;
      float* dst = Zs + (size_t)(j << P.log2p) * SZ + zo;
      for (int i = 0; i < P.p; ++i) dst[(size_t)i * SZ] = (i == am) ? v : 0.f;
    }
  };

  const int stride = gridDim.x;
  int chunk = blockIdx.x;
  for (int s = 0; s < NS - 1; ++s)
    if (chunk + s * stride < P.nchunks) issue(chunk + s * stride, s);
  for (int it = 0; chunk < P.nchunks; chunk += stride, ++it) {
    const int stage = it % NS;
    const int pre = chunk + (NS - 1) * stride;  // refills the stage consumed one iteration ago (barrier at the end)
    if (pre < P.nchunks) issue(pre, (it + NS - 1) % NS);
    mbar_wait(mbar + stage, (uint32_t)((it / NS) & 1));
    expand_z(chunk, stage);
    __syncthreads();
    const float* zs = Zs;
    const float* xs = reinterpret_cast<const float*>(smem + (size_t)stage * sbytes);
    for (int step = warp; step < CR / 8; step += 8) {
      const int r8 = step * 8;
      uint32_t bh[NT][2], bl[NT][2];
      const float* zr = zs + (size_t)(r8 + t) * SZ + g;
#pragma unroll
      for (int n = 0; n < NT; ++n) {
        split_trunc(zr[n * 8], bh[n][0], bl[n][0]);
        split_trunc(zr[n * 8 + 4 * SZ], bh[n][1], bl[n][1]);
      }
#pragma unroll
      for (int k = 0; k < K; ++k) {
        const float* xr = xs + ((size_t)k * CR + r8 + t) * SX + g;
#pragma unroll
        for (int m = 0; m < MT; ++m) {
          uint32_t ah[4], al[4];
          const bool hi_ok = (m * 16 + g + 8) < FP;
          split_trunc(xr[m * 16], ah[0], al[0]);
          split_trunc(hi_ok ? xr[m * 16 + 8] : 0.f, ah[1], al[1]);
          split_trunc(xr[m * 16 + 4 * SX], ah[2], al[2]);
          split_trunc(hi_ok ? xr[m * 16 + 8 + 4 * SX] : 0.f, ah[3], al[3]);
#pragma unroll
          for (int n = 0; n < NT; ++n) mma_3xtf32(acc[k][m][n], ah, al, bh[n][0], bh[n][1], bl[n][0], bl[n][1]);
        }
      }
    }
    __syncthreads();  // everyone done with this stage and the dZ tile before they are refilled
  }

  // ---- warps -> CTA (fixed order), CTA partial in the chunk layout k_dw_from_partials expects -----------------
  float* red = reinterpret_cast<float*>(smem);  // 8 warps x K*NCH*256 floats (fits: see host-side check)
  const int per_warp = K * NCH * 256;
#pragma unroll
  for (int k = 0; k < K; ++k)
#pragma unroll
    for (int m = 0; m < MT; ++m)
#pragma unroll
      for (int n = 0; n < NT; ++n)
#pragma unroll
        for (int c = 0; c < 4; ++c)
          red[(size_t)warp * per_warp + (k * NCH + m * (NT / 2) + n / 2) * 256 + ((n & 1) * 4 + c) * 32 + lane] =
              acc[k][m][n][c];
  __syncthreads();
  float* out = P.dw_part + (size_t)blockIdx.x * per_warp;
  for (int e = tid; e < per_warp; e += 256) {
    float s = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) s += red[(size_t)w * per_warp + e];
    out[e] = s;
  }
  if (P.db_part != nullptr) {
    __syncthreads();
    red[tid] = dbacc;
    __syncthreads();
    if (tid < P.FoP) {
      float s = 0.f;
      for (int i = tid; i < 256; i += P.FoP) s += red[i];
      P.db_part[(size_t)blockIdx.x * P.FoP + tid] = s;
    }
  }
}

struct StackPlan {
  bool ok;
  int FP, FoP, MT, NT, CR, SX, SZ, NS, ctas_per_sm;
  size_t smem;
};

int fused_feature_pad(int Fin) { return Fin < 1 || Fin > 32 ? 0 : (Fin <= 8 ? 8 : (Fin <= 16 ? 16 : 32)); }

static StackPlan plan_stack(const LayerShape& s) {
  StackPlan pl;
  pl.ok = false;
  pl.FP = fused_feature_pad(s.Fin);
  if (pl.FP == 0 || s.Fout < 1 || s.Fout > 32 || s.K < 1 || s.K > 5) return pl;
  if (s.p > 16 || s.M % s.p != 0) return pl;
  pl.FoP = s.Fout <= 16 ? 16 : 32;
  pl.MT = pl.FP <= 16 ? 1 : 2;
  pl.NT = pl.FoP / 8;
  pl.SX = pl.FP;  // dense rows: the tiles arrive by TMA bulk copies (2-way bank conflicts on the A fragments)
  pl.SZ = pl.FoP + 8;
  const size_t red = (size_t)8 * s.K * (pl.MT * pl.NT / 2) * 256 * 4;
  const bool light = s.K * pl.MT * pl.NT <= 20;
  for (int pass = light ? 0 : 1; pass < 2; ++pass) {  // pass 0: two CTAs per SM (<= 110 KB each); pass 1: one
    const size_t budget = pass == 0 ? 110 * 1024 : 220 * 1024;
    for (int cr : {128, 64, 32}) {
      if ((cr / s.p) * s.Fout % 16 != 0 || (cr / s.p) % 4 != 0) continue;  // pooled tiles start 16-byte aligned
      for (int ns : {3, 2}) {
        const size_t cprh = (size_t)cr / s.p;
        const size_t stage = (size_t)s.K * cr * pl.SX * 4 + 2 * cprh * s.Fout * 4 + (cprh * s.Fout + 15) / 16 * 16;
        const size_t need = ns * stage + (size_t)cr * pl.SZ * 4 + 64;
        if (std::max(need, red) <= budget) {
          pl.CR = cr;
          pl.NS = ns;
          pl.smem = std::max(need, red);
          pl.ctas_per_sm = pass == 0 ? 2 : 1;
          pl.ok = true;
          return pl;
        }
      }
    }
  }
  return pl;
}

bool stack_dw_supported(const LayerShape& s) { return plan_stack(s).ok; }

size_t stack_dw_workspace(const LayerShape& s) {
  const StackPlan pl = plan_stack(s);
  if (!pl.ok) return 0;
  return align_up((size_t)296 * (s.K * (pl.MT * pl.NT / 2) * 256 + 32) * 4, 256) + db_vertex_workspace(s) + 512;
}

template <int K, int MT, int NT>
static int launch_stack(const StackDwParams& P, const StackPlan& pl, int grid, cudaStream_t st) {
  auto kern = k_dw_from_stack<K, MT, NT>;
  GCNB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.smem));
  kern<<<grid, 256, pl.smem, st>>>(P);
  GCNB_LAUNCH_CHECK("k_dw_from_stack");
  return GCNB_OK;
}

int stack_dw(const float* xstack, const float* y, const uint8_t* argmax, const float* dy, int dy_is_mean, float* dW,
             float* db, const LayerShape& s, int bias_mode, int relu, Workspace& ws, cudaStream_t st) {
  const StackPlan pl = plan_stack(s);
  if (!pl.ok) {
    set_error("stack_dw: unsupported shape");
    return GCNB_ERR_INVALID;
  }
  DeviceInfo di;
  int rc = device_info(&di);
  if (rc) return rc;
  StackDwParams P;
  P.xstack = xstack; P.y = y; P.argmax = argmax; P.dy = dy;
  P.R = (long long)s.B * s.M; P.B = s.B; P.M = s.M; P.Mo = s.M / s.p; P.Fout = s.Fout; P.FoP = pl.FoP; P.FP = pl.FP;
  P.p = s.p; P.log2p = 0;
  while ((1 << P.log2p) < s.p) ++P.log2p;
  P.relu = relu; P.dy_is_mean = dy_is_mean;
  P.CR = pl.CR; P.SX = pl.SX; P.SZ = pl.SZ; P.NS = pl.NS;
  P.nchunks = (int)ceil_div_ll(P.R, pl.CR);
  const int grid = std::min(P.nchunks, std::min(di.sm_count * pl.ctas_per_sm, 296));
  const int nch = pl.MT * pl.NT / 2;
  float* part = ws.take<float>((size_t)grid * s.K * nch * 256);
  float* dbf = ws.take<float>((size_t)grid * 32);
  if (!part || !dbf) {
    set_error("stack_dw: workspace too small");
    return GCNB_ERR_WORKSPACE;
  }
  const bool db_fused = bias_mode == GCNB_BIAS_PER_FILTER && db != nullptr;
  P.dw_part = part;
  P.db_part = db_fused ? dbf : nullptr;
  rc = GCNB_ERR_INVALID;
#define GCNB_STACK_CASE(k, mt, nt) \
  if (s.K == k && pl.MT == mt && pl.NT == nt) rc = launch_stack<k, mt, nt>(P, pl, grid, st);
#define GCNB_STACK_K(k) GCNB_STACK_CASE(k, 1, 2) GCNB_STACK_CASE(k, 1, 4) GCNB_STACK_CASE(k, 2, 2) GCNB_STACK_CASE(k, 2, 4)
  GCNB_STACK_K(1) GCNB_STACK_K(2) GCNB_STACK_K(3) GCNB_STACK_K(4) GCNB_STACK_K(5)
#undef GCNB_STACK_K
#undef GCNB_STACK_CASE
  if (rc) return rc;
  rc = launch_dw_from_partials(part, dW, grid, s.K, pl.MT, pl.NT, s.Fin, s.Fout, P.db_part, db, pl.FoP, st);
  if (rc) return rc;
  if (bias_mode == GCNB_BIAS_PER_VERTEX && db != nullptr)
    return launch_db_vertex(dy, y, argmax, db, s, relu, dy_is_mean, ws, st);
  return GCNB_OK;
}

}  // namespace gcnb
