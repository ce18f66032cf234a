// Gradient of a ChebyNet layer w.r.t. the entries of its operator L~: a sampled dense-dense product (SDDMM) on the
// sparsity pattern of L~ plus its diagonal, between the two vertex-major stacks the general path keeps in HBM.
//
//   dL~[b][i][j] = sum_f b_1[i][b*Fin+f] X_0[j][b*Fin+f]  +  sum_{k=2}^{K-1} 2 sum_f b_k[i][b*Fin+f] X_{k-1}[j][b*Fin+f]
//
// X_k is the Chebyshev basis (build_stack) and b_k the Clenshaw states of the adjoint (general_cheb_bwd's loop), both
// [k][m][b*Fin + f], one contiguous row of C = B*Fin floats per vertex.  Each output is a dot of Fin products per order
// with no reuse, so there is no MMA shape to feed: like the recursion step (spmm_tma.cu) the kernel is a gather stream
// bounded by L2 -> SM traffic, and it uses the same persistent producer / consumer layout.
//
// Work item = (row i, chunk of nw windows).  The row's entries -- the CSR entries of row i, then the diagonal (i, i) --
// are taken kSlots at a time; per group and per order k the producer warp fills one stage of the ring with one
// cp.async.bulk copy per entry (the row chunk of X_{k-1}[j]) and one for b_k[i].  A copy starts at the 16-byte boundary
// at or below its row chunk and ends at the one at or above, so any B*Fin is served (the stage header tells the
// consumers where the chunk starts); the stacks are allocated with 16 bytes of slack behind them for that.
// Consumer thread t owns entry slot t % kSlots of window t / kSlots: it sums the orders in a fixed order into one
// register and writes its value once -- no atomics, bit-reproducible, and consecutive threads write consecutive CSR
// entries of one window.
//
// Outputs: dval[b][e] in L~'s CSR order, ddiag[b][i]; accumulate != 0 adds onto them (layers sharing an operator).

#include <algorithm>

#include "fused_common.cuh"

namespace gcnb {

namespace {

constexpr int kSlots = 8;                 // entries per stage
constexpr int kConsWarps = 8;             // 256 consumers = kSlots x 32 windows
constexpr int kWinMax = kConsWarps * 32 / kSlots;
constexpr int kChunkFloats = 1024;        // target floats per row chunk (nw * Fin)
constexpr int kThreads = (kConsWarps + 1) * 32;
constexpr int kMaxStages = 8;
constexpr int kHdrBytes = 64;

struct StageHdr {
  int n;                // entries in this stage
  int off[kSlots + 1];  // float offset of the row chunk inside its segment (segment kSlots: b_k[i])
  int pad[6];
};
static_assert(sizeof(StageHdr) == kHdrBytes, "stage header is 64 bytes");

struct SddmmArgs {
  const int32_t* rowptr;
  const int32_t* col;
  const float* X;   // basis stack, slab k = X_k
  const float* Bk;  // Clenshaw stack, slab k = b_k (k >= 1)
  float* dval;
  float* ddiag;
  long long C, slab;
  int M, nnz, B, Fin, K, nw, nchunk, NS, seg;  // seg: floats per segment
  uint32_t stage_bytes;
  int accumulate;
};

__device__ __forceinline__ void mbar_arrive1(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

__global__ void __launch_bounds__(kThreads, 1) k_sddmm_tma(SddmmArgs a) {
  extern __shared__ __align__(128) unsigned char smem[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  uint64_t* full = reinterpret_cast<uint64_t*>(smem);
  uint64_t* empty = full + kMaxStages;
  unsigned char* stages = smem + 256;
  if (tid == 0)
    for (int s = 0; s < a.NS; ++s) {
      mbar_init(full + s, 1);
      mbar_init(empty + s, kConsWarps);
    }
  __syncthreads();
  const long long total = (long long)a.M * a.nchunk;
  const int NS = a.NS, G = gridDim.x, orders = a.K - 1;

  if (warp == kConsWarps) {
    // ---- producer warp: stage use `it` goes to stage it % NS, phase it / NS
    long long it = 0;
    for (long long q = blockIdx.x; q < total; q += G) {
      const int i = (int)(q / a.nchunk), cc = (int)(q - (long long)i * a.nchunk);
      const int w0 = cc * a.nw, nwc = min(a.nw, a.B - w0);
      const long long c0 = (long long)w0 * a.Fin;
      const uint32_t wbytes = (uint32_t)nwc * a.Fin * 4;
      const int beg = __ldg(a.rowptr + i), deg = __ldg(a.rowptr + i + 1) - beg;
      const int nent = deg + 1;
      for (int g0 = 0; g0 < nent; g0 += kSlots) {
        const int n = min(kSlots, nent - g0);
        int j = i;
        if (lane < n && g0 + lane < deg) j = __ldg(a.col + beg + g0 + lane);
        for (int k = 1; k <= orders; ++k, ++it) {
          const int s = (int)(it % NS);
          const long long u = it / NS;
          if (u > 0) mbar_wait(empty + s, (uint32_t)((u - 1) & 1));
          unsigned char* st = stages + (size_t)s * a.stage_bytes;
          StageHdr* h = reinterpret_cast<StageHdr*>(st);
          float* seg = reinterpret_cast<float*>(st + kHdrBytes);
          // lanes [0, n): X_{k-1}[j] of the entries; lane n: b_k[i]
          const float* from = nullptr;
          float* to = seg + (size_t)lane * a.seg;
          if (lane < n) {
            from = a.X + (long long)(k - 1) * a.slab + (long long)j * a.C + c0;
          } else if (lane == n) {
            from = a.Bk + (long long)k * a.slab + (long long)i * a.C + c0;
            to = seg + (size_t)kSlots * a.seg;
          }
          uint32_t bytes = 0;
          const float* aligned = nullptr;
          if (from != nullptr) {
            const uintptr_t lo = reinterpret_cast<uintptr_t>(from) & ~(uintptr_t)15;
            const uintptr_t hi = (reinterpret_cast<uintptr_t>(from) + wbytes + 15) & ~(uintptr_t)15;
            aligned = reinterpret_cast<const float*>(lo);
            bytes = (uint32_t)(hi - lo);
            h->off[lane < n ? lane : kSlots] = (int)((reinterpret_cast<uintptr_t>(from) - lo) >> 2);
          }
          if (lane == 0) h->n = n;
          uint32_t tx = bytes;
#pragma unroll
          for (int d = 16; d > 0; d >>= 1) tx += __shfl_xor_sync(0xffffffffu, tx, d);
          __syncwarp();  // header complete before the (releasing) arrive
          if (lane == 0) mbar_expect_tx(full + s, tx);
          __syncwarp();
          if (from != nullptr) bulk_g2s_ring(to, aligned, bytes, full + s);
        }
      }
    }
    return;
  }

  // ---- consumers: thread t owns entry slot t % kSlots of window t / kSlots of the chunk
  const int slot = tid % kSlots, wl = tid / kSlots;
  long long it = 0;
  for (long long q = blockIdx.x; q < total; q += G) {
    const int i = (int)(q / a.nchunk), cc = (int)(q - (long long)i * a.nchunk);
    const int w0 = cc * a.nw, nwc = min(a.nw, a.B - w0);
    const int beg = __ldg(a.rowptr + i), deg = __ldg(a.rowptr + i + 1) - beg;
    const int nent = deg + 1;
    for (int g0 = 0; g0 < nent; g0 += kSlots) {
      float acc = 0.f;
      int n = 0;
      for (int k = 1; k <= orders; ++k, ++it) {
        const int s = (int)(it % NS);
        mbar_wait(full + s, (uint32_t)((it / NS) & 1));
        const unsigned char* st = stages + (size_t)s * a.stage_bytes;
        const StageHdr* h = reinterpret_cast<const StageHdr*>(st);
        const float* seg = reinterpret_cast<const float*>(st + kHdrBytes);
        n = h->n;
        if (slot < n && wl < nwc) {
          const float* xr = seg + (size_t)slot * a.seg + h->off[slot] + wl * a.Fin;
          const float* br = seg + (size_t)kSlots * a.seg + h->off[kSlots] + wl * a.Fin;
          float d = 0.f;
          for (int f = 0; f < a.Fin; ++f) d = fmaf(br[f], xr[f], d);
          acc = fmaf(k == 1 ? 1.f : 2.f, d, acc);
        }
        __syncwarp();
        if (lane == 0) mbar_arrive1(empty + s);
      }
      if (slot < n && wl < nwc) {
        const int e = g0 + slot;
        const long long b = w0 + wl;
        float* o = e < deg ? a.dval + b * a.nnz + beg + e : a.ddiag + b * a.M + i;
        *o = a.accumulate ? *o + acc : acc;
      }
    }
  }
}

bool plan_sddmm(const LayerShape& s, int* nw, int* nchunk, int* seg, int* NS, uint32_t* stage_bytes, size_t* smem) {
  if (s.K < 2 || s.Fin < 1) return false;
  *nw = std::max(1, std::min(kWinMax, kChunkFloats / s.Fin));
  *nchunk = ceil_div(s.B, *nw);
  // a copy spans the row chunk plus at most 12 bytes on each side; segments stay 16-byte aligned
  *seg = (int)align_up((size_t)*nw * s.Fin + 8, 4);
  *stage_bytes = (uint32_t)align_up((size_t)kHdrBytes + (size_t)(kSlots + 1) * *seg * 4, 128);
  DeviceInfo di;
  if (device_info(&di) != GCNB_OK) return false;
  if ((size_t)di.smem_optin < 256 + 2 * (size_t)*stage_bytes) return false;
  *NS = (int)std::min<size_t>(kMaxStages, ((size_t)di.smem_optin - 256) / *stage_bytes);
  *smem = 256 + (size_t)*NS * *stage_bytes;
  return true;
}

}  // namespace

int sddmm_tma(const gcnb_csr& L, const float* X, const float* Bk, float* dval, float* ddiag, int accumulate,
              const LayerShape& s, cudaStream_t st) {
  SddmmArgs a;
  size_t smem;
  if (!plan_sddmm(s, &a.nw, &a.nchunk, &a.seg, &a.NS, &a.stage_bytes, &smem)) {
    set_error("sddmm_tma: unsupported layer (Fin=%d, K=%d)", s.Fin, s.K);
    return GCNB_ERR_INVALID;
  }
  a.rowptr = L.rowptr; a.col = L.col; a.X = X; a.Bk = Bk; a.dval = dval; a.ddiag = ddiag;
  a.C = (long long)s.B * s.Fin; a.slab = (long long)s.M * a.C;
  a.M = s.M; a.nnz = L.nnz; a.B = s.B; a.Fin = s.Fin; a.K = s.K; a.accumulate = accumulate;
  DeviceInfo di;
  if (device_info(&di) != GCNB_OK) return GCNB_ERR_CUDA;
  GCNB_CUDA(cudaFuncSetAttribute(k_sddmm_tma, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const long long total = (long long)s.M * a.nchunk;
  const int grid = (int)std::min<long long>(total, di.sm_count);
  k_sddmm_tma<<<grid, kThreads, smem, st>>>(a);
  GCNB_LAUNCH_CHECK("k_sddmm_tma");
  return GCNB_OK;
}

}  // namespace gcnb
