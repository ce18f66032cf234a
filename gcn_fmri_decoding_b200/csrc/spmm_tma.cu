// TMA-staged sparse recursion step for state that lives in HBM / L2 (vertex-level graphs, BASELINE config 5).
//
//   out[m][:] = alpha * sum_j val_j * src[col_j][:] + beta * add[m][:] + beta2 * add2[m][:]
//
// The state is vertex-major, one contiguous row of C = B*Fin floats per vertex, so the neighbour rows an output
// row needs are whole contiguous spans: the four producer warps of a persistent CTA turn every CSR entry into one
// cp.async.bulk copy (global -> shared, mbarrier complete_tx) into a ring of stages -- up to 8 neighbour rows
// plus the two "add" rows per stage -- and the eight consumer warps reduce a stage with conflict-free LDS.128
// and write the result with coalesced 16-byte stores.  No register staging, NS stages (~30 KB each) in flight
// per SM.  Rows longer than 8 entries take several stages; the partial sum stays in registers in between.
// (One producer warp is instruction bound at ~1800 cycles per row -- measured 211 us per order against 104 us
// for the register path; four of them, each owning its own stages, reach 99.7 us.)
// Work items (row, column chunk of <= 1024 floats) are dealt round-robin so that concurrently running CTAs
// work on neighbouring rows and share their neighbour rows in L2.
//
// Summation order = CSR order with fmaf, the same as k_spmm_step (general.cu), so both give identical bits.
// Reference math: graph.chebyshev recursion, lib_new/graph.py:163-171 / models_gcn.py:600-609.

#include "fused_common.cuh"

namespace gcnb {

namespace {

constexpr int kSlots = 8;
constexpr int kChunkMax = 1024;  // floats per column chunk = 256 consumer threads x float4
constexpr int kConsWarps = 8;
constexpr int kProdWarps = 4;    // one warp cannot issue ~7 copies per row fast enough (it is instruction bound)
constexpr int kSpmmThreads = (kConsWarps + kProdWarps) * 32;
constexpr int kSpmmMaxStages = 8;
constexpr int kHdrBytes = 64;
constexpr int kFixedBytes = 2 * kSpmmMaxStages * 8 + kProdWarps * 32 * kSlots * 8;  // barriers + prefetch tables

struct StageHdr {
  int nflags;  // entries in this stage | (first stage of the row ? 256 : 0) | (last ? 512 : 0)
  int pad[3];
  float val[kSlots];
  int pad2[4];
};
static_assert((kProdWarps & (kProdWarps - 1)) == 0 && kSpmmMaxStages % kProdWarps == 0, "stage ownership");
static_assert(sizeof(StageHdr) == kHdrBytes, "stage header is 64 bytes");

struct SpmmArgs {
  const int32_t* rowptr;
  const int32_t* col;
  const float* val;
  const float* src;
  const float* add;
  const float* add2;
  float* out;
  long long C;
  int M, CW, nchunk, NS;
  uint32_t stage_bytes;
  float alpha, beta, beta2;
};

__device__ __forceinline__ void mbar_arrive1(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// kOne: the whole vertex row is one column chunk (C <= 1024 floats), item index == vertex
template <bool kOne>
__global__ void __launch_bounds__(kSpmmThreads, 1) k_spmm_tma(SpmmArgs a) {
  extern __shared__ __align__(128) unsigned char smem[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  uint64_t* full = reinterpret_cast<uint64_t*>(smem);
  uint64_t* empty = full + kSpmmMaxStages;
  unsigned char* stages = smem + align_up((size_t)kFixedBytes, 128);
  if (tid == 0)
    for (int s = 0; s < a.NS; ++s) {
      mbar_init(full + s, 1);
      mbar_init(empty + s, kConsWarps);
    }
  __syncthreads();
  const long long total = kOne ? (long long)a.M : (long long)a.M * a.nchunk;
  const int NS = a.NS;
  const int G = gridDim.x;

  if (warp >= kConsWarps) {
    // ---- producer warps.  The items of this CTA are q = blockIdx.x + i*G, i = 0, 1, ...; a row of more than kSlots
    // entries takes several stages, so the ring position `it` of a stage use is the running sum of the stage counts
    // of all earlier items: every producer scans the degrees of a batch of 32 items (one per lane) and they agree
    // on it without talking to each other.  Producer p fills the uses with it % kProdWarps == p.  NS is a multiple of
    // kProdWarps, so a given stage is always filled -- and its release always awaited -- by the same producer, one
    // phase after the other: exactly the single-producer ring discipline an mbarrier parity wait needs.
    const int p = warp - kConsWarps;
    int* pcol = reinterpret_cast<int*>(smem + 2 * kSpmmMaxStages * 8) + p * 32 * kSlots * 2;
    float* pval = reinterpret_cast<float*>(pcol + 32 * kSlots);
    const bool has_add = a.add != nullptr, has_add2 = a.add2 != nullptr;
    int it_base = 0;
    for (long long i0 = 0; blockIdx.x + i0 * G < total; i0 += 32) {
      const long long q = blockIdx.x + (i0 + lane) * G;
      int beg = 0, end = 0, m = 0, cc = 0;
      if (q < total) {
        m = kOne ? (int)q : (int)(q / a.nchunk);
        cc = kOne ? 0 : (int)(q - (long long)m * a.nchunk);
        beg = __ldg(a.rowptr + m);
        end = __ldg(a.rowptr + m + 1);
      }
      const int passes = q < total ? max(1, (end - beg + kSlots - 1) / kSlots) : 0;
      int incl = passes;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += t;
      }
      const int it_first = it_base + incl - passes;
      const int batch_uses = __shfl_sync(0xffffffffu, incl, 31);
      const int nvalid = __popc(__ballot_sync(0xffffffffu, q < total));
      const bool simple = batch_uses == nvalid;  // every row of the batch fits one stage: use i0 + l <-> item l
      if (simple && lane < nvalid && ((it_base + lane) & (kProdWarps - 1)) == p) {
#pragma unroll
        for (int e = 0; e < kSlots; ++e)
          if (beg + e < end) {
            pcol[lane * kSlots + e] = __ldg(a.col + beg + e);
            pval[lane * kSlots + e] = __ldg(a.val + beg + e);
          }
      }
      __syncwarp();

      // fill stage use `it` with pass `pass` (of npass) of item ii; executed by the whole warp
      auto fill = [&](int ii, int pass, int npass, int it) {
        const int ibeg = __shfl_sync(0xffffffffu, beg, ii), iend = __shfl_sync(0xffffffffu, end, ii);
        const int im = __shfl_sync(0xffffffffu, m, ii);
        long long c0 = 0;
        uint32_t wbytes = (uint32_t)a.C * 4;
        if (!kOne) {
          c0 = (long long)__shfl_sync(0xffffffffu, cc, ii) * a.CW;
          wbytes = (uint32_t)((a.C - c0 < a.CW ? a.C - c0 : a.CW) * 4);
        }
        const int j0 = ibeg + pass * kSlots;
        const int n = iend - j0 < kSlots ? iend - j0 : kSlots;
        const bool last = pass == npass - 1;
        const int s = it % NS, u = it / NS;
        if (u > 0) mbar_wait(empty + s, (uint32_t)((u - 1) & 1));
        unsigned char* st = stages + (size_t)s * a.stage_bytes;
        StageHdr* h = reinterpret_cast<StageHdr*>(st);
        float* seg = reinterpret_cast<float*>(st + kHdrBytes);
        // lanes [0, n): neighbour rows; lane n / n+1: the add rows (last stage of the row only)
        const int ncopy = n + (last ? (int)has_add + (int)has_add2 : 0);
        const float* from = nullptr;
        float* to = seg + (size_t)lane * a.CW;
        if (lane < n) {
          int cj;
          float v;
          if (simple) {
            cj = pcol[ii * kSlots + lane];
            v = pval[ii * kSlots + lane];
          } else {
            cj = __ldg(a.col + j0 + lane);
            v = __ldg(a.val + j0 + lane);
          }
          h->val[lane] = v;
          from = a.src + (long long)cj * a.C + c0;
        } else if (lane == n) {
          from = has_add ? a.add + (long long)im * a.C + c0 : nullptr;
          to = seg + (size_t)kSlots * a.CW;
        } else if (lane == n + 1) {
          from = has_add2 ? a.add2 + (long long)im * a.C + c0 : nullptr;
          to = seg + (size_t)(kSlots + 1) * a.CW;
        }
        if (lane == 0) h->nflags = n | (pass == 0 ? 256 : 0) | (last ? 512 : 0);
        __syncwarp();  // header complete before the (releasing) arrive
        if (lane == 0) mbar_expect_tx(full + s, (uint32_t)ncopy * wbytes);
        __syncwarp();
        if (lane < ncopy) bulk_g2s_ring(to, from, wbytes, full + s);
      };

      if (simple) {
        for (int ii = (p - it_base) & (kProdWarps - 1); ii < nvalid; ii += kProdWarps) fill(ii, 0, 1, it_base + ii);
      } else {
        for (int ii = 0; ii < nvalid; ++ii) {
          const int npass = __shfl_sync(0xffffffffu, passes, ii);
          const int itf = __shfl_sync(0xffffffffu, it_first, ii);
          for (int pass = 0; pass < npass; ++pass)
            if (((itf + pass) & (kProdWarps - 1)) == p) fill(ii, pass, npass, itf + pass);
        }
      }
      it_base += batch_uses;
      __syncwarp();
    }
    return;
  }

  // ---- consumers: thread t owns columns [4t, 4t+4) of the chunk
  long long it = 0;
  const int cw4 = a.CW >> 2;
  for (long long q = blockIdx.x; q < total; q += G) {
    const int m = kOne ? (int)q : (int)(q / a.nchunk);
    const long long c0 = kOne ? 0 : (q - (long long)m * a.nchunk) * a.CW;
    const int w = (int)(a.C - c0 < a.CW ? a.C - c0 : a.CW);
    const bool active = tid * 4 < w;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    while (true) {
      const int s = (int)(it % NS);
      mbar_wait(full + s, (uint32_t)((it / NS) & 1));
      const unsigned char* st = stages + (size_t)s * a.stage_bytes;
      const StageHdr* h = reinterpret_cast<const StageHdr*>(st);
      const float4* seg = reinterpret_cast<const float4*>(st + kHdrBytes) + tid;
      const int nflags = h->nflags;
      const int n = nflags & 255;
      if (nflags & 256) acc = make_float4(0.f, 0.f, 0.f, 0.f);
      if (active) {
        const float4 va = *reinterpret_cast<const float4*>(h->val), vb = *reinterpret_cast<const float4*>(h->val + 4);
        const float vals[kSlots] = {va.x, va.y, va.z, va.w, vb.x, vb.y, vb.z, vb.w};
#pragma unroll
        for (int i = 0; i < kSlots; ++i)
          if (i < n) {
            const float v = vals[i];
            const float4 x = seg[(size_t)i * cw4];
            acc.x = fmaf(v, x.x, acc.x);
            acc.y = fmaf(v, x.y, acc.y);
            acc.z = fmaf(v, x.z, acc.z);
            acc.w = fmaf(v, x.w, acc.w);
          }
        if (nflags & 512) {
          float4 r = make_float4(a.alpha * acc.x, a.alpha * acc.y, a.alpha * acc.z, a.alpha * acc.w);
          if (a.add != nullptr) {
            const float4 p = seg[(size_t)kSlots * cw4];
            r.x = fmaf(a.beta, p.x, r.x);
            r.y = fmaf(a.beta, p.y, r.y);
            r.z = fmaf(a.beta, p.z, r.z);
            r.w = fmaf(a.beta, p.w, r.w);
          }
          if (a.add2 != nullptr) {
            const float4 p = seg[(size_t)(kSlots + 1) * cw4];
            r.x = fmaf(a.beta2, p.x, r.x);
            r.y = fmaf(a.beta2, p.y, r.y);
            r.z = fmaf(a.beta2, p.z, r.z);
            r.w = fmaf(a.beta2, p.w, r.w);
          }
          *reinterpret_cast<float4*>(a.out + (long long)m * a.C + c0 + tid * 4) = r;
        }
      }
      __syncwarp();
      if (lane == 0) mbar_arrive1(empty + s);
      ++it;
      if (nflags & 512) break;
    }
  }
}

bool plan_spmm(long long C, int* CW, int* nchunk, int* NS, uint32_t* stage_bytes, size_t* smem) {
  if (C < 4 || C % 4 != 0) return false;
  *nchunk = (int)ceil_div_ll(C, kChunkMax);
  *CW = (int)((ceil_div_ll(C, *nchunk) + 3) / 4 * 4);
  *stage_bytes = (uint32_t)align_up((size_t)kHdrBytes + (size_t)(kSlots + 2) * *CW * 4, 128);
  DeviceInfo di;
  if (device_info(&di) != GCNB_OK) return false;
  const size_t fixed = align_up((size_t)kFixedBytes, 128);
  if ((size_t)di.smem_optin < fixed + 2 * (size_t)*stage_bytes) return false;
  if ((size_t)di.smem_optin < fixed + (size_t)kProdWarps * *stage_bytes) return false;
  *NS = (int)std::min<size_t>(kSpmmMaxStages, ((size_t)di.smem_optin - fixed) / *stage_bytes);
  *NS = *NS / kProdWarps * kProdWarps;  // each stage belongs to one producer warp
  *smem = fixed + (size_t)*NS * *stage_bytes;
  return true;
}

}  // namespace

bool spmm_tma_supported(const gcnb_csr& L, long long C, const float* src, const float* add, const float* add2,
                        const float* out) {
  int CW, nchunk, NS;
  uint32_t sb;
  size_t smem;
  const uintptr_t bits = reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(add) |
                         reinterpret_cast<uintptr_t>(add2) | reinterpret_cast<uintptr_t>(out);
  return L.M >= 1 && (bits & 15) == 0 && src != out && (add != nullptr || add2 == nullptr) && plan_spmm(C, &CW, &nchunk, &NS, &sb, &smem);
}

int spmm_tma(const gcnb_csr& L, const float* src, const float* add, const float* add2, float* out, long long C,
             float alpha, float beta, float beta2, cudaStream_t st) {
  SpmmArgs a;
  size_t smem;
  if (!plan_spmm(C, &a.CW, &a.nchunk, &a.NS, &a.stage_bytes, &smem)) {
    set_error("spmm_tma: unsupported row width %lld", C);
    return GCNB_ERR_INVALID;
  }
  a.rowptr = L.rowptr; a.col = L.col; a.val = L.val; a.src = src; a.add = add; a.add2 = add2; a.out = out;
  a.C = C; a.M = L.M; a.alpha = alpha; a.beta = beta; a.beta2 = beta2;
  DeviceInfo di;
  if (device_info(&di) != GCNB_OK) return GCNB_ERR_CUDA;
  // per device / context, so set on every launch like the other kernels (a process may drive several GPUs)
  GCNB_CUDA(cudaFuncSetAttribute(k_spmm_tma<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, di.smem_optin));
  GCNB_CUDA(cudaFuncSetAttribute(k_spmm_tma<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, di.smem_optin));
  const long long total = (long long)L.M * a.nchunk;
  const int grid = (int)std::min<long long>(total, di.sm_count);
  if (a.nchunk == 1)
    k_spmm_tma<true><<<grid, kSpmmThreads, smem, st>>>(a);
  else
    k_spmm_tma<false><<<grid, kSpmmThreads, smem, st>>>(a);
  GCNB_LAUNCH_CHECK("k_spmm_tma");
  return GCNB_OK;
}

}  // namespace gcnb
