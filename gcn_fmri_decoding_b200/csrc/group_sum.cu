// Grouped column sum: out[g][c] = sum over the rows r with group[r] == g of X[r][c] (|X[r][c]| with `absolute`) -- the
// per-class / per-subject sums of the saliency maps, one row per window.
//
// k_group_colsum: one CTA of 32 warps per 32-column chunk (as k_colsum_multi).  The CTA sorts the row indices by group
// (a block radix sort on the keys group[r], rows of an out-of-range group keyed past every valid id and dropped; the
// sort is stable, so a group's rows stay in row order).  Each warp walks one contiguous slice of that order, one column
// per lane, and sums every run of equal groups in row order.  A run that begins before the warp's slice (the slice's
// "head") is parked in shared memory; the warp that owns the run's first row adds the heads of the following warps in
// warp order and writes the result.  So every output has one writer and a summation order fixed by (rows, group): no
// float atomics, bit-reproducible.  Each element of X is read once; rows of no valid group are not read.  The sort keys
// take as many bits as `rows` does, so the work does not depend on n_groups (a capacity), only on rows x cols.

#include <cub/block/block_radix_sort.cuh>

#include "common.cuh"

namespace gcnb {

namespace {

constexpr int kThreads = 1024;
constexpr int kMaxRows = 8192;

template <int kItems>
__global__ void __launch_bounds__(kThreads) k_group_colsum(const float* __restrict__ X, int rows, int cols,
                                                           const int32_t* __restrict__ group, int n_groups, int absolute,
                                                           float* __restrict__ out) {
  using Sort = cub::BlockRadixSort<uint16_t, kThreads, kItems, uint16_t>;
  struct Sorted {
    uint16_t grp[kThreads * kItems], row[kThreads * kItems];
  };
  __shared__ union {
    typename Sort::TempStorage sort;
    Sorted sorted;
  } sm;
  __shared__ float head[32][32];
  __shared__ int n_valid;

  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) n_valid = 0;
  __syncthreads();
  // blocked arrangement: thread t holds rows t * kItems + i; an invalid row is keyed `rows` (> every valid id)
  uint16_t key[kItems], val[kItems];
  int valid = 0;
#pragma unroll
  for (int i = 0; i < kItems; ++i) {
    const int r = threadIdx.x * kItems + i;
    const int g = r < rows ? group[r] : -1;
    const bool ok = g >= 0 && g < n_groups;
    key[i] = (uint16_t)(ok ? g : rows);
    val[i] = (uint16_t)r;
    valid += ok;
  }
  if (valid) atomicAdd(&n_valid, valid);
  Sort(sm.sort).Sort(key, val, 0, 32 - __clz(rows));
  __syncthreads();  // the sort's storage is reused for its result
#pragma unroll
  for (int i = 0; i < kItems; ++i) {
    sm.sorted.grp[threadIdx.x * kItems + i] = key[i];
    sm.sorted.row[threadIdx.x * kItems + i] = val[i];
  }
  __syncthreads();

  const int nv = n_valid;
  const int len = (nv + 31) / 32;
  const int lo = min(warp * len, nv), hi = min(lo + len, nv);
  const int c = blockIdx.x * 32 + lane;
  const bool col_ok = c < cols;
  const uint16_t* sg = sm.sorted.grp;
  const uint16_t* sr = sm.sorted.row;
  // sum of the sorted positions [a, b) of one group, in row order; run_end: the end of the run that starts at a
  auto run_sum = [&](int a, int b) {
    float acc = 0.f;
    if (col_ok) {
#pragma unroll 8
      for (; a < b; ++a) {
        const float v = X[(long long)sr[a] * cols + c];
        acc += absolute ? fabsf(v) : v;
      }
    }
    return acc;
  };
  auto run_end = [&](int a) {
    int b = a + 1;
    while (b < hi && sg[b] == sg[a]) ++b;
    return b;
  };

  int p = lo;
  if (p < hi && p > 0 && sg[p - 1] == sg[p]) {  // the slice starts inside a run: its head goes to the run's owner
    const int q = run_end(p);
    head[warp][lane] = run_sum(p, q);
    p = q;
  }
  __syncthreads();
  while (p < hi) {
    const int q = run_end(p);
    const uint16_t g = sg[p];
    float acc = run_sum(p, q);
    if (q == hi)  // the run may go on into the following slices, each of which then starts with a head of group g
      for (int w = warp + 1; w < 32 && w * len < nv && sg[w * len] == g; ++w) acc += head[w][lane];
    if (col_ok) out[(long long)g * cols + c] = acc;
    p = q;
  }
}

template <int kItems>
void launch(const float* X, int rows, int cols, const int32_t* group, int n_groups, int absolute, float* out,
            cudaStream_t st) {
  k_group_colsum<kItems><<<ceil_div(cols, 32), kThreads, 0, st>>>(X, rows, cols, group, n_groups, absolute, out);
}

}  // namespace

}  // namespace gcnb

using namespace gcnb;

extern "C" int gcnb_group_colsum_f32(const float* X, int rows, int cols, const int32_t* group, int n_groups,
                                     int absolute, float* out, gcnb_stream_t stream) {
  GCNB_REQUIRE(X && group && out, "gcnb_group_colsum_f32: null pointer");
  GCNB_REQUIRE(rows >= 1 && rows <= kMaxRows, "gcnb_group_colsum_f32: rows = %d outside [1, %d]", rows, kMaxRows);
  GCNB_REQUIRE(cols >= 1, "gcnb_group_colsum_f32: cols = %d < 1", cols);
  GCNB_REQUIRE(n_groups >= 1 && n_groups <= rows, "gcnb_group_colsum_f32: n_groups = %d outside [1, rows = %d]",
               n_groups, rows);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (rows <= kThreads)
    launch<1>(X, rows, cols, group, n_groups, absolute, out, st);
  else if (rows <= 2 * kThreads)
    launch<2>(X, rows, cols, group, n_groups, absolute, out, st);
  else if (rows <= 4 * kThreads)
    launch<4>(X, rows, cols, group, n_groups, absolute, out, st);
  else
    launch<8>(X, rows, cols, group, n_groups, absolute, out, st);
  GCNB_LAUNCH_CHECK("k_group_colsum");
  return GCNB_OK;
}
