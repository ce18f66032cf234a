// Gradient w.r.t. the adjacency matrix: the chain rule from the per-window operator gradients G_l = d logit / d L~_l
// (gcnb_cheb_dL_f32's dval, one [B][nnz_l] block per coarsening level) to the undirected edge weights of the input
// graph A, through the degree normalisation of every level and the Graclus coarsening between levels.
//
// Level l: A_l the adjacency (zero diagonal), d_b = sum_a A_l[a][b], s = d^-1/2, L~_l = -s_a A_ab s_b off the diagonal.
//   r_b = sum_j G_bj L~_bj (row b),  c_b = sum_i G_ib L~_ib (column b),  both over the stored entries
//   dlogit/dA_l[a][b] = -G_ab s_a s_b - (r_b + c_b) / (2 d_b)
// Coarsening: A_{l+1} = P^T A_l P (vertices 2J, 2J+1 merge into J), diagonal zeroed, so the total gradient is
//   T_l[(a, b)] = dlogit/dA_l[a][b] + T_{l+1}[(a>>1, b>>1)]   (second term only when a>>1 != b>>1)
// -- a gather through a host-built parent-entry map.  Level 0 is A permuted: edge {i, j} of A gets
//   S_ij = T_0[(a, b)] + T_0[(b, a)],  a, b the model rows of ROIs i, j  (|S| per window with `absolute`).
//
// k_adjacency_level: one thread per (window, vertex b).  It sums r_b over row b of L~'s CSR and c_b over row b of L~^T
// (the transposed-position map names the entry of L~'s order, so both read G in place), then writes T_l for every
// entry of column b.  Every entry has one column, so each output is written by one thread in a fixed order: no atomics,
// bit-reproducible.  Nothing is staged in shared memory, so any level size is taken (config 5: one level of 32 492
// vertices).  k_adjacency_edges: one thread per (window, ROI edge).

#include <algorithm>

#include "common.cuh"

namespace gcnb {

namespace {

__global__ void k_adjacency_level(gcnb_adj_level lv, const float* __restrict__ Tnext, int nnz_next,
                                  float* __restrict__ T, int B) {
  const long long total = (long long)B * lv.M;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long w = i / lv.M;
    const int b = (int)(i - w * lv.M);
    const float* G = lv.dval + w * lv.nnz;
    const int r0 = lv.rowptr[b], r1 = lv.rowptr[b + 1];
    const int c0 = lv.rowptr_t[b], c1 = lv.rowptr_t[b + 1];
    float r = 0.f, c = 0.f;
    for (int e = r0; e < r1; ++e) r = fmaf(G[e], lv.val[e], r);
    for (int t = c0; t < c1; ++t) {
      const int e = lv.tpos[t];
      c = fmaf(G[e], lv.val[e], c);
    }
    const float q = -(r + c) * lv.hinv[b];
    float* Tw = T + w * lv.nnz;
    const float* Tp = Tnext ? Tnext + w * nnz_next : nullptr;
    for (int t = c0; t < c1; ++t) {
      const int e = lv.tpos[t];
      float v = fmaf(-G[e], lv.ss[e], q);
      if (Tp) {
        const int pe = lv.parent[e];
        if (pe >= 0) v += Tp[pe];
      }
      Tw[e] = v;
    }
  }
}

__global__ void k_adjacency_edges(const float* __restrict__ T0, int nnz0, const int32_t* __restrict__ edges, int E,
                                  float* __restrict__ out, int B, int absolute) {
  const long long total = (long long)B * E;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long w = i / E;
    const int k = (int)(i - w * E);
    const float* Tw = T0 + w * nnz0;
    const float v = Tw[edges[2 * k]] + Tw[edges[2 * k + 1]];
    out[i] = absolute ? fabsf(v) : v;
  }
}

unsigned grid_over(long long total) {
  return (unsigned)std::max<long long>(1, std::min<long long>(ceil_div_ll(total, 256), 148 * 16));
}

}  // namespace

size_t adjacency_grad_workspace(const gcnb_adj_level* levels, int nlevels, int B) {
  size_t n = 0;
  for (int l = 0; l < nlevels; ++l) n += align_up((size_t)B * levels[l].nnz * sizeof(float), 256) + 256;
  return n;
}

int adjacency_grad(const gcnb_adj_level* levels, int nlevels, const int32_t* edges, int E, float* out, int B,
                   int absolute, Workspace& ws, cudaStream_t st) {
  float* T[GCNB_ADJ_MAX_LEVELS];
  for (int l = 0; l < nlevels; ++l) {
    T[l] = ws.take<float>((size_t)B * levels[l].nnz);
    if (!T[l]) {
      set_error("gcnb_adjacency_grad_f32: workspace too small");
      return GCNB_ERR_WORKSPACE;
    }
  }
  for (int l = nlevels - 1; l >= 0; --l) {
    const gcnb_adj_level& lv = levels[l];
    if (lv.nnz == 0) continue;
    const bool top = l == nlevels - 1;
    k_adjacency_level<<<grid_over((long long)B * lv.M), 256, 0, st>>>(lv, top ? nullptr : T[l + 1],
                                                                       top ? 0 : levels[l + 1].nnz, T[l], B);
    GCNB_LAUNCH_CHECK("k_adjacency_level");
  }
  if (E == 0) return GCNB_OK;
  k_adjacency_edges<<<grid_over((long long)B * E), 256, 0, st>>>(T[0], levels[0].nnz, edges, E, out, B, absolute);
  GCNB_LAUNCH_CHECK("k_adjacency_edges");
  return GCNB_OK;
}

}  // namespace gcnb
