// bwd_dir.cu -- backward of the factor attention + aggregation w.r.t. Z for ANY 0/1 pattern
// (graphs marked directed).
//
// [ref: autograd of model.py:56-75].  For a symmetric pattern factor_bwd.cu collects the (j,i) term of
// every entry from the mirror entry in row j.  A directed pattern has no mirror, so the terms an entry
// sends to its column node are gathered over the transposed pattern instead: gt (a dl_graph of its own,
// row j = the in-entries of node j, with degree buckets and hub items) and tperm[p] = CSR index of
// in-entry p.  Closed form, entry e = (i,j) of A, k = kstar[e]:
//   pass 1 (k_dir_gather, per node j over its in-entries, view gt):
//     T_[j,k,:] = (1-beta)/s[j,k] * sum_{e=(i,j), kstar=k} w[e] G[i,k,:]
//     r[j,k]    = <Z[j,k], T_[j,k]> / s[j,k]  if row j of A has an entry routed to k, else 0
//     dZ[j,:]  += beta G[j,:] + T_[j,:]
//   pass 2, out-side (k_dir_edges<false>, per row i over its entries, view g):
//     dw[e]      = (1-beta) <G[i,k], Z[j,k]> / s[j,k] - r[i,k]         (kept per entry for the in-side)
//     coef[e,kk] = dw[e] a[e,k] / T ((kk==k) - a[e,kk])
//     dZ[i,kk,:] += coef[e,kk] Z[j,kk,:]
//   pass 2, in-side (k_dir_edges<true>, per node j over its in-entries, view gt):
//     dZ[j,kk,:] += coef[e,kk] Z[i,kk,:]       with dw[e] read through tperm, a[e,:] recomputed
// The clamp rule: the reference sets s = 1 where a (node, factor) has no routed out-entry, so no
// gradient flows through that s and r is 0 there.  s == 1 cannot tell (at K = 1, s is the out-degree),
// so the bit comes from the CSR and kstar (k_routed_mask).  In a symmetric pattern an in-entry routed to
// k implies an out-entry routed to k; in a directed one sinks and in-only factors break that.
//
// Every launch has one writer per dZ row (hub rows: per-segment partials in scratch, summed in segment
// order by a fixup kernel), no floating-point atomics, fixed summation orders: bitwise run-to-run
// deterministic.  Runtime (K, d): every shape dl_shape_ok accepts.  The softmax a[e,:] is recomputed
// with dl_generic_route, the canonical arithmetic of the forward (same bits as w and kstar).
//
// HBM bytes per entry (D = K d): mask 1;  pass 1  4 + 4 + 1 + 4 + 4d;  pass 2 out  4 + 1 + 4D + 4 + 4;
// pass 2 in  4 + 4 + 1 + 4 + 4D.
#include "dl_dispatch.cuh"

namespace {

constexpr int R1 = DL_MAX_D / 32;   // pass 1: one factor slice per lane group of 32
constexpr int R2 = 8;               // pass 2: 256-float windows of the row in registers

__device__ __forceinline__ float dir_warp_sum(float v) {
  for (int o = 16; o > 0; o >>= 1) v = __fadd_rn(v, __shfl_xor_sync(DL_FULL, v, o));
  return v;
}

// routed[i] bit k = row i has an entry with kstar == k
__global__ void __launch_bounds__(DL_CTA)
k_routed_mask(DlGraphDev g, const unsigned char* __restrict__ kstar, unsigned* __restrict__ routed) {
  const int lane = threadIdx.x & 31;
  const long long warp0 = (long long)blockIdx.x * DL_WARPS_PER_CTA + (threadIdx.x >> 5);
  const long long nwarps = (long long)gridDim.x * DL_WARPS_PER_CTA;
  for (long long row = warp0; row < g.N; row += nwarps) {
    unsigned m = 0;
    for (long long p = __ldg(g.rowptr + row) + lane; p < __ldg(g.rowptr + row + 1); p += 32)
      m |= 1u << __ldg(kstar + p);
    m = __reduce_or_sync(DL_FULL, m);
    if (lane == 0) routed[g.row_base + row] = m;
  }
}

// T_, r and dZ += beta G + T_ of factor k of node j from the summed slice acc (lane-strided over d)
__device__ __forceinline__ void dir_finish(long long j, int k, const float (&acc)[R1], unsigned has,
                                           const float* __restrict__ Z, const float* __restrict__ G,
                                           const float* __restrict__ s, int K, int d, float beta, float omb,
                                           float* __restrict__ dZ, float* __restrict__ r, int lane) {
  const long long D = (long long)K * d;
  const float sk = __ldg(s + j * K + k);
  const float scale = __fdiv_rn(omb, sk);
  float part = 0.0f;
#pragma unroll
  for (int x = 0; x < R1; ++x) {
    const int e = lane + 32 * x;
    if (e < d) {
      const float tv = __fmul_rn(scale, acc[x]);
      part = __fmaf_rn(Z[j * D + (long long)k * d + e], tv, part);
      float* dst = dZ + j * D + (long long)k * d + e;
      *dst = __fadd_rn(*dst, __fmaf_rn(beta, G[j * D + (long long)k * d + e], tv));
    }
  }
  part = dir_warp_sum(part);
  if (lane == 0) r[j * K + k] = ((has >> k) & 1u) ? __fdiv_rn(part, sk) : 0.0f;
}

// pass 1 over the transposed view: per factor the node's in-entries are rescanned so the accumulator
// fits in registers; the entries routed to k are picked with a ballot and summed in CSR order
__global__ void __launch_bounds__(DL_CTA)
k_dir_gather(DlGraphDev gt, const int* __restrict__ tperm, const float* __restrict__ Z,
             const float* __restrict__ G, const unsigned char* __restrict__ kstar, const float* __restrict__ w,
             const float* __restrict__ s, const unsigned* __restrict__ routed, int K, int d, float beta,
             float omb, float* __restrict__ dZ, float* __restrict__ r, float* __restrict__ hub_ws) {
  const int lane = threadIdx.x & 31;
  const long long warp0 = (long long)blockIdx.x * DL_WARPS_PER_CTA + (threadIdx.x >> 5);
  const long long nwarps = (long long)gridDim.x * DL_WARPS_PER_CTA;
  const long long n_items = dl_num_items(gt);
  const long long D = (long long)K * d;
  for (long long t = warp0; t < n_items; t += nwarps) {
    const DlItem it = dl_decode_item(gt, t);
    const unsigned has = it.hub_slot < 0 ? __ldg(routed + it.node) : 0u;
    for (int k = 0; k < K; ++k) {
      float acc[R1];
#pragma unroll
      for (int x = 0; x < R1; ++x) acc[x] = 0.0f;
      for (long long base = it.e0; base < it.e1; base += 32) {
        const int cnt = (int)min(32LL, it.e1 - base);
        int src = 0;
        float wv = 0.0f;
        bool mine = false;
        if (lane < cnt) {
          const int e = __ldg(tperm + base + lane);
          mine = __ldg(kstar + e) == k;
          if (mine) {
            src = __ldg(gt.col + base + lane);
            wv = __ldg(w + e);
          }
        }
        unsigned m = __ballot_sync(DL_FULL, mine);
        while (m) {
          const int b = __ffs(m) - 1;
          m &= m - 1;
          const long long i = __shfl_sync(DL_FULL, src, b);
          const float wb = __shfl_sync(DL_FULL, wv, b);
          const float* gi = G + i * D + (long long)k * d;
#pragma unroll
          for (int x = 0; x < R1; ++x) {
            const int e = lane + 32 * x;
            if (e < d) acc[x] = __fmaf_rn(wb, __ldg(gi + e), acc[x]);
          }
        }
      }
      if (it.hub_slot >= 0) {
#pragma unroll
        for (int x = 0; x < R1; ++x) {
          const int e = lane + 32 * x;
          if (e < d) hub_ws[it.hub_slot * D + (long long)k * d + e] = acc[x];
        }
      } else {
        dir_finish(it.node, k, acc, has, Z, G, s, K, d, beta, omb, dZ, r, lane);
      }
    }
  }
}

// pass 1, in-hub nodes: segment partials summed in segment order, then finished like a direct node
__global__ void __launch_bounds__(DL_CTA)
k_dir_gather_hub(DlGraphDev gt, const float* __restrict__ Z, const float* __restrict__ G,
                 const float* __restrict__ s, const unsigned* __restrict__ routed, int K, int d, float beta,
                 float omb, float* __restrict__ dZ, float* __restrict__ r, const float* __restrict__ hub_ws) {
  const int lane = threadIdx.x & 31;
  const long long warp0 = (long long)blockIdx.x * DL_WARPS_PER_CTA + (threadIdx.x >> 5);
  const long long nwarps = (long long)gridDim.x * DL_WARPS_PER_CTA;
  const long long D = (long long)K * d;
  for (long long h = warp0; h < gt.n_hub; h += nwarps) {
    const long long a = gt.hub_seg_ptr[h], b = gt.hub_seg_ptr[h + 1];
    const long long j = gt.row_base + gt.perm[h];
    const unsigned has = __ldg(routed + j);
    for (int k = 0; k < K; ++k) {
      float acc[R1];
#pragma unroll
      for (int x = 0; x < R1; ++x) {
        const int e = lane + 32 * x;
        acc[x] = 0.0f;
        if (e < d)
          for (long long sg = a; sg < b; ++sg) acc[x] = __fadd_rn(acc[x], hub_ws[sg * D + (long long)k * d + e]);
      }
      dir_finish(j, k, acc, has, Z, G, s, K, d, beta, omb, dZ, r, lane);
    }
  }
}

// pass 2.  IN = false: view g, own node = row i, other = column j, entry index = p; computes dw[e] and
// keeps it.  IN = true: view gt, own node = j, other = source i, entry index = tperm[p]; reads dw[e].
// The row of the own node is accumulated in 256-float windows held in registers.
template <bool IN>
__global__ void __launch_bounds__(DL_CTA)
k_dir_edges(DlGraphDev g, const int* __restrict__ tperm, const float* __restrict__ Z,
            const float* __restrict__ G, const unsigned char* __restrict__ kstar, const float* __restrict__ s,
            const float* __restrict__ r, int K, int d, float omb, float T, float* __restrict__ dw,
            float* __restrict__ dZ, float* __restrict__ hub_ws) {
  const int lane = threadIdx.x & 31;
  const long long warp0 = (long long)blockIdx.x * DL_WARPS_PER_CTA + (threadIdx.x >> 5);
  const long long nwarps = (long long)gridDim.x * DL_WARPS_PER_CTA;
  const long long n_items = dl_num_items(g);
  const long long D = (long long)K * d;
  float ev[DL_MAX_K], a[DL_MAX_K];
  for (long long t = warp0; t < n_items; t += nwarps) {
    const DlItem it = dl_decode_item(g, t);
    const long long v = it.node;
    const float* zv = Z + v * D;
    for (long long w0 = 0; w0 < D; w0 += 32 * R2) {
      float acc[R2];
#pragma unroll
      for (int q = 0; q < R2; ++q) acc[q] = 0.0f;
      for (long long p = it.e0; p < it.e1; ++p) {
        const long long u = __ldg(g.col + p);
        const long long ent = IN ? (long long)__ldg(tperm + p) : p;
        const float* zu = Z + u * D;
        // the forward's argument order (row node, column node)
        dl_generic_route(IN ? zu : zv, IN ? zv : zu, K, d, T, lane, ev, a);
        const int k = __ldg(kstar + ent);
        float dwv;
        if (IN) {
          dwv = __ldg(dw + ent);
        } else {
          float c = 0.0f;
          for (int x = lane; x < d; x += 32) c = __fmaf_rn(G[v * D + (long long)k * d + x], zu[(long long)k * d + x], c);
          c = __fmul_rn(omb, dir_warp_sum(c));
          dwv = __fsub_rn(__fdiv_rn(c, __ldg(s + u * K + k)), __ldg(r + v * K + k));
          if (lane == 0 && w0 == 0) dw[ent] = dwv;
        }
        const float basec = __fdiv_rn(__fmul_rn(dwv, a[k]), T);
#pragma unroll
        for (int q = 0; q < R2; ++q) {
          const long long x = w0 + lane + 32 * q;
          if (x < D) {
            const int kk = (int)(x / d);
            const float coef = __fmul_rn(basec, __fsub_rn((kk == k) ? 1.0f : 0.0f, a[kk]));
            acc[q] = __fmaf_rn(coef, zu[x], acc[q]);
          }
        }
      }
#pragma unroll
      for (int q = 0; q < R2; ++q) {
        const long long x = w0 + lane + 32 * q;
        if (x >= D) continue;
        if (it.hub_slot >= 0) {
          hub_ws[it.hub_slot * D + x] = acc[q];
        } else {
          float* dst = dZ + v * D + x;
          *dst = __fadd_rn(*dst, acc[q]);
        }
      }
    }
  }
}

// hub rows of pass 2: dZ[row] += sum of segment partials (in order)
__global__ void k_dir_hub_fixup(DlGraphDev g, long long D, const float* __restrict__ hub_ws,
                                float* __restrict__ dZ) {
  long long stride = (long long)gridDim.x * blockDim.x;
  for (long long x = (long long)blockIdx.x * blockDim.x + threadIdx.x; x < g.n_hub * D; x += stride) {
    long long h = x / D, o = x % D;
    long long a = g.hub_seg_ptr[h], b = g.hub_seg_ptr[h + 1];
    float v = 0.0f;
    for (long long sg = a; sg < b; ++sg) v = __fadd_rn(v, hub_ws[sg * D + o]);
    long long row = g.row_base + g.perm[h];
    dZ[row * D + o] = __fadd_rn(dZ[row * D + o], v);
  }
}

inline int fixup_blocks(long long n) {
  long long b = (n + 255) / 256;
  if (b < 1) b = 1;
  if (b > 148 * 16) b = 148 * 16;
  return (int)b;
}

template <bool IN>
int launch_dir_edges(const DlGraphDev& g, const int* tperm, const float* Z, const float* G, const uint8_t* kstar,
                     const float* s, const float* r, int K, int d, float omb, float T, float* dw, float* dZ,
                     float* hub_ws, cudaStream_t st) {
  int grid = 1;
  int rc = dl_grid_for(k_dir_edges<IN>, g.n_hub_items + (g.N - g.n_hub), &grid);
  if (rc) return rc;
  k_dir_edges<IN><<<grid, DL_CTA, 0, st>>>(g, tperm, Z, G, kstar, s, r, K, d, omb, T, dw, dZ, hub_ws);
  DL_LAUNCH_CHECK();
  if (g.n_hub > 0) {
    const long long D = (long long)K * d;
    k_dir_hub_fixup<<<fixup_blocks(g.n_hub * D), 256, 0, st>>>(g, D, hub_ws, dZ);
    DL_LAUNCH_CHECK();
  }
  return DL_OK;
}

// the three phases of the directed backward; arguments validated by the caller
int dir_phase(const DlGraphDev& g, const DlGraphDev& gt, const int32_t* tperm, const float* Z, const float* G,
              const uint8_t* kstar, const float* w, const float* s, int K, int d, float beta, float omb, float T,
              float* dZ, float* r, float* dw, uint32_t* routed, float* hub_ws, float* hub_ws_t, int phase,
              cudaStream_t st) {
  int grid = 1, rc = DL_OK;
  switch (phase) {
    case 1:
      rc = dl_grid_for(k_routed_mask, g.N, &grid);
      if (rc) return rc;
      k_routed_mask<<<grid, DL_CTA, 0, st>>>(g, kstar, routed);
      DL_LAUNCH_CHECK();
      rc = dl_grid_for(k_dir_gather, gt.n_hub_items + (gt.N - gt.n_hub), &grid);
      if (rc) return rc;
      k_dir_gather<<<grid, DL_CTA, 0, st>>>(gt, tperm, Z, G, kstar, w, s, routed, K, d, beta, omb, dZ, r, hub_ws_t);
      DL_LAUNCH_CHECK();
      if (gt.n_hub > 0) {
        rc = dl_grid_for(k_dir_gather_hub, gt.n_hub, &grid);
        if (rc) return rc;
        k_dir_gather_hub<<<grid, DL_CTA, 0, st>>>(gt, Z, G, s, routed, K, d, beta, omb, dZ, r, hub_ws_t);
        DL_LAUNCH_CHECK();
      }
      return DL_OK;
    case 2:
      return launch_dir_edges<false>(g, nullptr, Z, G, kstar, s, r, K, d, omb, T, dw, dZ, hub_ws, st);
    case 3:
      return launch_dir_edges<true>(gt, tperm, Z, G, kstar, s, r, K, d, omb, T, dw, dZ, hub_ws_t, st);
    default:
      return DL_EINVAL;
  }
}

// status |= 1 when some index of a[0, n) is outside [0, bound)
__global__ void k_dir_bounds(const int32_t* __restrict__ a, long long n, long long bound, int* __restrict__ status) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  bool bad = false;
  for (long long x = (long long)blockIdx.x * blockDim.x + threadIdx.x; x < n; x += stride) {
    const int v = __ldg(a + x);
    bad |= v < 0 || (long long)v >= bound;
  }
  if (__syncthreads_or(bad) && threadIdx.x == 0) atomicOr(status, 1);
}

}  // namespace

extern "C" {

int dl_factor_bwd_directed(const dl_graph* g_host, const dl_graph* gt_host, const int32_t* tperm,
                           const float* Z, const float* G, const uint8_t* kstar, const float* w, const float* s,
                           int K, int d, float beta, float one_minus_beta, float T, float* dZ, float* r,
                           float* dw_scratch, uint32_t* routed_scratch, float* hub_ws, float* hub_ws_t,
                           dl_stream_t stream) {
  if (!dl_graph_ok(g_host) || !dl_graph_ok(gt_host) || !dl_shape_ok(K, d)) return DL_EINVAL;
  if (gt_host->N != g_host->N || gt_host->nnz != g_host->nnz) return DL_EINVAL;
  if (g_host->row_base != 0 || gt_host->row_base != 0) return DL_EINVAL;
  if (!(T == T) || T == 0.0f) return DL_EINVAL;
  if (g_host->N == 0) return DL_OK;
  if (!Z || !G || !s || !dZ || !r || !routed_scratch) return DL_EINVAL;
  if (g_host->nnz > 0 && (!kstar || !w || !tperm || !dw_scratch)) return DL_EINVAL;
  if ((g_host->n_hub_items > 0 && !hub_ws) || (gt_host->n_hub_items > 0 && !hub_ws_t)) return DL_EINVAL;
  cudaStream_t st = (cudaStream_t)stream;
  const DlGraphDev g = dl_graph_dev(g_host);
  const DlGraphDev gt = dl_graph_dev(gt_host);
  for (int phase = 1; phase <= 3; ++phase) {
    const int rc = dir_phase(g, gt, tperm, Z, G, kstar, w, s, K, d, beta, one_minus_beta, T, dZ, r, dw_scratch,
                             routed_scratch, hub_ws, hub_ws_t, phase, st);
    if (rc) return rc;
  }
  return DL_OK;
}

int dl_factor_bwd_directed_phase(const dl_graph* g_host, const dl_graph* gt_host, const int32_t* tperm,
                                 const float* Z, const float* G, const uint8_t* kstar, const float* w,
                                 const float* s, int K, int d, float beta, float one_minus_beta, float T,
                                 int64_t n_tot, int64_t n_rec, float* dZ, float* r, float* dw,
                                 uint32_t* routed_scratch, float* hub_ws, float* hub_ws_t, int phase,
                                 dl_stream_t stream) {
  if (phase < 1 || phase > 3) return DL_EINVAL;
  if (!dl_graph_ok(g_host) || !dl_graph_ok(gt_host) || !dl_shape_ok(K, d)) return DL_EINVAL;
  if (gt_host->N != g_host->N || g_host->row_base != 0 || gt_host->row_base != 0) return DL_EINVAL;
  if (n_tot < g_host->N || n_tot >= (1LL << 31) || n_rec < g_host->nnz || n_rec >= (1LL << 31)) return DL_EINVAL;
  if (!(T == T) || T == 0.0f) return DL_EINVAL;
  if (g_host->N == 0) return DL_OK;
  const bool out_side = phase != 3, in_side = phase != 2;
  if (!Z || !dZ || (phase != 3 && (!G || !s || !r)) || (phase == 1 && !routed_scratch)) return DL_EINVAL;
  if ((out_side && g_host->nnz > 0 && !kstar) || (in_side && gt_host->nnz > 0 && (!kstar || !tperm))) return DL_EINVAL;
  if ((phase == 1 && gt_host->nnz > 0 && !w) || (phase == 2 && g_host->nnz > 0 && !dw) ||
      (phase == 3 && gt_host->nnz > 0 && !dw))
    return DL_EINVAL;
  if ((phase == 2 && g_host->n_hub_items > 0 && !hub_ws) || (in_side && gt_host->n_hub_items > 0 && !hub_ws_t))
    return DL_EINVAL;
  cudaStream_t st = (cudaStream_t)stream;
  const DlGraphDev g = dl_graph_dev(g_host);
  const DlGraphDev gt = dl_graph_dev(gt_host);
  // the phase's column and record indices against n_tot / n_rec: one pass and one synchronisation
  const long long n_g = phase == 2 ? g.nnz : 0, n_t = in_side ? gt.nnz : 0;
  if (n_g + n_t > 0) {
    int* status = nullptr;
    DL_CUDA_TRY(cudaMallocAsync((void**)&status, sizeof(int), st));
    DL_CUDA_TRY(cudaMemsetAsync(status, 0, sizeof(int), st));
    if (n_g > 0) k_dir_bounds<<<fixup_blocks(n_g), 256, 0, st>>>(g.col, n_g, n_tot, status);
    if (n_t > 0) {
      k_dir_bounds<<<fixup_blocks(n_t), 256, 0, st>>>(gt.col, n_t, n_tot, status);
      k_dir_bounds<<<fixup_blocks(n_t), 256, 0, st>>>(tperm, n_t, n_rec, status);
    }
    int bad = 0;
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaMemcpyAsync(&bad, status, sizeof(int), cudaMemcpyDeviceToHost, st);
    cudaFreeAsync(status, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return (int)e;
    if (bad) return DL_EINVAL;
  }
  return dir_phase(g, gt, tperm, Z, G, kstar, w, s, K, d, beta, one_minus_beta, T, dZ, r, dw, routed_scratch, hub_ws,
                   hub_ws_t, phase, st);
}

}  // extern "C"
