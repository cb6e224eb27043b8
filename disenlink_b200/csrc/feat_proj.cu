// feat_proj.cu -- the first layer of the factor MLPs from sparse (CSR / CSC) features, and its weight gradient.
//
// [ref: model.py:24-27,106]  A = act(x W1^T + b1) for the K factors at once, x [N, F] bag-of-words (~1 % dense),
// Wt = W1^T [F, J], act = ReLU (Factor2) or the identity (Factor, nhid == 1).  The dense SGEMM spends 2 N F J
// FLOPs on it; over the nonzeros it is 2 nnz J, bound by gathers of Wt rows (forward) and G' rows (gradient).
//
//   forward   A[n, j]  = act( (sum_{p in row n, CSR order} val[p] Wt[col[p], j]) + b[j] )
//   backward  G'       = G * 1[A > 0]                      (ReLU only: torch's threshold backward on the output)
//             dWt[f, j] = sum_{p in column f, CSC order} val[p] G'[row[p], j]
//             db[j]     = sum_n G'[n, j]
//
// Summation orders are fixed and depend on neither J, the tile width nor the launch shape: every element is one
// sequential fmaf chain over its row's (column's) entries, seeded with +0; db sums FP_DB_ROWS-row partials in row
// order.  A column longer than the chunk length of the caller's plan is cut into chunks that write partial rows
// to scratch, summed in chunk order afterwards (the hub-segment idea of dl_hub_items).  No atomics: the bits are
// the same run to run, and a run's block of a union's Wt gives that run's results on its own.
//
// Warp per (row or CSC item, 128-wide J tile), lane per 4 consecutive j (one float4 when J, the layout and the
// pointers allow it, four scalars otherwise -- the same arithmetic).  Grids are J-tile-major: one tile's F x 128
// block of Wt (or N x 128 block of G') is read by every row before the next tile starts, so it stays in L2 when
// the whole Wt does not (R = 10 runs: 147 MB > 126 MB of L2).
//
// A and G are read and written through a two-level layout: element (n, j) at n * row_stride + (j / blk) *
// blk_stride + j % blk, blk = nhid.  The second layer reads A as the [B, N, nhid] view of [N, J] and its backward
// returns G as a contiguous [B, N, nhid]; both are taken as they are, without a copy.
#include "dl_common.cuh"

namespace {

constexpr int FP_WARPS = 8;
constexpr int FP_THREADS = FP_WARPS * 32;
constexpr int FP_TILE = 128;       // j per warp, 4 per lane
constexpr int FP_DB_ROWS = 64;     // rows per partial of db
constexpr int FP_UNROLL = 4;       // gathers in flight per lane

struct Lay {
  long long rs, bs;
  int blk;
};

__device__ __forceinline__ long long lay_off(const Lay& L, long long n, int j) {
  return n * L.rs + (long long)(j / L.blk) * L.bs + (j % L.blk);
}

template <bool VEC>
__device__ __forceinline__ void load4(const float* __restrict__ p, int j0, int J, float (&o)[4]) {
  if (VEC) {
    if (j0 < J) {
      const float4 t = __ldg(reinterpret_cast<const float4*>(p + j0));
      o[0] = t.x; o[1] = t.y; o[2] = t.z; o[3] = t.w;
    } else {
      o[0] = o[1] = o[2] = o[3] = 0.f;
    }
  } else {
#pragma unroll
    for (int e = 0; e < 4; ++e) o[e] = (j0 + e < J) ? __ldg(p + j0 + e) : 0.f;
  }
}

// acc[e] += sum over entries [p0, p1) in order of val[p] * M[idx[p] * J + j0 + e]   (M row-major [*, J])
// Every lane of the warp must call it (the entries are broadcast with shuffles).
template <bool VEC>
__device__ __forceinline__ void gather_rows(const int* __restrict__ idx, const float* __restrict__ val, long long p0,
                                            long long p1, const float* __restrict__ M, int J, int j0, int lane,
                                            float (&acc)[4]) {
  for (long long base = p0; base < p1; base += 32) {
    const int cnt = (int)((p1 - base) < 32 ? (p1 - base) : 32);
    int c = 0;
    float v = 0.f;
    if (lane < cnt) {
      c = __ldg(idx + base + lane);
      v = __ldg(val + base + lane);
    }
    int q = 0;
    for (; q + FP_UNROLL <= cnt; q += FP_UNROLL) {
      float w[FP_UNROLL][4], vv[FP_UNROLL];
#pragma unroll
      for (int u = 0; u < FP_UNROLL; ++u) {
        const int cc = __shfl_sync(DL_FULL, c, q + u);
        vv[u] = __shfl_sync(DL_FULL, v, q + u);
        load4<VEC>(M + (long long)cc * J, j0, J, w[u]);
      }
#pragma unroll
      for (int u = 0; u < FP_UNROLL; ++u)
#pragma unroll
        for (int e = 0; e < 4; ++e) acc[e] = __fmaf_rn(vv[u], w[u][e], acc[e]);
    }
    for (; q < cnt; ++q) {
      const int cc = __shfl_sync(DL_FULL, c, q);
      const float vq = __shfl_sync(DL_FULL, v, q);
      float w[4];
      load4<VEC>(M + (long long)cc * J, j0, J, w);
#pragma unroll
      for (int e = 0; e < 4; ++e) acc[e] = __fmaf_rn(vq, w[e], acc[e]);
    }
  }
}

// ---- forward: warp per (row, tile), tile-major ------------------------------------------------------------
template <bool VEC>
__global__ void __launch_bounds__(FP_THREADS)
k_feat_proj_fwd(const long long* __restrict__ rowptr, const int* __restrict__ col, const float* __restrict__ val,
                long long N, const float* __restrict__ Wt, const float* __restrict__ b, int J, int relu,
                float* __restrict__ A, Lay la) {
  const long long wg = (long long)blockIdx.x * FP_WARPS + (threadIdx.x >> 5);
  const long long n_tiles = (J + FP_TILE - 1) / FP_TILE;
  if (wg >= N * n_tiles) return;                        // warp-uniform
  const int lane = threadIdx.x & 31;
  const int tile = (int)(wg / N);
  const long long n = wg - (long long)tile * N;
  const int j0 = tile * FP_TILE + lane * 4;
  float acc[4] = {0.f, 0.f, 0.f, 0.f};
  gather_rows<VEC>(col, val, __ldg(rowptr + n), __ldg(rowptr + n + 1), Wt, J, j0, lane, acc);
  if (j0 >= J) return;
  float bj[4], o[4];
  load4<VEC>(b, j0, J, bj);
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    const float t = __fadd_rn(acc[e], bj[e]);
    o[e] = (relu && !(t > 0.f) && t == t) ? 0.f : t;     // torch.relu: NaN passes through
  }
  if (VEC) {
    *reinterpret_cast<float4*>(A + lay_off(la, n, j0)) = make_float4(o[0], o[1], o[2], o[3]);
  } else {
#pragma unroll
    for (int e = 0; e < 4; ++e)
      if (j0 + e < J) A[lay_off(la, n, j0 + e)] = o[e];
  }
}

// ---- backward pass 1: G' = G * 1[A > 0] (contiguous [N, J]) and the db partials of FP_DB_ROWS-row chunks ----
template <bool VEC>
__global__ void __launch_bounds__(FP_THREADS)
k_feat_proj_mask(const float* __restrict__ A, Lay la, const float* __restrict__ G, Lay lg, long long N, int J,
                 int relu, long long n_chunks, float* __restrict__ Gp, float* __restrict__ part) {
  const long long wg = (long long)blockIdx.x * FP_WARPS + (threadIdx.x >> 5);
  const long long n_tiles = (J + FP_TILE - 1) / FP_TILE;
  if (wg >= n_chunks * n_tiles) return;
  const int lane = threadIdx.x & 31;
  const int tile = (int)(wg / n_chunks);
  const long long chunk = wg - (long long)tile * n_chunks;
  const int j0 = tile * FP_TILE + lane * 4;
  if (j0 >= J) return;
  const long long r0 = chunk * FP_DB_ROWS;
  const long long r1 = (r0 + FP_DB_ROWS < N) ? r0 + FP_DB_ROWS : N;
  float acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 4
  for (long long n = r0; n < r1; ++n) {
    float g[4], a[4];
    if (VEC) {
      const float4 tg = __ldg(reinterpret_cast<const float4*>(G + lay_off(lg, n, j0)));
      g[0] = tg.x; g[1] = tg.y; g[2] = tg.z; g[3] = tg.w;
      if (relu) {
        const float4 ta = __ldg(reinterpret_cast<const float4*>(A + lay_off(la, n, j0)));
        a[0] = ta.x; a[1] = ta.y; a[2] = ta.z; a[3] = ta.w;
      }
    } else {
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        g[e] = (j0 + e < J) ? __ldg(G + lay_off(lg, n, j0 + e)) : 0.f;
        a[e] = (relu && j0 + e < J) ? __ldg(A + lay_off(la, n, j0 + e)) : 1.f;
      }
    }
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      if (relu && a[e] <= 0.f) g[e] = 0.f;
      acc[e] = __fadd_rn(acc[e], g[e]);
    }
    if (VEC) {
      *reinterpret_cast<float4*>(Gp + n * J + j0) = make_float4(g[0], g[1], g[2], g[3]);
    } else {
#pragma unroll
      for (int e = 0; e < 4; ++e)
        if (j0 + e < J) Gp[n * J + j0 + e] = g[e];
    }
  }
#pragma unroll
  for (int e = 0; e < 4; ++e)
    if (j0 + e < J) part[chunk * J + j0 + e] = acc[e];
}

// db[j] = the partials of column j summed in chunk order
__global__ void __launch_bounds__(FP_THREADS)
k_feat_proj_db(const float* __restrict__ part, long long n_chunks, int J, float* __restrict__ db) {
  const long long j = (long long)blockIdx.x * FP_THREADS + threadIdx.x;
  if (j >= J) return;
  float acc = 0.f;
  for (long long c = 0; c < n_chunks; ++c) acc = __fadd_rn(acc, __ldg(part + c * J + j));
  db[j] = acc;
}

// ---- backward pass 2: warp per (CSC item, tile), tile-major ----------------------------------------------------
// Items [0, n_slots) are the chunks of the heavy columns and write their partial row to slots[item]; the others
// are whole (possibly empty) columns and write dWt[item_col] directly.
template <bool VEC>
__global__ void __launch_bounds__(FP_THREADS)
k_feat_proj_wgrad(const int* __restrict__ row, const float* __restrict__ cval, const int* __restrict__ item_col,
                  const long long* __restrict__ item_lo, const long long* __restrict__ item_hi, long long n_items,
                  long long n_slots, const float* __restrict__ Gp, int J, float* __restrict__ dWt,
                  float* __restrict__ slots) {
  const long long wg = (long long)blockIdx.x * FP_WARPS + (threadIdx.x >> 5);
  const long long n_tiles = (J + FP_TILE - 1) / FP_TILE;
  if (wg >= n_items * n_tiles) return;
  const int lane = threadIdx.x & 31;
  const int tile = (int)(wg / n_items);
  const long long it = wg - (long long)tile * n_items;
  const int j0 = tile * FP_TILE + lane * 4;
  float acc[4] = {0.f, 0.f, 0.f, 0.f};
  gather_rows<VEC>(row, cval, __ldg(item_lo + it), __ldg(item_hi + it), Gp, J, j0, lane, acc);
  if (j0 >= J) return;
  float* dst = it < n_slots ? slots + it * J : dWt + (long long)__ldg(item_col + it) * J;
  if (VEC) {
    *reinterpret_cast<float4*>(dst + j0) = make_float4(acc[0], acc[1], acc[2], acc[3]);
  } else {
#pragma unroll
    for (int e = 0; e < 4; ++e)
      if (j0 + e < J) dst[j0 + e] = acc[e];
  }
}

// dWt[heavy_col[h], j] = the slots of heavy column h summed in chunk order
__global__ void __launch_bounds__(FP_THREADS)
k_feat_proj_heavy(const float* __restrict__ slots, const int* __restrict__ heavy_col,
                  const long long* __restrict__ heavy_ptr, long long n_heavy, int J, float* __restrict__ dWt) {
  const long long t = (long long)blockIdx.x * FP_THREADS + threadIdx.x;
  if (t >= n_heavy * J) return;
  const long long h = t / J;
  const long long j = t - h * J;
  float acc = 0.f;
  for (long long s = __ldg(heavy_ptr + h); s < __ldg(heavy_ptr + h + 1); ++s)
    acc = __fadd_rn(acc, __ldg(slots + s * J + j));
  dWt[(long long)__ldg(heavy_col + h) * J + j] = acc;
}

inline bool aligned16(const void* p) { return ((uintptr_t)p & 15u) == 0; }

inline bool lay_ok(long long rs, long long bs, long long blk, long long J) {
  return rs >= 0 && bs >= 0 && blk >= 1 && J % blk == 0;
}

// float4 access to (n, j0 .. j0+3) of a layout: the four stay inside one block and are contiguous and aligned
inline bool lay_vec(const float* p, long long rs, long long bs, long long blk) {
  return aligned16(p) && rs % 4 == 0 && bs % 4 == 0 && blk % 4 == 0;
}

inline unsigned blocks_for_warps(long long warps) { return (unsigned)((warps + FP_WARPS - 1) / FP_WARPS); }

inline size_t round256(size_t b) { return (b + 255) & ~(size_t)255; }

}  // namespace

extern "C" {

int dl_feat_proj_fwd(const int64_t* rowptr, const int32_t* col, const float* val, int64_t N, int64_t F,
                     const float* Wt, const float* b, int64_t J, int relu, float* A, int64_t a_row_stride,
                     int64_t a_blk_stride, int64_t blk, dl_stream_t stream) {
  if (N < 0 || F < 0 || J < 1 || J > INT32_MAX || (relu != 0 && relu != 1)) return DL_EINVAL;
  if (!lay_ok(a_row_stride, a_blk_stride, blk, J)) return DL_EINVAL;
  if (N == 0) return DL_OK;
  if (!rowptr || !col || !val || !b || !A || (F > 0 && !Wt)) return DL_EINVAL;
  cudaStream_t st = (cudaStream_t)stream;
  const long long n_tiles = (J + FP_TILE - 1) / FP_TILE;
  const unsigned grid = blocks_for_warps(N * n_tiles);
  const Lay la{a_row_stride, a_blk_stride, (int)blk};
  const bool vec = J % 4 == 0 && aligned16(Wt) && aligned16(b) && lay_vec(A, a_row_stride, a_blk_stride, blk);
  if (vec)
    k_feat_proj_fwd<true><<<grid, FP_THREADS, 0, st>>>((const long long*)rowptr, col, val, N, Wt, b, (int)J, relu,
                                                       A, la);
  else
    k_feat_proj_fwd<false><<<grid, FP_THREADS, 0, st>>>((const long long*)rowptr, col, val, N, Wt, b, (int)J, relu,
                                                        A, la);
  DL_LAUNCH_CHECK();
  return DL_OK;
}

size_t dl_feat_proj_bwd_workspace_bytes(int64_t N, int64_t J, int64_t n_slots) {
  if (N < 0 || J < 1 || n_slots < 0) return 0;
  const size_t n_chunks = (size_t)((N + FP_DB_ROWS - 1) / FP_DB_ROWS);
  return round256((size_t)N * J * sizeof(float)) + round256(n_chunks * J * sizeof(float)) +
         round256((size_t)n_slots * J * sizeof(float));
}

int dl_feat_proj_bwd(const int32_t* row, const float* cval, const int32_t* item_col, const int64_t* item_lo,
                     const int64_t* item_hi, int64_t n_items, int64_t n_slots, const int32_t* heavy_col,
                     const int64_t* heavy_ptr, int64_t n_heavy, int64_t N, int64_t F, const float* A,
                     int64_t a_row_stride, int64_t a_blk_stride, const float* G, int64_t g_row_stride,
                     int64_t g_blk_stride, int64_t blk, int64_t J, int relu, float* dWt, float* db, void* ws,
                     size_t ws_bytes, dl_stream_t stream) {
  if (N < 0 || F < 0 || J < 1 || J > INT32_MAX || (relu != 0 && relu != 1)) return DL_EINVAL;
  if (n_items < 0 || n_slots < 0 || n_heavy < 0 || n_slots > n_items || n_items != F + n_slots - n_heavy)
    return DL_EINVAL;                                   // every light column one item, every heavy column its chunks
  if (!lay_ok(a_row_stride, a_blk_stride, blk, J) || !lay_ok(g_row_stride, g_blk_stride, blk, J)) return DL_EINVAL;
  if (!db || (F > 0 && !dWt) || (n_items > 0 && (!item_col || !item_lo || !item_hi))) return DL_EINVAL;
  if (n_heavy > 0 && (!heavy_col || !heavy_ptr)) return DL_EINVAL;
  if (N > 0 && (!G || (relu && !A) || !row || !cval)) return DL_EINVAL;
  if (!ws || ws_bytes < dl_feat_proj_bwd_workspace_bytes(N, J, n_slots)) return DL_EWORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  const long long n_tiles = (J + FP_TILE - 1) / FP_TILE;
  const long long n_chunks = (N + FP_DB_ROWS - 1) / FP_DB_ROWS;
  float* Gp = (float*)ws;
  float* part = (float*)((char*)ws + round256((size_t)N * J * sizeof(float)));
  float* slots = (float*)((char*)part + round256((size_t)n_chunks * J * sizeof(float)));
  const Lay la{a_row_stride, a_blk_stride, (int)blk}, lg{g_row_stride, g_blk_stride, (int)blk};
  if (n_chunks > 0) {
    const bool vec = J % 4 == 0 && aligned16(Gp) && lay_vec(G, g_row_stride, g_blk_stride, blk) &&
                     (!relu || lay_vec(A, a_row_stride, a_blk_stride, blk));
    const unsigned grid = blocks_for_warps(n_chunks * n_tiles);
    if (vec)
      k_feat_proj_mask<true><<<grid, FP_THREADS, 0, st>>>(A, la, G, lg, N, (int)J, relu, n_chunks, Gp, part);
    else
      k_feat_proj_mask<false><<<grid, FP_THREADS, 0, st>>>(A, la, G, lg, N, (int)J, relu, n_chunks, Gp, part);
    DL_LAUNCH_CHECK();
  }
  k_feat_proj_db<<<(unsigned)((J + FP_THREADS - 1) / FP_THREADS), FP_THREADS, 0, st>>>(part, n_chunks, (int)J, db);
  DL_LAUNCH_CHECK();
  if (n_items > 0) {
    const bool vec = J % 4 == 0 && aligned16(Gp) && aligned16(dWt) && aligned16(slots);
    const unsigned grid = blocks_for_warps(n_items * n_tiles);
    if (vec)
      k_feat_proj_wgrad<true><<<grid, FP_THREADS, 0, st>>>(row, cval, item_col, (const long long*)item_lo,
                                                           (const long long*)item_hi, n_items, n_slots, Gp,
                                                           (int)J, dWt, slots);
    else
      k_feat_proj_wgrad<false><<<grid, FP_THREADS, 0, st>>>(row, cval, item_col, (const long long*)item_lo,
                                                            (const long long*)item_hi, n_items, n_slots, Gp,
                                                            (int)J, dWt, slots);
    DL_LAUNCH_CHECK();
  }
  if (n_heavy > 0) {
    k_feat_proj_heavy<<<(unsigned)((n_heavy * J + FP_THREADS - 1) / FP_THREADS), FP_THREADS, 0, st>>>(
        slots, heavy_col, (const long long*)heavy_ptr, n_heavy, (int)J, dWt);
    DL_LAUNCH_CHECK();
  }
  return DL_OK;
}

}  // extern "C"
