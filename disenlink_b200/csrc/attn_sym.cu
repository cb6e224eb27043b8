// attn_sym.cu -- symmetric evaluation of the per-edge factor attention.
//
// [ref: model.py:56-73]  q_k(i,j) = <Z[i,k], Z[j,k]> / T is symmetric in (i,j), and with the canonical
// arithmetic of dl_common.cuh so are, BIT FOR BIT, the softmax a, the routed factor kstar and its weight
// w.  The adjacency is symmetric too (main_disentangled.py:141-142), so the attention kernel of
// attn_fl.cu -- which gathers the 512-byte row Z[j] for entry (i,j) AND Z[i] for entry (j,i) -- does
// every undirected edge twice.  Here each edge is evaluated once:
//
//   1. (integer, once per graph)  dl_sym_index: the PRIMARY view of the CSR (of the two entries of an edge
//      the one whose row has the larger degree, see dl_primary: rowptr uptr, columns ucol) and, for EVERY
//      entry e of the full CSR, eidx[e] = its position in the primary view, or ~(its mirror's position)
//      for a secondary entry.  ("upper" / "lower" in names = primary / secondary.)
//   2. k_attn_fl on the upper view: one row gather per undirected edge, result written as one packed
//      8-byte record kw[t] = (w, kstar) per upper entry (coalesced); optionally also the softmax a[t, :]
//      (4K bytes per upper entry, coalesced), which backward pass 2 then reads instead of recomputing it.
//   3. k_sym_expand (this file): a streaming pass over the full CSR that reads kw[eidx[e]] -- sequential
//      for the upper entries of a row, one random 8-byte access for the lower ones --, writes kstar[e]
//      and w[e] in the layout every other kernel reads, and makes the routed row sums s[i,k] in CSR
//      order (deterministic; rows cut by a range boundary go through the carry / chain mechanism of
//      gather_stream.cu, mode 2).
//
// Row gathers: nnz/2 x 4D bytes instead of nnz x 4D; extra: nnz x (4 + 4 + 5) streaming bytes and
// nnz/2 random 8-byte reads.  kstar / w are bit-identical to the two-sided evaluation.
#include "dl_dispatch.cuh"
#include "dl_prims.cuh"
#include "dl_stream.cuh"

namespace {

inline int blocks_for(long long n, int threads = 256) {
  long long b = (n + threads - 1) / threads;
  if (b < 1) b = 1;
  if (b > 148 * 32) b = 148 * 32;
  return (int)b;
}

// Which of the two entries (i,j), (j,i) of an undirected edge is evaluated ("primary")?  The one whose ROW
// has the larger degree (ties: the smaller id; a diagonal entry is its own mirror and primary).  Any
// antisymmetric rule would do for correctness; this one keeps the long rows long: a hub row keeps nearly all
// of its entries, the many low-degree rows keep few or none, so the per-row costs of the evaluating kernels
// (own-row loads, accumulator flush: measured at ~10 entries' worth per row start in backward pass 2) are
// paid for ~N/4 rows instead of N, where an id-based rule (col >= row) halves every row.
__device__ __forceinline__ bool dl_primary(const long long* __restrict__ rowptr, int i, int j) {
  if (i == j) return true;
  const long long di = __ldg(rowptr + i + 1) - __ldg(rowptr + i), dj = __ldg(rowptr + j + 1) - __ldg(rowptr + j);
  return di > dj || (di == dj && i < j);
}

struct PrimaryFlag {
  const long long* rowptr;
  const int* col;
  const int* erow;
  long long nnz;
  __device__ __forceinline__ int operator()(long long e) const {
    return (e < nnz && dl_primary(rowptr, erow[e], col[e])) ? 1 : 0;
  }
};

__global__ void k_sym_uptr(const long long* __restrict__ rowptr, const int* __restrict__ pos, long long N,
                           long long* __restrict__ uptr) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x; r <= N; r += stride) uptr[r] = pos[rowptr[r]];
}

// pos[e] = number of primary entries before e (their position in the primary view)
__global__ void k_sym_fill(const long long* __restrict__ rowptr, const int* __restrict__ col,
                           const int* __restrict__ erow, long long nnz, const int* __restrict__ pos,
                           int* __restrict__ ucol, int* __restrict__ eidx,
                           int* __restrict__ lcol, int* __restrict__ lmirror, int* __restrict__ status,
                           unsigned long long* __restrict__ n_diag) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < nnz; e += stride) {
    const int i = erow[e], j = col[e];
    if (j == i) atomicAdd(n_diag, 1ULL);          // integer count: order independent
    const int t = pos[e];
    if (pos[e + 1] != t) {                         // primary
      ucol[t] = j;
      eidx[e] = t;
    } else {                                       // secondary: its mirror (j, i) is primary, in row j
      long long a = rowptr[j], b = rowptr[j + 1];
      const long long b0 = b;
      while (a < b) {
        const long long mid = (a + b) >> 1;
        if (col[mid] < i) a = mid + 1; else b = mid;
      }
      int m = 0;
      if (a < b0 && col[a] == i && pos[a + 1] != pos[a]) {
        m = pos[a];
      } else {
        *status = DL_EASYM;
      }
      eidx[e] = ~m;                                // negative: "read the record of entry ~eidx in the primary view"
      if (lcol) {                                  // secondary view: entry e is its (e - pos[e])-th entry
        lcol[e - t] = j;
        lmirror[e - t] = m;
      }
    }
  }
}

// every secondary entry found a primary mirror (k_sym_fill); the pattern is symmetric iff, in addition, no
// primary off-diagonal entry is left without one: #secondary == #primary - #diagonal
__global__ void k_sym_check(long long nnz, const int* __restrict__ pos,
                            const unsigned long long* __restrict__ n_diag, int* __restrict__ status) {
  const long long nu = pos[nnz];
  if (nnz - nu != nu - (long long)*n_diag) *status = DL_EASYM;
}

// ---- the expand pass ----------------------------------------------------------------------------
constexpr int SX_WARPS = 8;

template <int KP>     // KP = 8 (K <= 8: 4 entries per step) or 32 (K <= 32: 1 entry per step)
__global__ void __launch_bounds__(SX_WARPS * 32)
k_sym_expand(DlGraphDev g, const int* __restrict__ eidx, const float2* __restrict__ kw, int K,
             unsigned char* __restrict__ kstar, float* __restrict__ w, float* __restrict__ s,
             float* __restrict__ carry) {
  const int lane = threadIdx.x & 31;
  const long long gw = (long long)blockIdx.x * SX_WARPS + (threadIdx.x >> 5);
  const long long RE = (long long)DL_CH * DL_RANGE;
  DlChunkStream cs;
  cs.init(g.nnz, (long long)gridDim.x * SX_WARPS, g.range_shift);

  // lane k (of every group of KP lanes) accumulates factor k of the current row; with KP = 8 the
  // four lane groups take the entries of a chunk round robin and are summed in a fixed order at the
  // end of the row (the association attn_fl.cu uses)
  constexpr int NG = 32 / KP;
  const int grp = lane / KP, kap = lane % KP;
  float acc = 0.0f;
  int cur_row = -1;
  bool first_run = true, head_open = false, tail_open = false;
  long long cur_range = -1;
  auto flush = [&](bool at_range_end) {
    if (cur_row >= 0) {
      float v = acc;
#pragma unroll
      for (int off = KP; off < 32; off <<= 1) v = __fadd_rn(v, __shfl_xor_sync(DL_FULL, v, off));
      const bool to_head = first_run && head_open;
      const bool to_tail = !to_head && at_range_end && tail_open;
      if (grp == 0 && kap < K) {
        if (to_head || to_tail) carry[(cur_range * 2 + (to_tail ? 1 : 0)) * K + kap] = v;
        else s[(g.row_base + cur_row) * K + kap] = (v == 0.0f) ? 1.0f : v;
      }
      first_run = false;
    }
    cur_row = -1;
    acc = 0.0f;
  };

  struct Meta { int row, idx; };
  auto load_meta = [&](long long cc, Meta& m) {
    m.row = -1; m.idx = 0;
    if (cc >= 0) {
      const long long e = cc * DL_CH + lane;
      if (e < g.nnz) {
        m.row = __ldg(g.erow + e);
        const int t = __ldg(eidx + e);
        m.idx = t < 0 ? ~t : t;             // own record (primary entry) or the mirror's (secondary)
      }
    }
  };
  auto gather = [&](const Meta& m) {
    float2 v = make_float2(0.0f, 0.0f);
    if (m.row >= 0) {
      asm volatile("ld.global.nc.L2::64B.v2.f32 {%0,%1}, [%2];" : "=f"(v.x), "=f"(v.y) : "l"(kw + m.idx));
    }
    return v;
  };

  long long c = cs.first(gw);
  Meta mA, mB, mC;
  load_meta(c, mA);
  long long cn = cs.next(c);
  load_meta(cn, mB);
  float2 vA = gather(mA), vB;
  while (c >= 0) {
    const long long cnn = cs.next(cn);
    load_meta(cnn, mC);                 // ids two chunks ahead, records one chunk ahead
    vB = gather(mB);
    const long long rg = c >> g.range_shift;
    if (rg != cur_range) {
      if (cur_range >= 0) flush(true);
      cur_range = rg;
      first_run = true;
      const long long R0 = rg * RE, R1 = min(R0 + RE, g.nnz);
      head_open = R0 > 0 && __ldg(g.erow + R0 - 1) == __ldg(g.erow + R0);
      tail_open = R1 < g.nnz && __ldg(g.erow + R1) == __ldg(g.erow + R1 - 1);
    }
    const int ks = __float_as_int(vA.y);
    if (mA.row >= 0) {
      const long long e = c * DL_CH + lane;
      kstar[e] = (unsigned char)ks;
      w[e] = vA.x;
    }
    const unsigned vmask = __ballot_sync(DL_FULL, mA.row >= 0);
    const int cnt = __popc(vmask);
    // walk the chunk NG entries per step; steps whose entries all continue the current row (the
    // common case) need no row bookkeeping
    for (int q = 0; q < cnt; q += NG) {
      const int src = q + grp;
      const int row_e = __shfl_sync(DL_FULL, mA.row, src & 31);
      const int ks_e = __shfl_sync(DL_FULL, ks, src & 31);
      const float w_e = __shfl_sync(DL_FULL, vA.x, src & 31);
      const bool valid = src < cnt;
      const float contrib = (valid && kap == ks_e) ? w_e : 0.0f;
      if (!__any_sync(DL_FULL, valid && row_e != cur_row)) {
        acc = __fadd_rn(acc, contrib);
      } else {
#pragma unroll 1
        for (int t = 0; t < NG && q + t < cnt; ++t) {
          const int re = __shfl_sync(DL_FULL, mA.row, q + t);
          if (re != cur_row) { flush(false); cur_row = re; }
          if (grp == t) acc = __fadd_rn(acc, contrib);
        }
      }
    }
    c = cn; cn = cnn;
    mA = mB; mB = mC;
    vA = vB;
  }
  if (cur_range >= 0) flush(true);
}

}  // namespace

extern "C" {

size_t dl_sym_index_workspace_bytes(int64_t N, int64_t nnz) {
  if (N < 0 || nnz < 0) return 0;
  return dlp::align256((size_t)(nnz + 2) * 4) + dlp::scan_ws_bytes(nnz + 1, 4) + 256;
}

int dl_sym_index(const int64_t* rowptr, const int32_t* col, const int32_t* erow, int64_t N, int64_t nnz,
                 int64_t* uptr, int32_t* ucol, int32_t* eidx, int32_t* lcol, int32_t* lmirror, int32_t* status_out,
                 void* ws, size_t ws_bytes, dl_stream_t stream) {
  if (N < 0 || nnz < 0 || !rowptr || !uptr || !ws || (nnz > 0 && (!col || !erow))) return DL_EINVAL;
  if (ws_bytes < dl_sym_index_workspace_bytes(N, nnz)) return DL_EWORKSPACE;
  if (nnz >= 0x7fffffffLL) return DL_EUNSUPPORTED;       // positions in the primary view are int32
  cudaStream_t st = (cudaStream_t)stream;
  int* pos = (int*)ws;
  void* scan_ws = (char*)ws + dlp::align256((size_t)(nnz + 2) * 4);
  // pos[e] = number of primary entries before e, e = 0 .. nnz (an exclusive scan of the orientation flags)
  int rc = dlp::scan<false, int>(PrimaryFlag{(const long long*)rowptr, col, erow, nnz}, dlp::StoreArr<int>{pos}, nnz + 1,
                                 dlp::OpSum<int>(), 0, scan_ws, st);
  if (rc) return rc;
  if (!ucol) {              // call 1: row pointers of the primary view (uptr[N] = number of primary entries)
    k_sym_uptr<<<blocks_for(N + 1), 256, 0, st>>>((const long long*)rowptr, pos, N, (long long*)uptr);
    DL_LAUNCH_CHECK();
    return DL_OK;
  }
  if (!eidx || !status_out || ((lcol == nullptr) != (lmirror == nullptr))) return DL_EINVAL;
  DL_CUDA_TRY(cudaMemsetAsync(status_out, 0, sizeof(int32_t), st));
  unsigned long long* n_diag =
      (unsigned long long*)((char*)ws + dlp::align256((size_t)(nnz + 2) * 4) + dlp::scan_ws_bytes(nnz + 1, 4));
  DL_CUDA_TRY(cudaMemsetAsync(n_diag, 0, sizeof(unsigned long long), st));
  if (nnz > 0) {
    k_sym_fill<<<blocks_for(nnz), 256, 0, st>>>((const long long*)rowptr, col, erow, nnz, pos, ucol, eidx, lcol,
                                                lmirror, status_out, n_diag);
    DL_LAUNCH_CHECK();
    k_sym_check<<<1, 1, 0, st>>>(nnz, pos, n_diag, status_out);
    DL_LAUNCH_CHECK();
  }
  return DL_OK;
}

int dl_edge_attn_fwd_sym(const dl_graph* g_host, const dl_graph* upper_host, const int32_t* eidx, const float* Z,
                         int K, int d, float T, uint8_t* kstar, float* w, float* s, float* hub_ws, float* kw_scratch,
                         float* a_out, dl_stream_t stream) {
  if (!dl_graph_ok(g_host) || !dl_graph_ok(upper_host) || !dl_shape_ok(K, d)) return DL_EINVAL;
  if (g_host->N == 0) return DL_OK;
  if (g_host->row_base != 0 || upper_host->row_base != 0 || upper_host->N != g_host->N) return DL_EINVAL;
  if (!Z || !s || (g_host->nnz > 0 && (!kstar || !w || !eidx || !kw_scratch || !hub_ws))) return DL_EINVAL;
  if (!g_host->erow || !upper_host->erow) return DL_EINVAL;
  if (!(T == T) || T == 0.0f) return DL_EINVAL;
  if (!dl_attn_fl_has(K, d) || g_host->nnz == 0) return DL_EUNSUPPORTED;
  cudaStream_t st = (cudaStream_t)stream;
  const DlGraphDev g = dl_graph_dev(g_host);
  const DlGraphDev gu = dl_graph_dev(upper_host);
  float2* kw = reinterpret_cast<float2*>(kw_scratch);
  if (g_host->flags & DL_F_NO_KEEPA) a_out = nullptr;
  int rc = dl_launch_attn_fl(gu, Z, K, d, T, nullptr, nullptr, nullptr, nullptr, st, kw, a_out);
  if (rc == -1000) return DL_EUNSUPPORTED;
  if (rc) return rc;
  int dev = 0, sms = 0;
  DL_CUDA_TRY(cudaGetDevice(&dev));
  DL_CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  const long long n_chunks = (g.nnz + DL_CH - 1) / DL_CH;
  const long long n_ranges = (n_chunks + DL_RANGE - 1) / DL_RANGE;
  long long grid = (n_ranges + SX_WARPS - 1) / SX_WARPS;
  if (grid > (long long)sms * 8) grid = (long long)sms * 8;
  if (grid < 1) grid = 1;
  if (K <= 8) k_sym_expand<8><<<(int)grid, SX_WARPS * 32, 0, st>>>(g, eidx, kw, K, kstar, w, s, hub_ws);
  else k_sym_expand<32><<<(int)grid, SX_WARPS * 32, 0, st>>>(g, eidx, kw, K, kstar, w, s, hub_ws);
  DL_LAUNCH_CHECK();
  return dl_gather_chain_rowsum(g, K, hub_ws, s, st);
}

}  // extern "C"
