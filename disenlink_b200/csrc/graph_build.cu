// graph_build.cu -- integer work: adjacency -> CSR, reverse-edge index, degree buckets, hub work
// items, pair incidence lists, transposed pattern.  All outputs are bit-exact functions of the inputs (no float, no
// order-dependent atomics).
//
// Reference being replaced: main_disentangled.py:137-142 builds a dense [N,N] adj_sym from the
// train edge columns (duplicates collapse, diagonal kept, symmetrised); model.py:62 multiplies it
// into the routing matrix.  Here the same set of non-zeros is produced as a CSR in
// adj_sym.nonzero() order.
//
// The device-wide steps (radix sort of the keys, unique, scans) are the hand-written primitives of
// dl_prims.cuh; no library code is involved.
#include "dl_common.cuh"
#include "dl_prims.cuh"

namespace {

__host__ __device__ inline int dl_bits_for(long long n) {  // bits needed to hold values < n
  int b = 1;
  while ((1LL << b) < n) ++b;
  return b;
}

inline size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

struct CsrWs {
  size_t keys_a, keys_b, marks, cub, total;
  size_t cub_bytes;
};

size_t cub_bytes_for_csr(long long M, long long N) {   // scratch of sort / unique / scan (largest of the three)
  const size_t a = dlp::sort_ws_bytes(M), b = dlp::unique_ws_bytes(M), c = dlp::scan_ws_bytes(N + 1, 8);
  size_t m = a > b ? a : b;
  return m > c ? m : c;
}

CsrWs csr_ws_layout(long long E, long long N) {
  CsrWs w;
  long long M = 2 * E;
  size_t off = 0;
  w.keys_a = off; off += align256((size_t)(M > 0 ? M : 1) * 8);
  w.keys_b = off; off += align256((size_t)(M > 0 ? M : 1) * 8);
  w.marks = off;  off += align256((size_t)(N + 1) * 8);
  w.cub_bytes = align256(cub_bytes_for_csr(M > 0 ? M : 1, N));
  w.cub = off;    off += w.cub_bytes;
  w.total = off;
  return w;
}

__global__ void k_make_keys(const long long* __restrict__ src, const long long* __restrict__ dst,
                            long long E, long long n_rows, long long n_cols, int symmetrize, int bits,
                            unsigned long long* __restrict__ keys, int* __restrict__ status) {
  long long stride = (long long)gridDim.x * blockDim.x;
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < E; e += stride) {
    long long s = src[e], t = dst[e];
    if (s < 0 || t < 0 || s >= n_rows || t >= n_cols) {
      *status = DL_ERANGE;  // benign race: every writer stores the same value
      s = 0; t = 0;
    }
    if (symmetrize) {
      keys[2 * e] = ((unsigned long long)s << bits) | (unsigned long long)t;
      keys[2 * e + 1] = ((unsigned long long)t << bits) | (unsigned long long)s;
    } else {
      keys[e] = ((unsigned long long)s << bits) | (unsigned long long)t;
    }
  }
}

// sorted unique keys -> col, and the END position of every non-empty row into marks[row+1]
// (marks is zero-filled; an inclusive max-scan then yields rowptr, because ends are
// non-decreasing in the row id).
__global__ void k_decode_keys(const unsigned long long* __restrict__ keys,
                              const long long* __restrict__ nnz_p, int bits, int* __restrict__ col,
                              long long* __restrict__ marks) {
  const long long nnz = *nnz_p;
  const unsigned long long mask = (1ULL << bits) - 1ULL;
  long long stride = (long long)gridDim.x * blockDim.x;
  for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < nnz; p += stride) {
    unsigned long long k = keys[p];
    col[p] = (int)(k & mask);
    long long row = (long long)(k >> bits);
    bool last = (p + 1 == nnz) || ((long long)(keys[p + 1] >> bits) != row);
    if (last) marks[row + 1] = p + 1;
  }
}

// ---- dense adjacency -> CSR (small N, drop-in path) ----------------------------------------
__global__ void k_dense_count(const float* __restrict__ adj, long long N, long long* __restrict__ marks) {
  int lane = threadIdx.x & 31;
  long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long r = warp; r < N; r += nwarps) {
    long long cnt = 0;
    for (long long c0 = 0; c0 < N; c0 += 32) {
      long long c = c0 + lane;
      bool nz = (c < N) && (adj[r * N + c] != 0.0f);
      cnt += __popc(__ballot_sync(DL_FULL, nz));
    }
    if (lane == 0) marks[r + 1] = cnt;
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) marks[0] = 0;
}

__global__ void k_dense_fill(const float* __restrict__ adj, long long N,
                             const long long* __restrict__ rowptr, int* __restrict__ col) {
  int lane = threadIdx.x & 31;
  long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long r = warp; r < N; r += nwarps) {
    long long pos = rowptr[r];
    for (long long c0 = 0; c0 < N; c0 += 32) {
      long long c = c0 + lane;
      bool nz = (c < N) && (adj[r * N + c] != 0.0f);
      unsigned m = __ballot_sync(DL_FULL, nz);
      if (nz) col[pos + __popc(m & ((1u << lane) - 1u))] = (int)c;
      pos += __popc(m);
    }
  }
}

// ---- reverse-edge index ---------------------------------------------------------------------
__global__ void k_rev_index(const long long* __restrict__ rowptr, const int* __restrict__ col,
                            long long N, long long nnz, long long* __restrict__ rev,
                            int* __restrict__ status) {
  long long stride = (long long)gridDim.x * blockDim.x;
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < nnz; e += stride) {
    // row of e: last r with rowptr[r] <= e
    long long lo = 0, hi = N;  // invariant rowptr[lo] <= e < rowptr[hi]
    while (hi - lo > 1) {
      long long mid = (lo + hi) >> 1;
      if (rowptr[mid] <= e) lo = mid; else hi = mid;
    }
    const int i = (int)lo;
    const int j = col[e];
    long long a = rowptr[j], b = rowptr[j + 1];
    while (a < b) {
      long long mid = (a + b) >> 1;
      if (col[mid] < i) a = mid + 1; else b = mid;
    }
    if (a < rowptr[j + 1] && col[a] == i) {
      rev[e] = a;
    } else {
      rev[e] = -1;
      *status = DL_EASYM;
    }
  }
}

// ---- degree buckets ---------------------------------------------------------------------------
__global__ void k_degree_keys(const long long* __restrict__ rowptr, long long N,
                              unsigned char* __restrict__ key, int* __restrict__ rowid) {
  long long stride = (long long)gridDim.x * blockDim.x;
  for (long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x; r < N; r += stride) {
    long long deg = rowptr[r + 1] - rowptr[r];
    int cls = deg > 0 ? 64 - __clzll(deg) : 0;  // bit length
    if (cls > 32) cls = 32;
    key[r] = (unsigned char)(32 - cls);
    rowid[r] = (int)r;
  }
}

__global__ void k_bucket_offsets(const unsigned char* __restrict__ sorted_key, long long N,
                                 long long* __restrict__ off) {
  long long stride = (long long)gridDim.x * blockDim.x;
  long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (N == 0) {
    if (tid <= DL_N_BUCKETS) off[tid] = 0;
    return;
  }
  for (long long p = tid; p < N; p += stride) {
    int k = sorted_key[p];
    int kprev = (p == 0) ? -1 : sorted_key[p - 1];
    for (int b = kprev + 1; b <= k; ++b) off[b] = p;
    if (p == N - 1)
      for (int b = k + 1; b <= DL_N_BUCKETS; ++b) off[b] = N;
  }
}

// ---- hub work items -----------------------------------------------------------------------------
// single-CTA exclusive scan of the per-hub-row segment counts (n_hub is at most nnz / DL_SEG)
__global__ void k_hub_seg_scan(const long long* __restrict__ rowptr, const int* __restrict__ perm,
                               long long n_hub, long long* __restrict__ seg_ptr) {
  __shared__ long long part[1024];
  const int t = threadIdx.x, T = blockDim.x;
  long long chunk = (n_hub + T - 1) / T;
  long long a = min((long long)t * chunk, n_hub), b = min(a + chunk, n_hub);
  long long sum = 0;
  for (long long h = a; h < b; ++h) {
    int row = perm[h];
    long long deg = rowptr[row + 1] - rowptr[row];
    sum += (deg + DL_SEG - 1) / DL_SEG;
  }
  part[t] = sum;
  __syncthreads();
  if (t == 0) {
    long long run = 0;
    for (int i = 0; i < T; ++i) { long long v = part[i]; part[i] = run; run += v; }
    seg_ptr[n_hub] = run;
  }
  __syncthreads();
  long long run = part[t];
  for (long long h = a; h < b; ++h) {
    int row = perm[h];
    long long deg = rowptr[row + 1] - rowptr[row];
    seg_ptr[h] = run;
    run += (deg + DL_SEG - 1) / DL_SEG;
  }
}

__global__ void k_hub_item_fill(const long long* __restrict__ seg_ptr, long long n_hub,
                                int* __restrict__ item_hub) {
  // one warp per hub row, lanes stride over its segments
  int lane = threadIdx.x & 31;
  long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long h = warp; h < n_hub; h += nwarps) {
    long long a = seg_ptr[h], b = seg_ptr[h + 1];
    for (long long t = a + lane; t < b; t += 32) item_hub[t] = (int)h;
  }
}

// ---- COO row array ---------------------------------------------------------------------------
__global__ void k_entry_rows(const long long* __restrict__ rowptr, long long N, int* __restrict__ erow) {
  int lane = threadIdx.x & 31;
  long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long r = warp; r < N; r += nwarps)
    for (long long e = rowptr[r] + lane; e < rowptr[r + 1]; e += 32) erow[e] = (int)r;
}

// ---- pair incidence ---------------------------------------------------------------------------
// key = local row of the endpoint if it lies in [row_lo, row_hi), else the sentinel n_local (sorts
// last and is dropped by the decode kernel)
__global__ void k_incidence_keys(const int* __restrict__ u, const int* __restrict__ v, long long P,
                                 long long row_lo, long long row_hi, unsigned* __restrict__ key,
                                 unsigned* __restrict__ val) {
  long long stride = (long long)gridDim.x * blockDim.x;
  const unsigned sentinel = (unsigned)(row_hi - row_lo);
  for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < P; p += stride) {
    long long a = u[p], b = v[p];
    key[2 * p] = (a >= row_lo && a < row_hi) ? (unsigned)(a - row_lo) : sentinel;
    val[2 * p] = (unsigned)(2 * p);
    key[2 * p + 1] = (b >= row_lo && b < row_hi) ? (unsigned)(b - row_lo) : sentinel;
    val[2 * p + 1] = (unsigned)(2 * p + 1);
  }
}

__global__ void k_incidence_decode(const unsigned* __restrict__ skey, const unsigned* __restrict__ sval,
                                   const int* __restrict__ u, const int* __restrict__ v, long long M,
                                   unsigned sentinel, int* __restrict__ other, int* __restrict__ pair,
                                   long long* __restrict__ marks) {
  long long stride = (long long)gridDim.x * blockDim.x;
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < M; t += stride) {
    if (skey[t] >= sentinel) continue;
    unsigned x = sval[t];
    long long p = x >> 1;
    other[t] = (x & 1u) ? u[p] : v[p];
    pair[t] = (int)p;
    unsigned node = skey[t];
    bool last = (t + 1 == M) || (skey[t + 1] != node);
    if (last) marks[(long long)node + 1] = t + 1;
  }
}

// ---- transposed pattern -----------------------------------------------------------------------
// key = column (the node the entry points to), value = CSR entry index; the stable sort keeps the
// in-entries of a node in CSR order (ascending source row)
__global__ void k_transpose_keys(const int* __restrict__ col, long long nnz, unsigned* __restrict__ key,
                                 unsigned* __restrict__ val) {
  long long stride = (long long)gridDim.x * blockDim.x;
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < nnz; e += stride) {
    key[e] = (unsigned)col[e];
    val[e] = (unsigned)e;
  }
}

__global__ void k_transpose_decode(const unsigned* __restrict__ skey, const unsigned* __restrict__ sval,
                                   const int* __restrict__ erow, long long nnz, long long N, int* __restrict__ tcol,
                                   int* __restrict__ tperm, long long* __restrict__ marks) {
  long long stride = (long long)gridDim.x * blockDim.x;
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < nnz; t += stride) {
    const unsigned e = sval[t];
    tperm[t] = (int)e;
    tcol[t] = erow[e];
    const unsigned node = skey[t];
    if (node < N && (t + 1 == nnz || skey[t + 1] != node)) marks[(long long)node + 1] = t + 1;
  }
}

inline int blocks_for(long long n, int threads = 256, int cap = 148 * 32) {
  long long b = (n + threads - 1) / threads;
  if (b < 1) b = 1;
  if (b > cap) b = cap;
  return (int)b;
}

}  // namespace

// ==================================================================================================
extern "C" {

size_t dl_csr_build_workspace_bytes(int64_t E, int64_t N) {
  if (E < 0 || N < 0) return 0;
  return csr_ws_layout(E, N).total;
}

int dl_csr_build(const int64_t* src, const int64_t* dst, int64_t E, int64_t N, int64_t* rowptr,
                 int32_t* col, int64_t* nnz_out, int32_t* status_out, void* ws, size_t ws_bytes,
                 dl_stream_t stream) {
  return dl_csr_build_rect(src, dst, E, N, N, 1, rowptr, col, nnz_out, status_out, ws, ws_bytes, stream);
}

int dl_csr_build_rect(const int64_t* src, const int64_t* dst, int64_t E, int64_t n_rows,
                      int64_t n_cols, int symmetrize, int64_t* rowptr, int32_t* col,
                      int64_t* nnz_out, int32_t* status_out, void* ws, size_t ws_bytes,
                      dl_stream_t stream) {
  const int64_t N = n_rows;
  if (E < 0 || n_rows < 0 || n_cols < 0 || n_rows >= (1LL << 31) || n_cols >= (1LL << 31)) return DL_EINVAL;
  if (symmetrize && n_rows != n_cols) return DL_EINVAL;
  if (!rowptr || !nnz_out || !status_out || !ws) return DL_EINVAL;
  if (E > 0 && (!src || !dst || !col)) return DL_EINVAL;
  if (E >= (1LL << 61)) return DL_EINVAL;
  CsrWs L = csr_ws_layout(E, N);
  if (ws_bytes < L.total) return DL_EWORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  char* base = (char*)ws;
  unsigned long long* ka = (unsigned long long*)(base + L.keys_a);
  unsigned long long* kb = (unsigned long long*)(base + L.keys_b);
  long long* marks = (long long*)(base + L.marks);
  void* cub_ws = base + L.cub;
  size_t cub_bytes = L.cub_bytes;
  const long long M = symmetrize ? 2 * E : E;
  const int bits = dl_bits_for(n_cols > 1 ? n_cols : 2);
  const int row_bits = dl_bits_for(n_rows > 1 ? n_rows : 2);

  DL_CUDA_TRY(cudaMemsetAsync(status_out, 0, sizeof(int32_t), st));
  DL_CUDA_TRY(cudaMemsetAsync(nnz_out, 0, sizeof(int64_t), st));
  DL_CUDA_TRY(cudaMemsetAsync(marks, 0, (size_t)(N + 1) * 8, st));
  if (M > 0) {
    k_make_keys<<<blocks_for(E), 256, 0, st>>>((const long long*)src, (const long long*)dst, E, n_rows,
                                               n_cols, symmetrize, bits, ka, status_out);
    DL_LAUNCH_CHECK();
    int rc = dlp::sort_keys<unsigned long long>(ka, kb, M, 0, bits + row_bits, cub_ws, st);
    if (rc) return rc;
    rc = dlp::unique_sorted<unsigned long long>(kb, ka, (long long*)nnz_out, M, cub_ws, st);
    if (rc) return rc;
    k_decode_keys<<<blocks_for(M), 256, 0, st>>>(ka, (const long long*)nnz_out, bits, col, marks);
    DL_LAUNCH_CHECK();
  }
  (void)cub_bytes;
  return dlp::scan<true, long long>(dlp::LoadArr<long long>{marks}, dlp::StoreArr<long long>{(long long*)rowptr}, N + 1,
                                    dlp::OpMax<long long>(), 0LL, cub_ws, st);
}

int dl_csr_from_dense(const float* adj, int64_t N, int64_t* rowptr, int32_t* col, void* ws,
                      size_t ws_bytes, dl_stream_t stream) {
  if (N < 0 || N >= (1LL << 31) || !rowptr || (N > 0 && !adj)) return DL_EINVAL;
  cudaStream_t st = (cudaStream_t)stream;
  if (!col) {
    // count pass: marks (in ws) -> inclusive sum scan -> rowptr
    const size_t cub_bytes = dlp::scan_ws_bytes(N + 1, 8);
    size_t need = align256((size_t)(N + 1) * 8) + align256(cub_bytes);
    if (!ws || ws_bytes < need) return DL_EWORKSPACE;
    long long* marks = (long long*)ws;
    void* cub_ws = (char*)ws + align256((size_t)(N + 1) * 8);
    DL_CUDA_TRY(cudaMemsetAsync(marks, 0, (size_t)(N + 1) * 8, st));
    if (N > 0) {
      k_dense_count<<<blocks_for(N * 32), 256, 0, st>>>(adj, N, marks);
      DL_LAUNCH_CHECK();
    }
    return dlp::scan<true, long long>(dlp::LoadArr<long long>{marks}, dlp::StoreArr<long long>{(long long*)rowptr},
                                      N + 1, dlp::OpSum<long long>(), 0LL, cub_ws, st);
  }
  if (N > 0) {
    k_dense_fill<<<blocks_for(N * 32), 256, 0, st>>>(adj, N, (const long long*)rowptr, col);
    DL_LAUNCH_CHECK();
  }
  return DL_OK;
}

int dl_entry_rows(const int64_t* rowptr, int64_t N, int64_t nnz, int32_t* erow, dl_stream_t stream) {
  if (N < 0 || nnz < 0 || !rowptr || (nnz > 0 && !erow)) return DL_EINVAL;
  if (N > 0 && nnz > 0) {
    k_entry_rows<<<blocks_for(N * 32), 256, 0, (cudaStream_t)stream>>>((const long long*)rowptr, N, erow);
    DL_LAUNCH_CHECK();
  }
  return DL_OK;
}

int dl_rev_index(const int64_t* rowptr, const int32_t* col, int64_t N, int64_t nnz, int64_t* rev,
                 int32_t* status_out, dl_stream_t stream) {
  if (N < 0 || nnz < 0 || !rowptr || !status_out || (nnz > 0 && (!col || !rev))) return DL_EINVAL;
  cudaStream_t st = (cudaStream_t)stream;
  DL_CUDA_TRY(cudaMemsetAsync(status_out, 0, sizeof(int32_t), st));
  if (nnz > 0) {
    k_rev_index<<<blocks_for(nnz), 256, 0, st>>>((const long long*)rowptr, col, N, nnz,
                                                 (long long*)rev, status_out);
    DL_LAUNCH_CHECK();
  }
  return DL_OK;
}

static size_t bucket_cub_bytes(long long N) { return dlp::sort_ws_bytes(N > 0 ? N : 1); }

size_t dl_degree_buckets_workspace_bytes(int64_t N) {
  if (N < 0) return 0;
  size_t n = (size_t)(N > 0 ? N : 1);
  return align256(n) * 2 + align256(n * 4) + align256(bucket_cub_bytes(N));
}

int dl_degree_buckets(const int64_t* rowptr, int64_t N, int32_t* perm, int64_t* bucket_off,
                      void* ws, size_t ws_bytes, dl_stream_t stream) {
  if (N < 0 || !rowptr || !bucket_off || (N > 0 && !perm) || !ws) return DL_EINVAL;
  if (ws_bytes < dl_degree_buckets_workspace_bytes(N)) return DL_EWORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  size_t n = (size_t)(N > 0 ? N : 1);
  char* base = (char*)ws;
  unsigned char* key_in = (unsigned char*)base;
  unsigned char* key_out = (unsigned char*)(base + align256(n));
  int* rowid = (int*)(base + 2 * align256(n));
  void* cub_ws = base + 2 * align256(n) + align256(n * 4);
  size_t cub_bytes = align256(bucket_cub_bytes(N));
  if (N > 0) {
    k_degree_keys<<<blocks_for(N), 256, 0, st>>>((const long long*)rowptr, N, key_in, rowid);
    DL_LAUNCH_CHECK();
    (void)cub_bytes;
    int rc = dlp::sort_pairs<unsigned char, int>(key_in, key_out, rowid, perm, N, 0, 6, cub_ws, st);
    if (rc) return rc;
  }
  k_bucket_offsets<<<blocks_for(N > 0 ? N : 1), 256, 0, st>>>(key_out, N, (long long*)bucket_off);
  DL_LAUNCH_CHECK();
  return DL_OK;
}

int dl_hub_items(const int64_t* rowptr, const int32_t* perm, int64_t n_hub, int64_t* hub_seg_ptr,
                 int32_t* item_hub, int64_t n_items, dl_stream_t stream) {
  if (n_hub < 0 || !hub_seg_ptr || (n_hub > 0 && (!rowptr || !perm))) return DL_EINVAL;
  cudaStream_t st = (cudaStream_t)stream;
  if (!item_hub) {
    k_hub_seg_scan<<<1, 1024, 0, st>>>((const long long*)rowptr, perm, n_hub, (long long*)hub_seg_ptr);
    DL_LAUNCH_CHECK();
    return DL_OK;
  }
  if (n_items < 0) return DL_EINVAL;
  if (n_hub > 0 && n_items > 0) {
    k_hub_item_fill<<<blocks_for(n_hub * 32), 256, 0, st>>>((const long long*)hub_seg_ptr, n_hub, item_hub);
    DL_LAUNCH_CHECK();
  }
  return DL_OK;
}

static size_t incidence_cub_bytes(long long M, long long N) {
  const size_t a = dlp::sort_ws_bytes(M > 0 ? M : 1), c = dlp::scan_ws_bytes(N + 1, 8);
  return a > c ? a : c;
}

size_t dl_pair_incidence_workspace_bytes(int64_t P, int64_t N) {
  if (P < 0 || N < 0) return 0;
  size_t m = (size_t)(P > 0 ? 2 * P : 1);
  return 4 * align256(m * 4) + align256((size_t)(N + 1) * 8) + align256(incidence_cub_bytes(2 * P, N));
}

int dl_pair_incidence(const int32_t* u, const int32_t* v, int64_t P, int64_t N, int64_t* inc_ptr,
                      int32_t* inc_other, int32_t* inc_pair, void* ws, size_t ws_bytes,
                      dl_stream_t stream) {
  return dl_pair_incidence_range(u, v, P, 0, N, inc_ptr, inc_other, inc_pair, ws, ws_bytes, stream);
}

int dl_pair_incidence_range(const int32_t* u, const int32_t* v, int64_t P, int64_t row_lo,
                            int64_t row_hi, int64_t* inc_ptr, int32_t* inc_other, int32_t* inc_pair,
                            void* ws, size_t ws_bytes, dl_stream_t stream) {
  const int64_t N = row_hi - row_lo;
  if (row_lo < 0 || N < 0 || N >= (1LL << 31) - 1) return DL_EINVAL;
  if (P < 0 || P >= (1LL << 30) || !inc_ptr || !ws) return DL_EINVAL;
  if (P > 0 && (!u || !v || !inc_other || !inc_pair)) return DL_EINVAL;
  if (ws_bytes < dl_pair_incidence_workspace_bytes(P, N)) return DL_EWORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  const long long M = 2 * P;
  size_t m = (size_t)(M > 0 ? M : 1);
  char* base = (char*)ws;
  unsigned* key_in = (unsigned*)base;
  unsigned* key_out = (unsigned*)(base + align256(m * 4));
  unsigned* val_in = (unsigned*)(base + 2 * align256(m * 4));
  unsigned* val_out = (unsigned*)(base + 3 * align256(m * 4));
  long long* marks = (long long*)(base + 4 * align256(m * 4));
  void* cub_ws = base + 4 * align256(m * 4) + align256((size_t)(N + 1) * 8);
  size_t cub_bytes = align256(incidence_cub_bytes(M, N));
  DL_CUDA_TRY(cudaMemsetAsync(marks, 0, (size_t)(N + 1) * 8, st));
  if (M > 0) {
    k_incidence_keys<<<blocks_for(P), 256, 0, st>>>(u, v, P, row_lo, row_hi, key_in, val_in);
    DL_LAUNCH_CHECK();
    const int bits = dl_bits_for(N + 1 > 1 ? N + 1 : 2);
    int rc = dlp::sort_pairs<unsigned, unsigned>(key_in, key_out, val_in, val_out, M, 0, bits, cub_ws, st);
    if (rc) return rc;
    k_incidence_decode<<<blocks_for(M), 256, 0, st>>>(key_out, val_out, u, v, M, (unsigned)N, inc_other,
                                                      inc_pair, marks);
    DL_LAUNCH_CHECK();
  }
  (void)cub_bytes;
  return dlp::scan<true, long long>(dlp::LoadArr<long long>{marks}, dlp::StoreArr<long long>{(long long*)inc_ptr}, N + 1,
                                    dlp::OpMax<long long>(), 0LL, cub_ws, st);
}

static size_t transpose_sort_bytes(long long nnz, long long N) {
  const size_t a = dlp::sort_ws_bytes(nnz > 0 ? nnz : 1), c = dlp::scan_ws_bytes(N + 1, 8);
  return a > c ? a : c;
}

size_t dl_transpose_index_workspace_bytes(int64_t N, int64_t nnz) {
  if (N < 0 || nnz < 0) return 0;
  size_t m = (size_t)(nnz > 0 ? nnz : 1);
  return 4 * align256(m * 4) + align256((size_t)(N + 1) * 8) + align256(transpose_sort_bytes(nnz, N));
}

int dl_transpose_index(const int32_t* col, const int32_t* erow, int64_t N, int64_t nnz, int64_t* trowptr,
                       int32_t* tcol, int32_t* tperm, void* ws, size_t ws_bytes, dl_stream_t stream) {
  if (N < 0 || N >= (1LL << 31) - 1 || nnz < 0 || nnz >= (1LL << 31) - 1) return DL_EINVAL;
  if (!trowptr || !ws || (nnz > 0 && (!col || !erow || !tcol || !tperm))) return DL_EINVAL;
  if (ws_bytes < dl_transpose_index_workspace_bytes(N, nnz)) return DL_EWORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  size_t m = (size_t)(nnz > 0 ? nnz : 1);
  char* base = (char*)ws;
  unsigned* key_in = (unsigned*)base;
  unsigned* key_out = (unsigned*)(base + align256(m * 4));
  unsigned* val_in = (unsigned*)(base + 2 * align256(m * 4));
  unsigned* val_out = (unsigned*)(base + 3 * align256(m * 4));
  long long* marks = (long long*)(base + 4 * align256(m * 4));
  void* sort_ws = base + 4 * align256(m * 4) + align256((size_t)(N + 1) * 8);
  DL_CUDA_TRY(cudaMemsetAsync(marks, 0, (size_t)(N + 1) * 8, st));
  if (nnz > 0) {
    k_transpose_keys<<<blocks_for(nnz), 256, 0, st>>>(col, nnz, key_in, val_in);
    DL_LAUNCH_CHECK();
    const int bits = dl_bits_for(N > 1 ? N : 2);
    int rc = dlp::sort_pairs<unsigned, unsigned>(key_in, key_out, val_in, val_out, nnz, 0, bits, sort_ws, st);
    if (rc) return rc;
    k_transpose_decode<<<blocks_for(nnz), 256, 0, st>>>(key_out, val_out, erow, nnz, N, tcol, tperm, marks);
    DL_LAUNCH_CHECK();
  }
  return dlp::scan<true, long long>(dlp::LoadArr<long long>{marks}, dlp::StoreArr<long long>{(long long*)trowptr},
                                    N + 1, dlp::OpMax<long long>(), 0LL, sort_ws, st);
}

}  // extern "C"
