// peer_copy.cu -- the all-gather of the node-partitioned step as one push kernel over NVLink peer memory.
//
// Every rank owns a contiguous slice of each per-node array (Z, s, H, prob, dH, r) and every rank
// needs the whole array before the next kernel.  NCCL's ring all-gather moves 25.6 GB at C5 in
// 33.4 ms (670 GB/s per rank, whatever the algorithm / protocol / channel settings).  With NVSwitch
// every GPU reaches every peer at full NVLink bandwidth, so the owner simply WRITES its slice into
// the same position of every peer's buffer: one kernel, one 16-byte load from local HBM and one
// 16-byte store per peer, no staging, no ring latency.  Peer buffers are mapped with CUDA IPC by the
// host side (disenlink_b200/partition.py); ordering between ranks is the caller's (a barrier after
// the kernel: stores to peer memory are visible to the peer once the writing kernel has completed).
#include <string.h>

#include "dl_common.cuh"

namespace {

constexpr int DL_MAX_PEERS = 15;

struct PeerDst {
  uint4* p[DL_MAX_PEERS];
  int n;
};

__global__ void __launch_bounds__(256)
k_push_slice(const uint4* __restrict__ src, long long n_vec, PeerDst dst) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n_vec; i += stride) {
    const uint4 v = __ldg(src + i);
#pragma unroll 1
    for (int q = 0; q < dst.n; ++q) dst.p[q][i] = v;
  }
}

__global__ void k_push_tail(const unsigned char* __restrict__ src, long long n_bytes, long long offset,
                            PeerDst dst) {
  const long long i = offset + (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n_bytes)
    for (int q = 0; q < dst.n; ++q) reinterpret_cast<unsigned char*>(dst.p[q])[i] = src[i];
}

}  // namespace

extern "C" int dl_push_slice(const void* src, void* const* peer_dst, int n_peers, int64_t n_bytes,
                             dl_stream_t stream) {
  if (n_peers < 0 || n_peers > DL_MAX_PEERS || n_bytes < 0 || (n_bytes > 0 && !src)) return DL_EINVAL;
  if (n_peers == 0 || n_bytes == 0) return DL_OK;
  if (!peer_dst) return DL_EINVAL;
  if (((uintptr_t)src & 15) != 0) return DL_EINVAL;
  PeerDst d;
  d.n = n_peers;
  for (int q = 0; q < n_peers; ++q) {
    if (!peer_dst[q] || ((uintptr_t)peer_dst[q] & 15) != 0) return DL_EINVAL;
    d.p[q] = (uint4*)peer_dst[q];
  }
  cudaStream_t st = (cudaStream_t)stream;
  const long long n_vec = n_bytes / 16;
  if (n_vec > 0) {
    long long grid = (n_vec + 255) / 256;
    if (grid > 148 * 16) grid = 148 * 16;
    k_push_slice<<<(int)grid, 256, 0, st>>>((const uint4*)src, n_vec, d);
    DL_LAUNCH_CHECK();
  }
  if (n_bytes % 16) {
    k_push_tail<<<1, 16, 0, st>>>((const unsigned char*)src, n_bytes, n_vec * 16, d);
    DL_LAUNCH_CHECK();
  }
  return DL_OK;
}

// ---- halo exchange: the owner pushes exactly the rows (or routed slices) a peer reads -----------------
namespace {

struct PushTable {
  dl_push_desc d[DL_MAX_PEERS];
};

// A group of L = 2^lsh lanes (L <= 32, L <= vectors per row) copies one row, 16 bytes per lane and step; a warp
// moves 32 / L rows at a time.  The PEERS are the inner loop: a lane group takes row position t of every peer's list
// in turn, U peers in flight, so that consecutive stores of a warp go to different destinations.  Measured on 4 and 8
// B200 (tools/a2a_bench.py): a warp that streams to ONE peer sustains ~280-380 GB/s per rank, alternating peers
// ~690 GB/s -- the rate of the all-gather-style dl_push_slice and above NCCL's all-to-all (614 GB/s).
// No per-vector index arithmetic beyond a shift (the first version divided a 64-bit vector index for every 16 bytes).
// vsh >= 0: the row is K factor slices of 2^vsh vectors each and only the slices whose bit is set in
// mask[source row] are sent.
__global__ void __launch_bounds__(256)
k_push_rows(const uint4* __restrict__ src, int vpr, int lsh, int vsh /* log2(vpf), -1: no masks */, int n_peers,
            long long most, const __grid_constant__ PushTable tab) {
  const int L = 1 << lsh;
  const int lane = threadIdx.x & 31;
  const int sub = lane & (L - 1);                          // my first vector of the row
  const long long rpw = 32 >> lsh;                         // rows per warp and step
  const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  constexpr int U = 4;
  for (long long t = warp * rpw + (lane >> lsh); t < most; t += nwarps * rpw) {
    for (int q0 = 0; q0 < n_peers; q0 += U) {
      long long sr[U], dr[U];
      unsigned mk[U];
      uint4* dq[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int q = q0 + u;
        sr[u] = -1;
        if (q < n_peers && t < tab.d[q].n) {
          const dl_push_desc& d = tab.d[q];
          sr[u] = d.src_idx ? (long long)__ldg(d.src_idx + t) : t;
          dr[u] = d.dst_idx ? (long long)__ldg(d.dst_idx + t) : t;
          mk[u] = (vsh >= 0 && d.mask) ? __ldg(d.mask + sr[u]) : 0xffffffffu;
          dq[u] = reinterpret_cast<uint4*>(d.dst);
        }
      }
      for (int c = sub; c < vpr; c += L) {
        const int k = vsh >= 0 ? (c >> vsh) : 0;
        uint4 v[U];
        bool on[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
          on[u] = sr[u] >= 0 && ((mk[u] >> k) & 1u);
          if (on[u]) v[u] = __ldg(src + sr[u] * vpr + c);
        }
#pragma unroll
        for (int u = 0; u < U; ++u)
          if (on[u]) dq[u][dr[u] * vpr + c] = v[u];
      }
    }
  }
}

// masks[part][row] |= 1 << kstar[e] for every entry e = (row, col) whose column belongs to part's halo block
__global__ void __launch_bounds__(256)
k_need_masks(DlGraphDev g, const unsigned char* __restrict__ kstar, const int* __restrict__ halo_off, int n_parts,
             unsigned* __restrict__ masks) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  const long long nnz32 = (g.nnz + 31) / 32 * 32;
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < nnz32; e += stride) {
    int key = -1;
    unsigned bit = 0;
    if (e < g.nnz) {
      const int c = __ldg(g.col + e);
      if (c >= g.N) {                                        // a halo column: find its owner's block
        int part = 0;
        while (part + 1 < n_parts && c >= __ldg(halo_off + part + 1)) ++part;
        key = __ldg(g.erow + e) * 16 + part;                 // n_parts <= 16
        bit = 1u << __ldg(kstar + e);
      }
    }
    // consecutive entries of a row are column-sorted, i.e. grouped by owner: OR inside the warp first
    const unsigned same = __match_any_sync(DL_FULL, key);
    const unsigned bits = __reduce_or_sync(same, bit);
    if (key >= 0 && (__ffs(same) - 1) == (int)(threadIdx.x & 31))
      atomicOr(masks + (long long)(key & 15) * g.N + (key >> 4), bits);     // integer: order independent
  }
}

}  // namespace

extern "C" int dl_push_rows(const void* src, int64_t row_bytes, int vec_per_factor, const dl_push_desc* descs_host,
                            int n_peers, dl_stream_t stream) {
  if (n_peers < 0 || n_peers > DL_MAX_PEERS || row_bytes <= 0 || row_bytes % 16 || vec_per_factor < 0) return DL_EINVAL;
  if (n_peers == 0) return DL_OK;
  if (!src || !descs_host || ((uintptr_t)src & 15) != 0) return DL_EINVAL;
  PushTable tab;
  long long most = 0;
  for (int q = 0; q < n_peers; ++q) {
    tab.d[q] = descs_host[q];
    if (tab.d[q].n < 0 || (tab.d[q].n > 0 && (!tab.d[q].dst || ((uintptr_t)tab.d[q].dst & 15) != 0))) return DL_EINVAL;
    if (tab.d[q].n > most) most = tab.d[q].n;
  }
  if (most == 0) return DL_OK;
  const int vpr = (int)(row_bytes / 16);
  int vsh = -1;
  if (vec_per_factor > 0) {
    if (vec_per_factor & (vec_per_factor - 1)) return DL_EINVAL;      // slices of 2^n vectors only
    vsh = 0;
    while ((1 << vsh) < vec_per_factor) ++vsh;
  }
  int lsh = 0;
  while (lsh < 5 && (2 << lsh) <= vpr) ++lsh;              // lanes per row: largest power of two <= min(32, vpr)
  const long long rows_per_block = 8LL * (32 >> lsh);
  long long gx = (most + rows_per_block - 1) / rows_per_block;
  if (gx > 148LL * 8) gx = 148LL * 8;
  if (gx < 1) gx = 1;
  k_push_rows<<<(unsigned)gx, 256, 0, (cudaStream_t)stream>>>((const uint4*)src, vpr, lsh, vsh, n_peers, most, tab);
  DL_LAUNCH_CHECK();
  return DL_OK;
}

extern "C" int dl_need_masks(const dl_graph* g_host, const uint8_t* kstar, const int32_t* halo_off, int n_parts,
                             uint32_t* masks, dl_stream_t stream) {
  if (!dl_graph_ok(g_host) || n_parts < 1 || n_parts > 16 || !halo_off || !masks) return DL_EINVAL;
  if (g_host->N == 0) return DL_OK;
  if (g_host->nnz > 0 && (!kstar || !g_host->erow)) return DL_EINVAL;
  cudaStream_t st = (cudaStream_t)stream;
  DL_CUDA_TRY(cudaMemsetAsync(masks, 0, (size_t)n_parts * (size_t)g_host->N * sizeof(uint32_t), st));
  if (g_host->nnz == 0) return DL_OK;
  const DlGraphDev g = dl_graph_dev(g_host);
  long long grid = (g.nnz + 255) / 256;
  if (grid > 148 * 16) grid = 148 * 16;
  k_need_masks<<<(int)grid, 256, 0, st>>>(g, kstar, halo_off, n_parts, masks);
  DL_LAUNCH_CHECK();
  return DL_OK;
}

// ---- per-entry records of the directed step (kstar, w, dw): the owner of an entry pushes it to the owner of its
// column.  Elements of 1 or 4 bytes, one thread per (element, peer), peers inner so consecutive stores of a warp
// alternate destinations like k_push_rows.
namespace {

template <typename E>
__global__ void __launch_bounds__(256)
k_push_entries(const E* __restrict__ src, int n_peers, long long most, const __grid_constant__ PushTable tab) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < most; t += stride) {
#pragma unroll 1
    for (int q = 0; q < n_peers; ++q) {
      const dl_push_desc& d = tab.d[q];
      if (t >= d.n) continue;
      const long long sr = d.src_idx ? (long long)__ldg(d.src_idx + t) : t;
      const long long dr = d.dst_idx ? (long long)__ldg(d.dst_idx + t) : t;
      reinterpret_cast<E*>(d.dst)[dr] = __ldg(src + sr);
    }
  }
}

}  // namespace

extern "C" int dl_push_entries(const void* src, int elem_bytes, const dl_push_desc* descs_host, int n_peers,
                               dl_stream_t stream) {
  if (n_peers < 0 || n_peers > DL_MAX_PEERS || (elem_bytes != 1 && elem_bytes != 4)) return DL_EINVAL;
  if (n_peers == 0) return DL_OK;
  if (!descs_host) return DL_EINVAL;
  PushTable tab;
  long long most = 0;
  for (int q = 0; q < n_peers; ++q) {
    tab.d[q] = descs_host[q];
    const dl_push_desc& d = tab.d[q];
    if (d.n < 0 || d.mask) return DL_EINVAL;
    if (d.n > 0 && (!d.dst || ((uintptr_t)d.dst & (elem_bytes - 1)) != 0)) return DL_EINVAL;
    if (d.n > most) most = d.n;
  }
  if (most == 0) return DL_OK;
  if (!src || ((uintptr_t)src & (elem_bytes - 1)) != 0) return DL_EINVAL;
  long long grid = (most + 255) / 256;
  if (grid > 148LL * 8) grid = 148LL * 8;
  cudaStream_t st = (cudaStream_t)stream;
  if (elem_bytes == 1)
    k_push_entries<unsigned char><<<(unsigned)grid, 256, 0, st>>>((const unsigned char*)src, n_peers, most, tab);
  else
    k_push_entries<unsigned><<<(unsigned)grid, 256, 0, st>>>((const unsigned*)src, n_peers, most, tab);
  DL_LAUNCH_CHECK();
  return DL_OK;
}

// enable stores from the current device into `peer_device`'s memory (idempotent)
extern "C" int dl_enable_peer_access(int peer_device) {
  int cur = 0, can = 0;
  DL_CUDA_TRY(cudaGetDevice(&cur));
  if (cur == peer_device) return DL_OK;
  DL_CUDA_TRY(cudaDeviceCanAccessPeer(&can, cur, peer_device));
  if (!can) return DL_EINVAL;
  cudaError_t e = cudaDeviceEnablePeerAccess(peer_device, 0);
  if (e == cudaErrorPeerAccessAlreadyEnabled) { cudaGetLastError(); return DL_OK; }
  return (int)e;
}

// Map a peer process's allocation into THIS device's address space.  handle = the 64 bytes of a
// cudaIpcMemHandle_t exported by the owner (torch: tensor.untyped_storage()._share_cuda_()[1]).
// The handle is opened with the caller's current device, so the mapping is a peer mapping from this
// device (opening it with the owner's device index current, as torch's own IPC path does, gives a
// pointer that kernels of another device cannot dereference).
extern "C" int dl_ipc_open(const void* handle, void** base_out) {
  if (!handle || !base_out) return DL_EINVAL;
  cudaIpcMemHandle_t h;
  memcpy(&h, handle, sizeof(h));
  void* p = nullptr;
  cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
  if (e != cudaSuccess) {
    cudaGetLastError();                  // not sticky: leave the context clean for the caller's fallback
    return (int)e;
  }
  *base_out = p;
  return DL_OK;
}

extern "C" int dl_ipc_close(void* base) {
  if (!base) return DL_OK;
  DL_CUDA_TRY(cudaIpcCloseMemHandle(base));
  return DL_OK;
}
