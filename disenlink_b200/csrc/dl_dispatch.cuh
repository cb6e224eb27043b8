// dl_dispatch.cuh -- (K, d) -> compile-time lane map.  The listed shapes get the register-resident
// fast kernels; every other shape (any K <= DL_MAX_K, d <= DL_MAX_D, including d % 4 != 0) runs the
// runtime-generic kernels, which implement the same canonical arithmetic.
#pragma once
#include "dl_common.cuh"

// X(K, d): shapes of the reference's tuned configurations (hyperparameters_setting:2-17),
// BASELINE.json's configs (K=8 with D=64/128/512) and a few narrow shapes used by the tests.
#define DL_FOR_EACH_SHAPE(X) \
  X(8, 16)                   \
  X(8, 8)                    \
  X(8, 64)                   \
  X(5, 32)                   \
  X(5, 64)                   \
  X(3, 32)                   \
  X(10, 32)                  \
  X(10, 64)                  \
  X(20, 32)                  \
  X(4, 32)                   \
  X(3, 8)                    \
  X(2, 8)                    \
  X(3, 4)                    \
  X(2, 4)                    \
  X(1, 16)

#define DL_DISPATCH_CASE_(KK, DD) \
  if (K == KK && d == DD) { using M = DlMap<KK, DD>; BODY_MACRO(M) }

// usage:
//   #define BODY_MACRO(M) return launch_xyz<M>(args...);
//   DL_DISPATCH_SHAPES()      // falls through when the shape is not listed
//   #undef BODY_MACRO
#define DL_DISPATCH_SHAPES() DL_FOR_EACH_SHAPE(DL_DISPATCH_CASE_)

static inline int dl_shape_ok(int K, int d) {
  return K >= 1 && K <= DL_MAX_K && d >= 1 && d <= DL_MAX_D;
}

// ---- helpers shared by the runtime-generic kernels ------------------------------------------
// canonical dot of two length-d slices held in global memory, evaluated by a full warp; every
// lane returns the same value.  V = 4 if d % 4 == 0 else 1; chunk c lives on lane c % 32.
__device__ __forceinline__ float dl_generic_dot(const float* __restrict__ x,
                                                const float* __restrict__ y, int d, int lane) {
  const int V = (d & 3) ? 1 : 4;
  const int nv = d / V;
  int P = 1;
  while (P < nv) P <<= 1;
  const int G = (P + 31) / 32;  // groups of 32 chunks (power of two when > 1)
  float gs[DL_MAX_D / 32 + 1];
#pragma unroll 1
  for (int grp = 0; grp < G; ++grp) {
    int c = grp * 32 + lane;
    float part = 0.0f;
    if (c < nv) {
      for (int t = 0; t < V; ++t) part = __fmaf_rn(x[c * V + t], y[c * V + t], part);
    }
    const int width = P < 32 ? P : 32;
    for (int off = 1; off < width; off <<= 1) part = __fadd_rn(part, __shfl_xor_sync(DL_FULL, part, off));
    gs[grp] = part;
  }
  for (int stride = 1; stride < G; stride <<= 1)
    for (int i = 0; i + stride < G; i += 2 * stride) gs[i] = __fadd_rn(gs[i], gs[i + stride]);
  // lanes outside the first P-lane group (P < 32) hold sums of zeros; broadcast lane 0
  return __shfl_sync(DL_FULL, gs[0], 0);
}

// softmax over factors + routing for one (i, j) pair, runtime K, d.  e[] and a[] (size K) are
// filled on every lane; returns kstar.
__device__ __forceinline__ int dl_generic_route(const float* __restrict__ zi,
                                                const float* __restrict__ zj, int K, int d, float T,
                                                int lane, float* e, float* a) {
  float sum = 0.0f;
  for (int k = 0; k < K; ++k) {
    float q = __fdiv_rn(dl_generic_dot(zi + k * d, zj + k * d, d, lane), T);
    e[k] = dl_expf(q);
    sum = (k == 0) ? e[0] : __fadd_rn(sum, e[k]);
  }
  int best = 0;
  float bv = 0.0f;
  for (int k = 0; k < K; ++k) {
    float v = __fdiv_rn(e[k], sum);
    a[k] = v;
    if (k == 0) { bv = v; }
    else if (v > bv || (v != v && bv == bv)) { bv = v; best = k; }
  }
  return best;
}

// Shared launcher of the slice-gather kernel (slice_gather.cu).  mode 0: aggregation forward
// (SRC = Z, OUT = H); mode 1: backward pass 1 (SRC = G, OUT = dZ accumulated, r written, hub rows
// finished by their own kernel).  Returns -1000 when (K, d) has no fast-path instantiation.
int dl_launch_slice_gather(int mode, const DlGraphDev& g, long long n_items, const float* Z,
                           const float* SRC, const unsigned char* kstar, const float* w,
                           const float* s, int K, int d, float beta, float omb, float* OUT, float* r,
                           float* hub_ws, cudaStream_t st);

// Streaming attention (attn_stream.cu): routing + row sums.  Returns -1000 when (K, d) has no
// streaming instantiation.
int dl_launch_attn_stream(const DlGraphDev& g, const int* erow, const float* Z, int K, int d, float T,
                          unsigned char* kstar, float* w, float* s, float* hub_ws, cudaStream_t st);

// Streaming slice gather with per-row register accumulators (gather_stream.cu).
// mode 0: aggregation forward (SRC = Z, OUT = H); mode 1: backward pass 1 (SRC = G, OUT = dZ
// accumulated, r written); mode 2: routed row sums (OUT = s).  Returns -1000 when (K, d) has no
// streaming instantiation or the graph has no COO row array.
size_t dl_gather_stream_scratch_floats(long long nnz, int mode, int K, int d);
int dl_launch_gather_stream(int mode, const DlGraphDev& g, const float* Z, const float* SRC,
                            const unsigned char* kstar, const float* w, const float* s, int K, int d,
                            float beta, float omb, float* OUT, float* r, float* scratch,
                            cudaStream_t st, float* xout = nullptr, const int* xidx = nullptr,
                            unsigned char* ku_out = nullptr);
// whether the streaming pass 1 of shape (K, d) leaves the per-entry dots in xout (needs d/4 a power of two)
bool dl_gather_stream_has_x(int K, int d);
int dl_gather_chain_add(const DlGraphDev& g, int K, int d, float* scratch, float* OUT, cudaStream_t st);

// Streaming backward pass 2, fused single kernel (bwd_stream.cu).  Returns -1000 when (K, d) has no streaming
// instantiation.
int dl_launch_bwd_edges_stream(const DlGraphDev& g, const float* Z, const float* G,
                               const unsigned char* kstar, const float* s, const float* r, int K, int d,
                               float omb, float T, float* dZ, float* scratch, cudaStream_t st);

// Streaming decoder backward (pair_stream.cu).  Returns -1000 when (K, d) has no instantiation.
int dl_gather_chain_pair(const DlGraphDev& g, int K, int d, float* scratch, float* dZ, float* dH,
                         cudaStream_t st);
int dl_launch_pair_bwd_stream(const DlGraphDev& g, const int* inc_pair, const float* Z, const float* H,
                              const float* dS, int K, int d, float T, float* dZ, float* dH, float* scratch,
                              cudaStream_t st);

// Factor-per-lane backward pass 2 (bwd_fl.cu).  Returns -1000 when (K, d) has no instantiation.
int dl_launch_bwd_edges_fl(const DlGraphDev& g, const float* Z, const float* G, const unsigned char* kstar,
                           const float* s, const float* r, const float* sj, float* sr_scratch, long long n_nodes,
                           const float* x, int K, int d, float omb, float T, float* dZ, float* scratch,
                           cudaStream_t st);

// Factor-per-lane attention + row sums (attn_fl.cu).  Returns -1000 when (K, d) has no instantiation.
int dl_gather_chain_rowsum(const DlGraphDev& g, int K, float* scratch, float* s_out, cudaStream_t st);
int dl_launch_attn_fl(const DlGraphDev& g, const float* Z, int K, int d, float T, unsigned char* kstar,
                      float* w, float* s, float* scratch, cudaStream_t st, float2* kw_out = nullptr,
                      float* a_out = nullptr);
bool dl_attn_fl_has(int K, int d);
