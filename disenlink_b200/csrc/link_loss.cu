// link_loss.cu -- weighted binary cross-entropy over a list of link scores, forward and backward fused.
//
// [ref: main_disentangled.py:195]  loss = sum_m BCE(a_pred[pos_mask], 1) + BCE(a_pred[neg_mask_m], 0)
// with F.binary_cross_entropy's numerics: log terms clamped at -100, and -- through autograd of
// BCE(sigmoid(S)) -- dL/dS = w (p - y) / max(p (1 - p), 1e-12) * (1 - p) p, so a score that
// saturated to exactly 0 or 1 in fp32 gets a zero gradient.  The per-pair weights fold the
// 1/count of the means and the 1/m of the script.
// One pass over (prob, labels, weights): 12 B read + 4 B written per pair; partial sums are
// combined in a fixed order (double accumulators), so the loss is run-to-run deterministic.
#include "dl_common.cuh"

namespace {

constexpr int BCE_THREADS = 256;
constexpr int BCE_MAX_BLOCKS = 148 * 8;
constexpr int BCE_SEG_MAX_SLICES = 64;      // blocks per segment of dl_link_bce_segments

// -w * (y log p + (1 - y) log(1 - p)) of one pair, logs clamped at -100 (torch's BCE)
__device__ __forceinline__ float bce_term(float pr, float y, float wt) {
  const float omp = __fsub_rn(1.0f, pr);
  const float lp = fmaxf(logf(pr), -100.0f), lq = fmaxf(logf(omp), -100.0f);
  const float term = __fadd_rn(__fmul_rn(y, lp), __fmul_rn(__fsub_rn(1.0f, y), lq));
  return __fmul_rn(wt, term);
}

__global__ void __launch_bounds__(BCE_THREADS)
k_link_bce(const float* __restrict__ prob, const float* __restrict__ labels,
           const float* __restrict__ weights, long long P, float* __restrict__ dS,
           double* __restrict__ partial) {
  double acc = 0.0;
  const long long stride = (long long)gridDim.x * BCE_THREADS;
  for (long long p = (long long)blockIdx.x * BCE_THREADS + threadIdx.x; p < P; p += stride) {
    const float pr = __ldg(prob + p), y = __ldg(labels + p);
    const float wt = weights ? __ldg(weights + p) : 1.0f;
    const float omp = __fsub_rn(1.0f, pr);
    acc -= (double)bce_term(pr, y, wt);
    if (dS) {
      const float pq = __fmul_rn(omp, pr);
      const float dprob = __fdiv_rn(__fmul_rn(wt, __fsub_rn(pr, y)), fmaxf(pq, 1e-12f));
      dS[p] = __fmul_rn(dprob, pq);
    }
  }
  __shared__ double red[BCE_THREADS / 32];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(DL_FULL, acc, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
#pragma unroll
    for (int i = 0; i < BCE_THREADS / 32; ++i) t += red[i];
    partial[blockIdx.x] = t;
  }
}

__global__ void __launch_bounds__(32) k_link_bce_final(const double* __restrict__ partial, int n,
                                                      float* __restrict__ loss) {
  double acc = 0.0;
  for (int i = threadIdx.x; i < n; i += 32) acc += partial[i];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(DL_FULL, acc, o);
  if (threadIdx.x == 0) *loss = (float)acc;
}

// Segment r = blockIdx.x, slice blockIdx.y of gridDim.y: a block-stride walk over the segment, partial sums
// in double, reduced in a fixed order into partial[r * slices + slice].
__global__ void __launch_bounds__(BCE_THREADS)
k_link_bce_seg(const float* __restrict__ prob, const float* __restrict__ labels,
               const float* __restrict__ weights, long long P, const long long* __restrict__ seg_ptr,
               double* __restrict__ partial) {
  const long long r = blockIdx.x;
  long long lo = __ldg(seg_ptr + r), hi = __ldg(seg_ptr + r + 1);
  lo = lo < 0 ? 0 : (lo > P ? P : lo);                 // a malformed seg_ptr cannot read outside [0, P)
  hi = hi < lo ? lo : (hi > P ? P : hi);
  double acc = 0.0;
  const long long stride = (long long)gridDim.y * BCE_THREADS;
  for (long long p = lo + (long long)blockIdx.y * BCE_THREADS + threadIdx.x; p < hi; p += stride) {
    const float wt = weights ? __ldg(weights + p) : 1.0f;
    acc -= (double)bce_term(__ldg(prob + p), __ldg(labels + p), wt);
  }
  __shared__ double red[BCE_THREADS / 32];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(DL_FULL, acc, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
#pragma unroll
    for (int i = 0; i < BCE_THREADS / 32; ++i) t += red[i];
    partial[r * gridDim.y + blockIdx.y] = t;
  }
}

// one warp per segment sums its slices in a fixed order
__global__ void __launch_bounds__(BCE_THREADS)
k_link_bce_seg_final(const double* __restrict__ partial, int slices, long long R, float* __restrict__ loss) {
  const long long r = (long long)blockIdx.x * (BCE_THREADS / 32) + (threadIdx.x >> 5);
  if (r >= R) return;                                  // warp-uniform
  double acc = 0.0;
  for (int i = threadIdx.x & 31; i < slices; i += 32) acc += partial[r * slices + i];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(DL_FULL, acc, o);
  if ((threadIdx.x & 31) == 0) loss[r] = (float)acc;
}

int bce_seg_slices(long long R) {
  long long s = BCE_MAX_BLOCKS / (R > 0 ? R : 1);
  return (int)(s < 1 ? 1 : (s > BCE_SEG_MAX_SLICES ? BCE_SEG_MAX_SLICES : s));
}

}  // namespace

extern "C" {

int64_t dl_link_bce_workspace_bytes(void) { return (int64_t)BCE_MAX_BLOCKS * (int64_t)sizeof(double); }

int dl_link_bce(const float* prob, const float* labels, const float* weights, int64_t P, float* dS,
                float* loss, void* ws, int64_t ws_bytes, dl_stream_t stream) {
  if (P < 0 || !loss || (P > 0 && (!prob || !labels))) return DL_EINVAL;
  if (!ws || ws_bytes < dl_link_bce_workspace_bytes()) return DL_EWORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  long long grid = (P + BCE_THREADS * 4 - 1) / (BCE_THREADS * 4);
  if (grid > BCE_MAX_BLOCKS) grid = BCE_MAX_BLOCKS;
  if (grid < 1) grid = 1;
  k_link_bce<<<(int)grid, BCE_THREADS, 0, st>>>(prob, labels, weights, P, dS, (double*)ws);
  DL_LAUNCH_CHECK();
  k_link_bce_final<<<1, 32, 0, st>>>((const double*)ws, (int)grid, loss);
  DL_LAUNCH_CHECK();
  return DL_OK;
}

int64_t dl_link_bce_segments_workspace_bytes(int64_t R) {
  if (R < 1) return 0;
  return R * (int64_t)bce_seg_slices(R) * (int64_t)sizeof(double);
}

int dl_link_bce_segments(const float* prob, const float* labels, const float* weights, int64_t P,
                         const int64_t* seg_ptr, int64_t R, float* loss, void* ws, int64_t ws_bytes,
                         dl_stream_t stream) {
  if (P < 0 || R < 1 || R >= (1LL << 31) || !loss || !seg_ptr || (P > 0 && (!prob || !labels))) return DL_EINVAL;
  if (!ws || ws_bytes < dl_link_bce_segments_workspace_bytes(R)) return DL_EWORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  const int slices = bce_seg_slices(R);
  k_link_bce_seg<<<dim3((unsigned)R, (unsigned)slices), BCE_THREADS, 0, st>>>(prob, labels, weights, P,
                                                                              (const long long*)seg_ptr, (double*)ws);
  DL_LAUNCH_CHECK();
  const long long per = BCE_THREADS / 32;
  k_link_bce_seg_final<<<(unsigned)((R + per - 1) / per), BCE_THREADS, 0, st>>>((const double*)ws, slices, R, loss);
  DL_LAUNCH_CHECK();
  return DL_OK;
}

}  // extern "C"
