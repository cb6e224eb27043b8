// eval_metrics.cu -- ROC-AUC of a list of link scores on the device.
//
// [ref: main_disentangled.py:202-204, 217-219]  the script copies a_pred[val_mask == 1] to the host
// every epoch and calls sklearn.metrics.roc_auc_score.  For binary labels that number is the
// Mann-Whitney statistic with ties counted half:
//   2U  = sum over positives i of ( #negatives with score < s_i ) * 2 + ( #negatives with score == s_i )
//   AUC = 2U / (2 n_pos n_neg)
// 2U is an integer, so it is computed exactly (and compared bit-exactly with the oracle); only the
// final division is floating point (double).
//
// Steps: scores -> order-preserving u32 keys (-0.0 == +0.0, like the comparison sklearn makes);
// radix sort of (key, label); exclusive scan of the negative flags; then every positive finds the
// two ends of its tie group (neighbour test, galloping + binary search only inside ties) and adds
// negpre[first] + negpre[last + 1] to a 64-bit integer accumulator (integer atomics: the sum does
// not depend on the order).  The sort and the scan are the hand-written primitives of dl_prims.cuh.
#include "dl_common.cuh"
#include "dl_prims.cuh"

namespace {

inline size_t ev_align256(size_t x) { return (x + 255) & ~(size_t)255; }

struct AucWs {
  size_t key_a, key_b, lab_a, lab_b, negpre, acc, cub, cub_bytes, total;
};

struct NegFlag {                       // scan input: 1 for a negative
  const unsigned char* lab;
  __device__ __forceinline__ unsigned operator()(long long i) const { return lab[i] ? 0u : 1u; }
};

AucWs auc_ws_layout(long long P) {
  AucWs w;
  const size_t n = (size_t)(P > 0 ? P : 1);
  const size_t a = dlp::sort_ws_bytes((long long)n), b = dlp::scan_ws_bytes((long long)n, 4);
  size_t off = 0;
  w.key_a = off; off += ev_align256(n * 4);
  w.key_b = off; off += ev_align256(n * 4);
  w.lab_a = off; off += ev_align256(n);
  w.lab_b = off; off += ev_align256(n);
  w.negpre = off; off += ev_align256(n * 4);
  w.acc = off; off += 256;                               // u64: 2U, n_pos, n_nan
  w.cub_bytes = ev_align256(a > b ? a : b);
  w.cub = off; off += w.cub_bytes;
  w.total = off;
  return w;
}

__global__ void k_auc_keys(const float* __restrict__ score, const float* __restrict__ labels, long long P,
                           unsigned* __restrict__ key, unsigned char* __restrict__ lab,
                           unsigned long long* __restrict__ acc) {
  unsigned long long npos = 0, nnan = 0;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < P; i += stride) {
    const float sc = __fadd_rn(__ldg(score + i), 0.0f);            // -0.0 -> +0.0
    const unsigned b = __float_as_uint(sc);
    key[i] = (b & 0x80000000u) ? ~b : (b | 0x80000000u);           // ascending float order
    const unsigned char l = __ldg(labels + i) != 0.0f;
    lab[i] = l;
    npos += l;
    nnan += (sc != sc);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    npos += __shfl_xor_sync(DL_FULL, npos, o);
    nnan += __shfl_xor_sync(DL_FULL, nnan, o);
  }
  if ((threadIdx.x & 31) == 0) {
    if (npos) atomicAdd(acc + 1, npos);
    if (nnan) atomicAdd(acc + 2, nnan);
  }
}

__global__ void k_auc_ranksum(const unsigned* __restrict__ key, const unsigned char* __restrict__ lab,
                              const unsigned* __restrict__ negpre, long long P,
                              unsigned long long* __restrict__ acc) {
  const unsigned long long total_neg = (unsigned long long)P - acc[1];
  unsigned long long part = 0;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < P; i += stride) {
    if (!lab[i]) continue;
    const unsigned k = key[i];
    long long first = i, last = i;                                 // tie group [first, last]
    if (i > 0 && key[i - 1] == k) {                                // gallop left, then bisect
      long long step = 1, hi = i;                                  // key[hi] == k
      long long lo = hi - step;
      while (lo >= 0 && key[lo] == k) { hi = lo; step <<= 1; lo = hi - step; }
      if (lo < -1) lo = -1;                                        // key[lo] < k (or lo == -1)
      while (hi - lo > 1) {
        const long long mid = lo + (hi - lo) / 2;
        if (key[mid] == k) hi = mid; else lo = mid;
      }
      first = hi;
    }
    if (i + 1 < P && key[i + 1] == k) {                            // gallop right
      long long step = 1, lo = i;                                  // key[lo] == k
      long long hi = lo + step;
      while (hi < P && key[hi] == k) { lo = hi; step <<= 1; hi = lo + step; }
      if (hi > P) hi = P;                                          // key[hi] > k (or hi == P)
      while (hi - lo > 1) {
        const long long mid = lo + (hi - lo) / 2;
        if (key[mid] == k) lo = mid; else hi = mid;
      }
      last = lo;
    }
    const unsigned long long below = negpre[first];
    const unsigned long long upto = (last + 1 < P) ? negpre[last + 1] : total_neg;
    part += below + upto;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(DL_FULL, part, o);
  if ((threadIdx.x & 31) == 0 && part) atomicAdd(acc, part);
}

__global__ void k_auc_final(const unsigned long long* __restrict__ acc, long long P, double* __restrict__ out) {
  const double npos = (double)acc[1], nneg = (double)((unsigned long long)P - acc[1]);
  const double nnan = (double)acc[2];
  double auc = (double)acc[0] / (2.0 * npos * nneg);
  if (npos == 0.0 || nneg == 0.0 || nnan != 0.0) auc = __longlong_as_double(0x7ff8000000000000LL);
  out[0] = auc; out[1] = npos; out[2] = nneg; out[3] = nnan;
  out[4] = (double)acc[0];                                          // 2U (exact below 2^53)
}

// ---- per-segment AUC (dl_roc_auc_segments) ---------------------------------------------------------
// The same statistic on every segment [seg_ptr[r], seg_ptr[r+1]) of one list.  Each element's key carries its
// segment above the 32 score bits, so one stable radix sort orders the list by (segment, score): segment r's
// elements then occupy exactly its own index range, and a tie group -- elements with equal 64-bit keys --
// can never reach into a neighbouring segment even where the scores are equal.  The negative flags are
// scanned once over the whole list; a positive subtracts the prefix at its segment's base.  Counts and 2U are
// per-segment 64-bit integer sums (order-independent atomics), so each row equals dl_roc_auc on the segment
// alone bit for bit.
struct SegAucWs {
  size_t key_a, key_b, lab_a, lab_b, negpre, acc, tmp, total;
};

SegAucWs seg_auc_ws_layout(long long P, long long R) {
  SegAucWs w;
  const size_t n = (size_t)(P > 0 ? P : 1);
  const size_t a = dlp::sort_ws_bytes((long long)n), b = dlp::scan_ws_bytes((long long)n + 1, 4);
  size_t off = 0;
  w.key_a = off; off += ev_align256(n * 8);
  w.key_b = off; off += ev_align256(n * 8);
  w.lab_a = off; off += ev_align256(n);
  w.lab_b = off; off += ev_align256(n);
  w.negpre = off; off += ev_align256((n + 1) * 4);
  w.acc = off; off += ev_align256((size_t)(R > 0 ? R : 1) * 3 * 8);   // u64 [3][R]: 2U, n_pos, n_nan
  w.tmp = off; off += ev_align256(a > b ? a : b);
  w.total = off;
  return w;
}

// segment of element i: the largest r with seg_ptr[r] <= i (empty segments are skipped), clamped to [0, R)
__device__ __forceinline__ int seg_of(const long long* __restrict__ seg_ptr, int R, long long i) {
  int lo = 0, hi = R;
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (__ldg(seg_ptr + mid) <= i) lo = mid; else hi = mid;
  }
  return lo;
}

// acc[seg] += v over the warp (all 32 lanes call it): one atomic when the warp sits in one segment
__device__ __forceinline__ void seg_add(unsigned long long* acc, int seg, unsigned long long v) {
  const int s0 = __shfl_sync(DL_FULL, seg, 0);
  if (__all_sync(DL_FULL, seg == s0)) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(DL_FULL, v, o);
    if ((threadIdx.x & 31) == 0 && v) atomicAdd(acc + s0, v);
  } else if (v) {
    atomicAdd(acc + seg, v);
  }
}

__global__ void k_seg_auc_keys(const float* __restrict__ score, const float* __restrict__ labels, long long P,
                               const long long* __restrict__ seg_ptr, int R,
                               unsigned long long* __restrict__ key, unsigned char* __restrict__ lab,
                               unsigned long long* __restrict__ acc) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i0 = (long long)blockIdx.x * blockDim.x + (threadIdx.x & ~31); i0 < P; i0 += stride) {
    const long long i = i0 + (threadIdx.x & 31);
    const bool valid = i < P;
    const int seg = seg_of(seg_ptr, R, valid ? i : P - 1);
    unsigned long long pos = 0, nan = 0;
    if (valid) {
      const float sc = __fadd_rn(__ldg(score + i), 0.0f);          // -0.0 -> +0.0
      const unsigned b = __float_as_uint(sc);
      const unsigned k = (b & 0x80000000u) ? ~b : (b | 0x80000000u); // ascending float order
      key[i] = ((unsigned long long)seg << 32) | k;
      const unsigned char l = __ldg(labels + i) != 0.0f;
      lab[i] = l;
      pos = l;
      nan = (sc != sc);
    }
    seg_add(acc + R, seg, pos);
    seg_add(acc + 2 * (long long)R, seg, nan);
  }
}

struct NegFlagEnd {                    // scan input over P + 1 items: 1 for a negative, 0 past the end
  const unsigned char* lab;
  long long P;
  __device__ __forceinline__ unsigned operator()(long long i) const { return (i < P && !lab[i]) ? 1u : 0u; }
};

__global__ void k_seg_auc_ranksum(const unsigned long long* __restrict__ key, const unsigned char* __restrict__ lab,
                                  const unsigned* __restrict__ negpre, long long P,
                                  const long long* __restrict__ seg_ptr, unsigned long long* __restrict__ acc) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i0 = (long long)blockIdx.x * blockDim.x + (threadIdx.x & ~31); i0 < P; i0 += stride) {
    const long long i = i0 + (threadIdx.x & 31);
    const unsigned long long k = key[i < P ? i : P - 1];
    const int seg = (int)(k >> 32);
    unsigned long long part = 0;
    if (i < P && lab[i]) {
      long long first = i, last = i;                               // tie group [first, last]: equal 64-bit keys
      if (i > 0 && key[i - 1] == k) {                              // gallop left, then bisect
        long long step = 1, hi = i;
        long long lo = hi - step;
        while (lo >= 0 && key[lo] == k) { hi = lo; step <<= 1; lo = hi - step; }
        if (lo < -1) lo = -1;
        while (hi - lo > 1) {
          const long long mid = lo + (hi - lo) / 2;
          if (key[mid] == k) hi = mid; else lo = mid;
        }
        first = hi;
      }
      if (i + 1 < P && key[i + 1] == k) {                          // gallop right
        long long step = 1, lo = i;
        long long hi = lo + step;
        while (hi < P && key[hi] == k) { lo = hi; step <<= 1; hi = lo + step; }
        if (hi > P) hi = P;
        while (hi - lo > 1) {
          const long long mid = lo + (hi - lo) / 2;
          if (key[mid] == k) lo = mid; else hi = mid;
        }
        last = lo;
      }
      long long base = __ldg(seg_ptr + seg);
      base = base < 0 ? 0 : (base > first ? first : base);
      const unsigned long long nb = negpre[base];
      part = (unsigned long long)(negpre[first] - nb) + (unsigned long long)(negpre[last + 1] - nb);
    }
    seg_add(acc, seg, part);
  }
}

__global__ void k_seg_auc_final(const unsigned long long* __restrict__ acc, const long long* __restrict__ seg_ptr,
                                int R, double* __restrict__ out) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= R) return;
  const long long n = seg_ptr[r + 1] - seg_ptr[r];
  const unsigned long long u2 = acc[r], pos = acc[R + r], nan = acc[2 * (long long)R + r];
  const double npos = (double)pos, nneg = (double)((unsigned long long)n - pos);
  const double nnan = (double)nan;
  double auc = (double)u2 / (2.0 * npos * nneg);
  if (npos == 0.0 || nneg == 0.0 || nnan != 0.0) auc = __longlong_as_double(0x7ff8000000000000LL);
  double* o = out + 5 * (long long)r;
  o[0] = auc; o[1] = npos; o[2] = nneg; o[3] = nnan;
  o[4] = (double)u2;
}

}  // namespace

extern "C" {

int64_t dl_roc_auc_workspace_bytes(int64_t P) {
  if (P < 0) return 0;
  return (int64_t)auc_ws_layout(P).total;
}

int dl_roc_auc(const float* score, const float* labels, int64_t P, double* out, void* ws, int64_t ws_bytes,
               dl_stream_t stream) {
  if (P < 0 || P >= (1LL << 31) || !out || (P > 0 && (!score || !labels))) return DL_EINVAL;
  const AucWs w = auc_ws_layout(P);
  if (!ws || ws_bytes < (int64_t)w.total) return DL_EWORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  unsigned char* base = (unsigned char*)ws;
  unsigned* key_a = (unsigned*)(base + w.key_a);
  unsigned* key_b = (unsigned*)(base + w.key_b);
  unsigned char* lab_a = base + w.lab_a;
  unsigned char* lab_b = base + w.lab_b;
  unsigned* negpre = (unsigned*)(base + w.negpre);
  unsigned long long* acc = (unsigned long long*)(base + w.acc);
  size_t cub_bytes = w.cub_bytes;
  DL_CUDA_TRY(cudaMemsetAsync(acc, 0, 256, st));
  if (P > 0) {
    long long grid = (P + 255) / 256;
    if (grid > 148 * 16) grid = 148 * 16;
    k_auc_keys<<<(int)grid, 256, 0, st>>>(score, labels, P, key_a, lab_a, acc);
    DL_LAUNCH_CHECK();
    (void)cub_bytes;
    int rc = dlp::sort_pairs<unsigned, unsigned char>(key_a, key_b, lab_a, lab_b, P, 0, 32, base + w.cub, st);
    if (rc) return rc;
    rc = dlp::scan<false, unsigned>(NegFlag{lab_b}, dlp::StoreArr<unsigned>{negpre}, P, dlp::OpSum<unsigned>(), 0u,
                                    base + w.cub, st);
    if (rc) return rc;
    k_auc_ranksum<<<(int)grid, 256, 0, st>>>(key_b, lab_b, negpre, P, acc);
    DL_LAUNCH_CHECK();
  }
  k_auc_final<<<1, 1, 0, st>>>(acc, P, out);
  DL_LAUNCH_CHECK();
  return DL_OK;
}

int64_t dl_roc_auc_segments_workspace_bytes(int64_t P, int64_t R) {
  if (P < 0 || R < 1) return 0;
  return (int64_t)seg_auc_ws_layout(P, R).total;
}

int dl_roc_auc_segments(const float* score, const float* labels, int64_t P, const int64_t* seg_ptr, int64_t R,
                        double* out, void* ws, int64_t ws_bytes, dl_stream_t stream) {
  if (P < 0 || P >= (1LL << 31) || R < 1 || R >= (1LL << 31) || !out || !seg_ptr ||
      (P > 0 && (!score || !labels)))
    return DL_EINVAL;
  const SegAucWs w = seg_auc_ws_layout(P, R);
  if (!ws || ws_bytes < (int64_t)w.total) return DL_EWORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  unsigned char* base = (unsigned char*)ws;
  unsigned long long* key_a = (unsigned long long*)(base + w.key_a);
  unsigned long long* key_b = (unsigned long long*)(base + w.key_b);
  unsigned char* lab_a = base + w.lab_a;
  unsigned char* lab_b = base + w.lab_b;
  unsigned* negpre = (unsigned*)(base + w.negpre);
  unsigned long long* acc = (unsigned long long*)(base + w.acc);
  const long long* sp = (const long long*)seg_ptr;
  DL_CUDA_TRY(cudaMemsetAsync(acc, 0, (size_t)R * 3 * 8, st));
  if (P > 0) {
    int seg_bits = 0;                                              // bits of the largest segment id, R - 1
    while ((1LL << seg_bits) < R) ++seg_bits;
    long long grid = (P + 255) / 256;
    if (grid > 148 * 16) grid = 148 * 16;
    k_seg_auc_keys<<<(int)grid, 256, 0, st>>>(score, labels, P, sp, (int)R, key_a, lab_a, acc);
    DL_LAUNCH_CHECK();
    int rc = dlp::sort_pairs<unsigned long long, unsigned char>(key_a, key_b, lab_a, lab_b, P, 0, 32 + seg_bits,
                                                                base + w.tmp, st);
    if (rc) return rc;
    rc = dlp::scan<false, unsigned>(NegFlagEnd{lab_b, P}, dlp::StoreArr<unsigned>{negpre}, P + 1,
                                    dlp::OpSum<unsigned>(), 0u, base + w.tmp, st);
    if (rc) return rc;
    k_seg_auc_ranksum<<<(int)grid, 256, 0, st>>>(key_b, lab_b, negpre, P, sp, acc);
    DL_LAUNCH_CHECK();
  }
  k_seg_auc_final<<<(int)((R + 127) / 128), 128, 0, st>>>(acc, sp, (int)R, out);
  DL_LAUNCH_CHECK();
  return DL_OK;
}

}  // extern "C"
