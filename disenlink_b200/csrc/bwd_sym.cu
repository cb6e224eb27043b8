// bwd_sym.cu -- backward pass 2 of the factor attention, evaluating every undirected edge once.
//
// [ref: autograd of model.py:56-75]  Pass 2 adds, for every entry e = (i,j) with routed factor k,
//     dZ[i, kap] += coef_e[kap] * Z[j, kap],   coef_e[kap] = dwsum_e * w_e / T * ((kap == k) - a_e[kap]),
//     dwsum_e = c_ij / s[j,k] + c_ji / s[i,k] - r[i,k] - r[j,k]
// (DESIGN.md).  q, a, w, k are symmetric in (i,j) bit for bit and dwsum is symmetric by its form, so the K
// coefficients of (i,j) and (j,i) are the same numbers: the dots, the exponentials, the softmax and the two
// (s, r) gathers only have to be done for ONE of the two entries.
//
//   phase A  k_bwd_edges_fl<K, d, 2> (bwd_fl.cu) on the upper-triangle view (col >= row): the full
//            evaluation; adds coef * Z[j] to dZ[i] and stores coef [nnz_u, K] (coalesced, 4K bytes per entry).
//            When the symmetric attention left its softmax a [nnz_u, K] in the same buffer (a_valid),
//            k_bwd_edges_fl<K, d, 3> reads a there instead of recomputing the dots, exponentials and softmax,
//            and overwrites it with coef
//   phase B  k_bwd_sym_lower (here) on the strictly-lower view: gathers the row Z[j] and the mirror's K
//            coefficients (one random 4K-byte access) and adds coef * Z[j] to dZ[i] -- ~1/4 of phase A's
//            instructions per entry, no own-row state at all
//
// Row gathers stay at one per entry (dZ[i] needs every neighbour's row); what halves is everything else.
// The same balanced chunk / range decomposition, per-warp cp.async ring, XOR-swizzled staging, per-row register
// accumulators and carry / chain fix-up as bwd_fl.cu; no float atomics on shared results (each row of a view
// has one direct writer per launch, rows cut by a range boundary go through the carries).
#include "dl_dispatch.cuh"
#include "dl_stream.cuh"
#include "dl_fl.cuh"

namespace {

#ifndef SL_RING_N
#define SL_RING_N 3
#endif
#ifndef SL_MAXW
#define SL_MAXW 24
#endif

template <int K_, int d_>
struct SlCfg {
  static constexpr int RING = SL_RING_N;
  static constexpr int K = K_, d = d_, D = K_ * d_;
  static constexpr int LPE = 8, EPS = 32 / LPE, QPC = DL_CH / EPS, C4 = d_ / 4;
  static constexpr int ROWB = D * 4;
  static constexpr int ROWS = ((ROWB + 127) / 128) * 128;
  static constexpr int COEF_OFF = EPS * ROWS;
  static constexpr int STAGE_B = COEF_OFF + 128;            // EPS x 32 bytes of coefficients
  static constexpr int BUDGET = 226 * 1024;
  static constexpr int NW_RAW = BUDGET / (RING * STAGE_B);
  static constexpr int MAXW = (C4 == 8) ? (SL_MAXW < 16 ? SL_MAXW : 16) : SL_MAXW;      // d = 32: 2x the registers
  static constexpr int NW = NW_RAW >= MAXW ? MAXW : (NW_RAW >= 4 ? NW_RAW : 4);
  static constexpr int THREADS = NW * 32;
  static constexpr size_t SMEM = (size_t)NW * RING * STAGE_B;
  __device__ static __forceinline__ int key(int kap) { return (kap / (8 / C4)) & (C4 - 1); }
};

struct LMeta {
  int row, col, mir;
  unsigned vmask, smask;          // warp-uniform: valid entries, row starts per step
};

template <int K_, int d_>
__global__ void __launch_bounds__(SlCfg<K_, d_>::THREADS, 1)
k_bwd_sym_lower(DlGraphDev g, const int* __restrict__ lmirror, const float* __restrict__ Z,
                const float* __restrict__ coef, float* __restrict__ dZ, float* __restrict__ carry) {
  using C = SlCfg<K_, d_>;
  constexpr int K = C::K, d = C::d, D = C::D, LPE = C::LPE, EPS = C::EPS, QPC = C::QPC, C4 = C::C4;
  constexpr int RING = C::RING, ROWS = C::ROWS, STAGE_B = C::STAGE_B;
  constexpr int PIECES = K * C4;
  extern __shared__ __align__(128) unsigned char dl_smem_raw[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const unsigned ring = dl_smem_u32(dl_smem_raw) + (unsigned)warp * RING * STAGE_B;
  const long long gw = (long long)blockIdx.x * C::NW + warp;
  const long long RE = (long long)DL_CH * DL_RANGE;
  const int grp = lane / LPE, kap = lane % LPE;
  const bool factive = (K == LPE) || kap < K;
  const int pk = lane / C4, pc = lane % C4;
  const unsigned pdst = (unsigned)(pk * C4 + (pc ^ C::key(pk))) * 16u;
  const bool pact = lane < PIECES;
  const int pk2 = (lane + 32) / C4;                      // rows of more than 32 pieces (D > 128)
  const unsigned pdst2 = (unsigned)(pk2 * C4 + (pc ^ C::key(pk2))) * 16u;
  const bool pact2 = PIECES > 32 && lane + 32 < PIECES;
  // (idle factor lanes, kap >= K, read factor 0's block: their own would lie beyond the row and, for wide rows,
  // beyond the stage)
  const unsigned myblk = factive ? ((unsigned)(kap * C4 * 16) | ((unsigned)C::key(kap) << 4)) : 0u;

  DlChunkStream cs;
  cs.init(g.nnz, (long long)gridDim.x * C::NW, g.range_shift);

  // unconditional loads from a clamped index; validity is applied in finish_meta (see bwd_fl.cu)
  auto load_meta = [&](long long cc, LMeta& m) {
    const long long e = cc * DL_CH + lane;
    const long long ec = (cc >= 0 && e < g.nnz) ? e : 0;
    m.row = __ldg(g.erow + ec); m.col = __ldg(g.col + ec); m.mir = __ldg(lmirror + ec);
  };
  auto finish_meta = [&](LMeta& m, long long cc) {
    if (!(cc >= 0 && cc * DL_CH + lane < g.nnz)) m.row = -1;
    const int prev1 = __shfl_up_sync(DL_FULL, m.row, 1);
    const bool start = m.row >= 0 && ((lane % EPS) == 0 || prev1 != m.row);
    m.smask = __ballot_sync(DL_FULL, start);
    m.vmask = __ballot_sync(DL_FULL, m.row >= 0);
  };
  auto issue_stage = [&](unsigned st, const LMeta& m, int q) {
    const unsigned vq = (m.vmask >> (q * EPS)) & ((1u << EPS) - 1u);
    if (vq == 0) return;
#pragma unroll
    for (int e = 0; e < EPS; ++e) {
      const long long cc = __shfl_sync(DL_FULL, m.col, q * EPS + e);
      if ((vq >> e) & 1u) {
        if (pact) fl_cp16(st + e * ROWS + pdst, Z + cc * D + lane * 4);
        if (PIECES > 32) {
          if (pact2) fl_cp16(st + e * ROWS + pdst2, Z + cc * D + (lane + 32) * 4);
        }
      }
    }
    // the mirror's K coefficients: lane (e, kap) copies its own
    const long long mi = __shfl_sync(DL_FULL, m.mir, q * EPS + grp);
    if (((vq >> grp) & 1u) && factive) fl_cp4(st + C::COEF_OFF + grp * 32 + kap * 4, coef + mi * K + kap);
  };

  float4 dz[C4];
#pragma unroll
  for (int c = 0; c < C4; ++c) dz[c] = dl_zero4();
  int cur_row = -1;
  bool first_run = true, head_open = false, tail_open = false;
  long long cur_range = -1;
  auto flush = [&](bool at_range_end) {
    if (cur_row >= 0) {
#pragma unroll
      for (int c = 0; c < C4; ++c) {
#pragma unroll
        for (int off = LPE; off < 32; off <<= 1) {
          dz[c].x = __fadd_rn(dz[c].x, __shfl_xor_sync(DL_FULL, dz[c].x, off));
          dz[c].y = __fadd_rn(dz[c].y, __shfl_xor_sync(DL_FULL, dz[c].y, off));
          dz[c].z = __fadd_rn(dz[c].z, __shfl_xor_sync(DL_FULL, dz[c].z, off));
          dz[c].w = __fadd_rn(dz[c].w, __shfl_xor_sync(DL_FULL, dz[c].w, off));
        }
      }
      const bool to_head = first_run && head_open;
      const bool to_tail = !to_head && at_range_end && tail_open;
      if (grp == 0 && factive) {
        if (to_head || to_tail) {
          float* dst = carry + (cur_range * 2 + (to_tail ? 1 : 0)) * D + kap * d;
#pragma unroll
          for (int c = 0; c < C4; ++c) *reinterpret_cast<float4*>(dst + c * 4) = dz[c];
        } else {
          // this warp is the row's only direct writer in this launch (see bwd_fl.cu)
          float* dst = dZ + (g.row_base + cur_row) * D + kap * d;
#pragma unroll
          for (int c = 0; c < C4; ++c) fl_red_add4(dst + c * 4, dz[c]);
        }
      }
      first_run = false;
    }
    cur_row = -1;
#pragma unroll
    for (int c = 0; c < C4; ++c) dz[c] = dl_zero4();
  };

  static_assert(RING - 1 <= QPC / 2, "the next chunk's metadata is completed half a chunk ahead");
  long long c = cs.first(gw);
  LMeta mA, mB;
  load_meta(c, mA);
  finish_meta(mA, c);
#pragma unroll
  for (int pq = 0; pq < RING - 1; ++pq) {
    issue_stage(ring + pq * STAGE_B, mA, pq);
    dl_cp_async_commit();
  }
  int rslot = 0;

  while (c >= 0) {
    const long long cn = cs.next(c);
    load_meta(cn, mB);
    const long long rg = c >> g.range_shift;
    if (rg != cur_range) {
      if (cur_range >= 0) flush(true);
      cur_range = rg;
      first_run = true;
      const long long R0 = rg * RE, R1 = min(R0 + RE, g.nnz);
      head_open = R0 > 0 && __ldg(g.erow + R0 - 1) == __ldg(g.erow + R0);
      tail_open = R1 < g.nnz && __ldg(g.erow + R1) == __ldg(g.erow + R1 - 1);
    }
#pragma unroll 1
    for (int q = 0; q < QPC; ++q) {
      if (q == QPC / 2) finish_meta(mB, cn);
      int islot = rslot + (RING - 1);
      if (islot >= RING) islot -= RING;
      const unsigned ist = ring + islot * STAGE_B;
      if (q < QPC - (RING - 1)) issue_stage(ist, mA, q + (RING - 1));
      else issue_stage(ist, mB, q + (RING - 1) - QPC);
      dl_cp_async_commit();
      dl_cp_async_wait<RING - 1>();
      __syncwarp();
      const unsigned st = ring + rslot * STAGE_B;
      const unsigned vq = (mA.vmask >> (q * EPS)) & ((1u << EPS) - 1u);
      if (vq) {
        const int row_e = __shfl_sync(DL_FULL, mA.row, q * EPS + grp);
        const bool valid = row_e >= 0;
        float4 zj[C4];
#pragma unroll
        for (int cc = 0; cc < C4; ++cc) zj[cc] = fl_lds4((st + grp * ROWS + myblk) ^ (cc << 4));
        float cf = fl_lds1(st + C::COEF_OFF + grp * 32 + kap * 4);
        cf = (valid && factive) ? cf : 0.0f;          // (idle groups / factor lanes read stale bytes)
        unsigned runs = (mA.smask >> (q * EPS)) & ((1u << EPS) - 1u);
        if (!__any_sync(DL_FULL, valid && row_e != cur_row)) {
          if (valid && factive) {
#pragma unroll
            for (int cc = 0; cc < C4; ++cc) dl_fma4(dz[cc], cf, zj[cc]);
          }
          runs = 0;
        }
        while (runs) {
          const int pos = __ffs(runs) - 1;
          runs &= runs - 1;
          const int nxt = runs ? (__ffs(runs) - 1) : EPS;
          const int re = __shfl_sync(DL_FULL, mA.row, q * EPS + pos);
          if (re != cur_row) { flush(false); cur_row = re; }
          if (grp >= pos && grp < nxt && valid && factive) {
#pragma unroll
            for (int cc = 0; cc < C4; ++cc) dl_fma4(dz[cc], cf, zj[cc]);
          }
        }
      }
      __syncwarp();
      rslot = (rslot + 1 == RING) ? 0 : rslot + 1;
    }
    c = cn;
    mA = mB;
  }
  if (cur_range >= 0) flush(true);
  dl_cp_async_wait<0>();
}

template <int K_, int d_>
int launch_lower(const DlGraphDev& g, const int* lmirror, const float* Z, const float* coef, float* dZ, float* carry,
                 cudaStream_t st) {
  using C = SlCfg<K_, d_>;
  int dev = 0, sms = 0;
  DL_CUDA_TRY(cudaGetDevice(&dev));
  DL_CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  DL_CUDA_TRY(cudaFuncSetAttribute(k_bwd_sym_lower<K_, d_>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C::SMEM));
  const long long n_chunks = (g.nnz + DL_CH - 1) / DL_CH;
  const long long n_ranges = (n_chunks + DL_RANGE - 1) / DL_RANGE;
  long long grid = (n_ranges + C::NW - 1) / C::NW;
  if (grid > sms) grid = sms;
  if (grid < 1) grid = 1;
  k_bwd_sym_lower<K_, d_><<<(int)grid, C::THREADS, C::SMEM, st>>>(g, lmirror, Z, coef, dZ, carry);
  DL_LAUNCH_CHECK();
  return DL_OK;
}

}  // namespace

// bwd_fl.cu
bool dl_bwd_edges_fl_has(int K, int d);
int dl_launch_bwd_sym_upper(const DlGraphDev& gu, const float* Z, const float* G, const unsigned char* ku,
                            const float* s, const float* r, const float2* sr, const float* xu, int K, int d, float omb,
                            float T, float* dZ, float* coef_out, bool keep_a, float* scratch, cudaStream_t st);
void dl_pack_sr(const float* s, const float* r, long long n, float* sr_scratch, cudaStream_t st);

extern "C" int dl_factor_bwd_edges_sym_supported(int K, int d) { return dl_bwd_edges_fl_has(K, d) ? 1 : 0; }

extern "C" int dl_factor_bwd_edges_sym(const dl_graph* upper_host, const dl_graph* lower_host, const int32_t* lmirror,
                                       const float* Z, const float* G, const uint8_t* ku, const float* s, const float* r,
                                       float* sr_scratch, int64_t n_nodes, const float* xu, float* coef_scratch, int K,
                                       int d, float one_minus_beta, float T, int a_valid, float* dZ,
                                       float* hub_ws, dl_stream_t stream) {
  if (!dl_graph_ok(upper_host) || !dl_graph_ok(lower_host) || !dl_shape_ok(K, d)) return DL_EINVAL;
  if (upper_host->N != lower_host->N || upper_host->row_base != 0 || lower_host->row_base != 0) return DL_EINVAL;
  if (upper_host->N == 0 || upper_host->nnz == 0) return DL_OK;
  if (!Z || !G || !ku || !s || !r || !sr_scratch || !xu || !coef_scratch || !dZ || !hub_ws || n_nodes <= 0) return DL_EINVAL;
  if (lower_host->nnz > 0 && !lmirror) return DL_EINVAL;
  if (!upper_host->erow || (lower_host->nnz > 0 && !lower_host->erow)) return DL_EINVAL;
  if (!(T == T) || T == 0.0f) return DL_EINVAL;
  if (!dl_bwd_edges_fl_has(K, d)) return DL_EUNSUPPORTED;
  cudaStream_t st = (cudaStream_t)stream;
  const DlGraphDev gu = dl_graph_dev(upper_host);
  const DlGraphDev gl = dl_graph_dev(lower_host);
  dl_pack_sr(s, r, (long long)n_nodes * K, sr_scratch, st);
  DL_LAUNCH_CHECK();
  const bool keep_a = a_valid && !(upper_host->flags & DL_F_NO_KEEPA);
  int rc = dl_launch_bwd_sym_upper(gu, Z, G, ku, s, r,
                                   reinterpret_cast<const float2*>(sr_scratch), xu, K, d, one_minus_beta, T, dZ,
                                   coef_scratch, keep_a, hub_ws, st);
  if (rc == -1000) return DL_EUNSUPPORTED;
  if (rc) return rc;
  if (gl.nnz == 0) return DL_OK;
  rc = -1000;
  if (K == 8 && d == 16) rc = launch_lower<8, 16>(gl, lmirror, Z, coef_scratch, dZ, hub_ws, st);
  else if (K == 8 && d == 8) rc = launch_lower<8, 8>(gl, lmirror, Z, coef_scratch, dZ, hub_ws, st);
  else if (K == 5 && d == 16) rc = launch_lower<5, 16>(gl, lmirror, Z, coef_scratch, dZ, hub_ws, st);
  else if (K == 5 && d == 32) rc = launch_lower<5, 32>(gl, lmirror, Z, coef_scratch, dZ, hub_ws, st);
  else if (K == 3 && d == 32) rc = launch_lower<3, 32>(gl, lmirror, Z, coef_scratch, dZ, hub_ws, st);
  if (rc == -1000) return DL_EUNSUPPORTED;
  if (rc) return rc;
  return dl_gather_chain_add(gl, K, d, hub_ws, dZ, st);
}
