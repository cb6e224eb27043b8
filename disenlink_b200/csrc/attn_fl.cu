// attn_fl.cu -- per-edge factor attention + hard routing + row sums, "factor per lane" streaming kernel.
//
// [ref: model.py:56-73]  per CSR entry (i,j):  q_k = <Z[i,k], Z[j,k]> / T,  a = softmax_k(q),
// kstar = first argmax_k a (NaN counts as the maximum),  w = a[kstar];  per node
// s[i,k] = sum of w over the entries of row i routed to k  (0 -> 1, model.py:72).
//
// Same decomposition as attn_stream.cu (balanced 32-entry chunks, 64-chunk ranges per warp, per-warp
// cp.async ring) with the lane mapping of bwd_fl.cu: a stage is 4 entries x 8 factor lanes, lane
// (e, kap) holds the whole d-float slice of factor kap, so the K dots are lane-local FMA chains in
// the canonical order (float4 chunk chains + balanced tree: the same bits as every other kernel and
// the oracle), the softmax denominator is the canonical sequential sum over k (K broadcasts per
// stage, not per entry), every lane divides its own e_k once, and the first-maximum search is an
// integer max butterfly over the 8 lanes plus a ballot.  The row sums ride along: lane kap adds w to
// its register when its factor wins, lane groups are summed in a fixed order when the row ends, rows
// cut by a range boundary go through the carry / chain mechanism of gather_stream.cu (mode 2).
// This replaces two launches (routing, row sums) and ~66 warp instructions per entry by one launch
// and ~35.
//
// Instantiated for K <= 8, d in {8, 16, 32} (the shapes of the reference's configs with K <= 8);
// other shapes use attn_stream.cu.
#include "dl_dispatch.cuh"
#include "dl_stream.cuh"
#include "dl_fl.cuh"

namespace {

#ifndef AFL_RING_N
#define AFL_RING_N 2
#endif
#ifndef AFL_OWN_N
#define AFL_OWN_N 2
#endif
#ifndef AFL_MAXW
#define AFL_MAXW 24
#endif
constexpr int AFL_RING = AFL_RING_N;
constexpr int AFL_OWN = AFL_OWN_N;

template <int K_, int d_>
struct AflCfg {
  static constexpr int K = K_, d = d_, D = K_ * d_;
  static constexpr int LPE = 8, EPS = 32 / LPE, QPC = DL_CH / EPS, C4 = d_ / 4;
  static constexpr bool SHAPE_OK = (K_ <= LPE) && (d_ % 4 == 0) && (C4 == 1 || C4 == 2 || C4 == 4 || C4 == 8) &&
                                   (K_ * C4 <= 64);
  static constexpr int MAXW = (C4 == 8) ? (AFL_MAXW < 16 ? AFL_MAXW : 16) : AFL_MAXW;   // d = 32: 2x the registers
  static constexpr int ROWB = D * 4;
  static constexpr int ROWS = ((ROWB + 127) / 128) * 128;
  static constexpr int OWN_OFF = EPS * ROWS;
  static constexpr int STAGE_B = OWN_OFF + AFL_OWN * ROWS;
  static constexpr int BUDGET = 226 * 1024;
  static constexpr int NW_RAW = BUDGET / (AFL_RING * STAGE_B);
  static constexpr bool OK = SHAPE_OK && NW_RAW >= 4;
  static constexpr int NW = NW_RAW >= MAXW ? MAXW : (NW_RAW >= 4 ? NW_RAW : 4);
  static constexpr int THREADS = NW * 32;
  static constexpr size_t SMEM = (size_t)NW * AFL_RING * STAGE_B;
  __device__ static __forceinline__ int key(int kap) { return (kap / (8 / C4)) & (C4 - 1); }
};

struct AMeta {
  int row, col;
  int info;                       // need << 2 | own-row slot of the entry inside its stage
  unsigned vmask, smask, nmask;   // warp-uniform: valid entries, row starts per stage, need flags
};

template <class C>
__device__ __forceinline__ float afl_dot(const float4 (&a)[C::C4], const float4 (&b)[C::C4]) {
  float p[C::C4];
#pragma unroll
  for (int c = 0; c < C::C4; ++c) p[c] = dl_chunk_dot(a[c], b[c]);
  if (C::C4 == 8)
    return __fadd_rn(__fadd_rn(__fadd_rn(p[0], p[1 % C::C4]), __fadd_rn(p[2 % C::C4], p[3 % C::C4])),
                     __fadd_rn(__fadd_rn(p[4 % C::C4], p[5 % C::C4]), __fadd_rn(p[6 % C::C4], p[7 % C::C4])));
  if (C::C4 == 4) return __fadd_rn(__fadd_rn(p[0], p[1]), __fadd_rn(p[2], p[3 % C::C4]));
  if (C::C4 == 2) return __fadd_rn(p[0], p[1 % C::C4]);
  return p[0];
}

template <int K_, int d_>
__global__ void __launch_bounds__(AflCfg<K_, d_>::THREADS, 1)
k_attn_fl(DlGraphDev g, const float* __restrict__ Z, float T, unsigned char* __restrict__ kstar,
          float* __restrict__ w, float* __restrict__ s, float* __restrict__ carry, float2* __restrict__ kw_out,
          float* __restrict__ a_out) {
  // kw_out != nullptr (symmetric attention, attn_sym.cu): g is the UPPER-triangle view of the graph; the
  // routing of entry e goes to kw_out[e] = (w, kstar) as one 8-byte record and no row sums are made here.
  // a_out != nullptr (only with kw_out): the softmax of entry e goes to a_out[e * K + kap] for backward pass 2
  using C = AflCfg<K_, d_>;
  constexpr int K = C::K, d = C::d, D = C::D, LPE = C::LPE, EPS = C::EPS, QPC = C::QPC, C4 = C::C4;
  constexpr int ROWS = C::ROWS, STAGE_B = C::STAGE_B;
  constexpr int PIECES = K * C4;
  extern __shared__ __align__(128) unsigned char dl_smem_raw[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const unsigned ring = dl_smem_u32(dl_smem_raw) + (unsigned)warp * AFL_RING * STAGE_B;
  const long long gw = (long long)blockIdx.x * C::NW + warp;
  const long long RE = (long long)DL_CH * DL_RANGE;

  const int grp = lane / LPE, kap = lane % LPE, gbase = lane & ~(LPE - 1);
  const bool factive = (K == LPE) || kap < K;
  const bool unit_T = (T == 1.0f);
  const int pk = lane / C4, pc = lane % C4;
  const unsigned pdst = (unsigned)(pk * C4 + (pc ^ C::key(pk))) * 16u;
  const bool pact = lane < PIECES;
  // rows of more than 32 pieces (D > 128): lane t also copies piece t + 32
  const int pk2 = (lane + 32) / C4;
  const unsigned pdst2 = (unsigned)(pk2 * C4 + (pc ^ C::key(pk2))) * 16u;
  const bool pact2 = PIECES > 32 && lane + 32 < PIECES;
  auto stage_row = [&](unsigned dst, const float* src) {
    if (pact) fl_cp16(dst + pdst, src + lane * 4);
    if (PIECES > 32) {
      if (pact2) fl_cp16(dst + pdst2, src + (lane + 32) * 4);
    }
  };
  // (idle factor lanes, kap >= K, read factor 0's block: their own would lie beyond the row and, for wide rows,
  // beyond the stage)
  const unsigned myblk = factive ? ((unsigned)(kap * C4 * 16) | ((unsigned)C::key(kap) << 4)) : 0u;

  DlChunkStream cs;
  cs.init(g.nnz, (long long)gridDim.x * C::NW, g.range_shift);

  // unconditional loads from a clamped index (a select against a default right after the load would
  // make the warp wait for it at once); validity is applied in finish_meta, half a chunk later
  auto load_meta = [&](long long cc, AMeta& m) {
    const long long e = cc * DL_CH + lane;
    const long long ec = (cc >= 0 && e < g.nnz) ? e : 0;
    m.row = __ldg(g.erow + ec); m.col = __ldg(g.col + ec);
    m.info = 0;
  };
  auto finish_meta = [&](AMeta& m, long long cc, int prow) {
    if (!(cc >= 0 && cc * DL_CH + lane < g.nnz)) m.row = -1;
    const int up = __shfl_up_sync(DL_FULL, m.row, EPS);
    const int wrap = __shfl_sync(DL_FULL, prow, (lane + 32 - EPS) & 31);
    const int prevE = lane >= EPS ? up : wrap;
    const bool need = m.row >= 0 && m.row != prevE;
    const int prev1 = __shfl_up_sync(DL_FULL, m.row, 1);
    const bool start = m.row >= 0 && ((lane % EPS) == 0 || prev1 != m.row);
    m.smask = __ballot_sync(DL_FULL, start);
    m.nmask = __ballot_sync(DL_FULL, need);
    m.vmask = __ballot_sync(DL_FULL, m.row >= 0);
    const unsigned sbits = ((1u << EPS) - 1u) << ((lane / EPS) * EPS);
    const int rank = __popc(m.smask & sbits & (0xffffffffu >> (31 - lane))) - 1;
    m.info = (need ? 4 : 0) | (rank & 3);
  };
  auto issue_stage = [&](unsigned st, const AMeta& m, int q) {
    const unsigned vq = (m.vmask >> (q * EPS)) & ((1u << EPS) - 1u);
    if (vq == 0) return;
#pragma unroll
    for (int e = 0; e < EPS; ++e) {
      const long long cc = __shfl_sync(DL_FULL, m.col, q * EPS + e);
      if ((vq >> e) & 1u) stage_row(st + e * ROWS, Z + cc * D);
    }
    if ((m.nmask >> (q * EPS)) & ((1u << EPS) - 1u)) {
      unsigned starts = (m.smask >> (q * EPS)) & ((1u << EPS) - 1u);
      int o = 0;
      while (starts && o < AFL_OWN) {
        const int pos = __ffs(starts) - 1;
        starts &= starts - 1;
        const long long node = g.row_base + __shfl_sync(DL_FULL, m.row, q * EPS + pos);
        stage_row(st + C::OWN_OFF + o * ROWS, Z + node * D);
        ++o;
      }
    }
  };

  float4 zi[C4];
#pragma unroll
  for (int c = 0; c < C4; ++c) zi[c] = dl_zero4();
  float acc_s = 0.0f;                       // this lane group's share of s[cur_row, kap]
  int cur_row = -1;
  bool first_run = true, head_open = false, tail_open = false;
  long long cur_range = -1;
  auto flush = [&](bool at_range_end) {
    if (cur_row >= 0) {
      float v = acc_s;
#pragma unroll
      for (int off = LPE; off < 32; off <<= 1) v = __fadd_rn(v, __shfl_xor_sync(DL_FULL, v, off));
      const bool to_head = first_run && head_open;
      const bool to_tail = !to_head && at_range_end && tail_open;
      if (grp == 0 && factive && s != nullptr) {
        if (to_head || to_tail) carry[(cur_range * 2 + (to_tail ? 1 : 0)) * K + kap] = v;
        else {
          const float sv = (v == 0.0f) ? 1.0f : v;
          s[(g.row_base + cur_row) * K + kap] = sv;
          for (int q = 0; q < g.n_peer_out; ++q) g.peer_out[q][(g.row_base + cur_row) * K + kap] = sv;
        }
      }
      first_run = false;
    }
    cur_row = -1;
    acc_s = 0.0f;
  };

  static_assert(EPS == 4, "info packs the own-row slot in 2 bits");
  static_assert(AFL_RING - 1 <= QPC / 2, "the next chunk's metadata is completed half a chunk ahead");
  long long c = cs.first(gw);
  AMeta mA, mB;
  load_meta(c, mA);
  finish_meta(mA, c, -1);
#pragma unroll
  for (int pq = 0; pq < AFL_RING - 1; ++pq) {
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
      if (q == QPC / 2) finish_meta(mB, cn, mA.row);
      int islot = rslot + (AFL_RING - 1);
      if (islot >= AFL_RING) islot -= AFL_RING;
      const unsigned ist = ring + islot * STAGE_B;
      if (q < QPC - (AFL_RING - 1)) issue_stage(ist, mA, q + (AFL_RING - 1));
      else issue_stage(ist, mB, q + (AFL_RING - 1) - QPC);
      dl_cp_async_commit();
      dl_cp_async_wait<AFL_RING - 1>();
      __syncwarp();
      const unsigned st = ring + rslot * STAGE_B;
      const unsigned vq = (mA.vmask >> (q * EPS)) & ((1u << EPS) - 1u);
      if (vq) {
        const int src = q * EPS + grp;
        const int row_e = __shfl_sync(DL_FULL, mA.row, src);
        const int info = __shfl_sync(DL_FULL, mA.info, src);
        const bool valid = row_e >= 0;
        if ((info & 4) && factive) {
          const int rk = info & 3;
          if (AFL_OWN >= EPS || rk < AFL_OWN) {
            const unsigned ow = st + C::OWN_OFF + rk * ROWS;
#pragma unroll
            for (int cc = 0; cc < C4; ++cc) zi[cc] = fl_lds4((ow + myblk) ^ (cc << 4));
          } else {
            const long long node = g.row_base + row_e;
#pragma unroll
            for (int cc = 0; cc < C4; ++cc) zi[cc] = dl_ldg4(Z + node * D + kap * d + cc * 4);
          }
        }
        float4 zj[C4];
#pragma unroll
        for (int cc = 0; cc < C4; ++cc) zj[cc] = fl_lds4((st + grp * ROWS + myblk) ^ (cc << 4));
        float qv = afl_dot<C>(zi, zj);
        if (!unit_T) qv = __fdiv_rn(qv, T);
        const float ev = factive ? dl_expf(qv) : 0.0f;
        // canonical softmax: sequential sum over k, one IEEE division per factor
        float sum = 0.0f;
#pragma unroll
        for (int k = 0; k < K; ++k) {
          const float ek = __shfl_sync(DL_FULL, ev, gbase + k);
          sum = (k == 0) ? ek : __fadd_rn(sum, ek);
        }
        const float a = __fdiv_rn(ev, sum);
        // first maximum over the K factors, NaN counts as the maximum (torch.argmax): a >= 0, so the
        // bit pattern is order preserving; idle lanes hold 0 and sit above every real lane
        unsigned key = (a != a) ? 0xffffffffu : __float_as_uint(a);
        if (!factive) key = 0u;
        unsigned mx = key;                       // 8-lane butterfly (a partial-mask redux is emulated by a loop)
#pragma unroll
        for (int off = 1; off < LPE; off <<= 1) mx = max(mx, __shfl_xor_sync(DL_FULL, mx, off));
        const unsigned hit = __ballot_sync(DL_FULL, key == mx && factive);
        const int ks = __ffs((hit >> gbase) & 0xffu) - 1;
        const float wv = __shfl_sync(DL_FULL, a, gbase + ks);
        if (a_out && valid && factive) a_out[(c * DL_CH + src) * K + kap] = a;   // 4K contiguous bytes per entry
        if (valid && kap == 0) {
          const long long e = c * DL_CH + src;
          if (kw_out) {
            kw_out[e] = make_float2(wv, __int_as_float(ks));
          } else {
            kstar[e] = (unsigned char)ks;
            w[e] = wv;
          }
        }
        const float contrib = (valid && kap == ks) ? wv : 0.0f;
        // row sums: the whole stage continues the current row (common), or run by run
        unsigned runs = (mA.smask >> (q * EPS)) & ((1u << EPS) - 1u);
        if (!__any_sync(DL_FULL, valid && row_e != cur_row)) {
          acc_s = __fadd_rn(acc_s, contrib);
          runs = 0;
        }
        while (runs) {
          const int pos = __ffs(runs) - 1;
          runs &= runs - 1;
          const int nxt = runs ? (__ffs(runs) - 1) : EPS;
          const int re = __shfl_sync(DL_FULL, mA.row, q * EPS + pos);
          if (re != cur_row) { flush(false); cur_row = re; }
          if (grp >= pos && grp < nxt) acc_s = __fadd_rn(acc_s, contrib);
        }
      }
      __syncwarp();
      rslot = (rslot + 1 == AFL_RING) ? 0 : rslot + 1;
    }
    c = cn;
    mA = mB;
  }
  if (cur_range >= 0) flush(true);
  dl_cp_async_wait<0>();
}

template <int K_, int d_>
struct AflLaunch {
  static int run(const DlGraphDev& g, const float* Z, float T, unsigned char* kstar, float* w, float* s,
                 float* carry, float2* kw_out, float* a_out, cudaStream_t st) {
    using C = AflCfg<K_, d_>;
    int dev = 0, sms = 0;
    DL_CUDA_TRY(cudaGetDevice(&dev));
    DL_CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    DL_CUDA_TRY(cudaFuncSetAttribute(k_attn_fl<K_, d_>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     (int)C::SMEM));
    const long long n_chunks = (g.nnz + DL_CH - 1) / DL_CH;
    const long long n_ranges = (n_chunks + DL_RANGE - 1) / DL_RANGE;
    long long grid = (n_ranges + C::NW - 1) / C::NW;
    if (grid > sms) grid = sms;
    if (grid < 1) grid = 1;
    k_attn_fl<K_, d_><<<(int)grid, C::THREADS, C::SMEM, st>>>(g, Z, T, kstar, w, s, carry, kw_out, a_out);
    DL_LAUNCH_CHECK();
    return DL_OK;
  }
};

}  // namespace

// returns -1000 when (K, d) has no factor-per-lane instantiation; scratch: 3 * n_ranges * K floats.
// kw_out != nullptr: packed (w, kstar) records, no row sums (kstar, w, s, scratch may be null); a_out (only
// with kw_out, may be null): the softmax a [nnz, K]
int dl_launch_attn_fl(const DlGraphDev& g, const float* Z, int K, int d, float T, unsigned char* kstar,
                      float* w, float* s, float* scratch, cudaStream_t st, float2* kw_out, float* a_out) {
  if (!g.erow || g.nnz == 0 || (!scratch && !kw_out)) return -1000;
  if (kw_out) s = nullptr;
  else a_out = nullptr;
  int rc = -1000;
#define AFL_CASE(KK, DD) \
  if (K == KK && d == DD) rc = AflLaunch<KK, DD>::run(g, Z, T, kstar, w, s, scratch, kw_out, a_out, st);
  AFL_CASE(8, 16)
  AFL_CASE(8, 8)
  AFL_CASE(5, 16)
  AFL_CASE(5, 32)
  AFL_CASE(3, 32)
  AFL_CASE(4, 32)
  AFL_CASE(8, 32)
#undef AFL_CASE
  if (rc != DL_OK) return rc;
  if (kw_out) return DL_OK;
  return dl_gather_chain_rowsum(g, K, scratch, s, st);
}

bool dl_attn_fl_has(int K, int d) {
  return (K == 8 && (d == 16 || d == 8 || d == 32)) || (K == 5 && (d == 16 || d == 32)) || (K == 3 && d == 32) ||
         (K == 4 && d == 32);
}
