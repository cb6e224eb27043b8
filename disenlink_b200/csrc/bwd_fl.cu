// bwd_fl.cu -- backward pass 2 of the factor attention, "factor per lane" streaming kernel.
//
// [ref: autograd of model.py:56-75]  same math and same chunk / range / carry decomposition as
// bwd_stream.cu; what changes is the lane mapping.  bwd_stream.cu spreads ONE row over the 32
// lanes (lane = one float4 chunk) and pays for it in shuffles: every dot needs a reduce-scatter
// and every per-entry scalar is broadcast.  ncu showed that kernel issue-bound at ~150 warp
// instructions per entry with the FMA work a small minority.  Here a step handles EPS = 32/LPE
// entries at once: lane (e, kap) owns factor kap of entry e and holds the whole d-float slice in
// registers, so
//   * the K dots <Z[i,kap], Z[j,kap]> are lane-local FMA chains (same canonical order: float4
//     chunk chains + balanced tree, so exp / softmax reproduce the forward's bits),
//   * per-entry scalars (row, kstar, s[j,k], r[j,k]) are fetched by ONE shuffle per step instead
//     of one per entry,
//   * the own row (Z[i], G[i], s[i,:], r[i,:]) stays in registers while a lane group keeps seeing
//     the same row and is re-read from the staged copy only when it changes,
//   * the row accumulator is per lane group; groups are summed (fixed xor order) when the row ends.
// Staging is the same per-warp cp.async ring; rows are stored with an XOR swizzle of the 16-byte
// pieces so that the factor-strided 128-bit shared loads are bank-conflict free.
//
// Instantiated for K <= 8, d in {4, 8, 16} (the headline K=8, d=16 shape class); other shapes use
// bwd_stream.cu.
#include "dl_dispatch.cuh"
#include "dl_stream.cuh"
#include "dl_fl.cuh"

// -DDL_DEBUG_SINGLE_WRITER: every direct row update claims the row in a per-launch counter array; the
// launcher returns DL_EINTERNAL if any row was claimed twice.  The fire-and-forget reduction below is
// only schedule-independent because each row has ONE direct writer per launch (rows cut by a range
// boundary go through the carries); this build asserts it (tests/test_gpu_parity.py runs it when the
// variant library tools/build_variant.sh produced is present).
#ifdef DL_DEBUG_SINGLE_WRITER
__device__ unsigned int* dl_dbg_claims = nullptr;
__device__ unsigned int dl_dbg_violations = 0;
#endif

namespace {

#ifndef FL_RING_N
#define FL_RING_N 2
#endif
#ifndef FL_OWN_N
#define FL_OWN_N 2
#endif
#ifndef FL_MAXW
#define FL_MAXW 16
#endif
#ifndef FL_RING_X
#define FL_RING_X 2
#endif
#ifndef FL_RING_A
#define FL_RING_A 3
#endif
#ifndef FL_MAXW_A
#define FL_MAXW_A 16
#endif
constexpr int FL_OWN = FL_OWN_N;     // staged own-row slots per stage; further rows of a step are read with plain loads

// MODE 0: the routed slice G[j,k*] is staged and <G[j,k*], Z[i,k*]> computed here;
// MODE 1 (HAS_X): the per-entry dots come from pass 1 (x array), no routed slice is staged;
// MODE 2 (symmetric pass 2, phase A, see bwd_sym.cu): MODE 1 on the UPPER-triangle view of the graph
//        (kstar and x in upper-view order, left there by pass 1), and the K coefficients of every entry
//        are stored for the lower-triangle phase
// MODE 3 (KEEPA): MODE 2 with the softmax a[e, :] the symmetric attention stored in coef_out (same layout):
//        a is staged with the neighbour rows and overwritten in place by the coefficients, so neither the
//        own row Z[i] nor the K dots, exponentials and the softmax sum are needed here
template <int K_, int d_, int MODE>
struct FlCfg {
  static constexpr bool HAS_X = MODE >= 1;
  static constexpr bool KEEPA = MODE == 3;
  // stages per warp ring (FL_RING - 1 in flight); KEEPA stages are ~0.8x the size, which leaves room for one
  // more stage in flight
  static constexpr int FL_RING = KEEPA ? FL_RING_A : (HAS_X ? FL_RING_X : FL_RING_N);
  static constexpr int K = K_, d = d_, D = K_ * d_;
  static constexpr int LPE = 8;                       // lanes per entry (factors padded to 8)
  static constexpr int EPS = 32 / LPE;                // entries per step
  static constexpr int QPC = DL_CH / EPS;             // steps per chunk
  static constexpr int C4 = d_ / 4;                   // float4 chunks per factor slice
  static constexpr bool SHAPE_OK = (K_ <= LPE) && (d_ % 4 == 0) && (C4 == 1 || C4 == 2 || C4 == 4 || C4 == 8) &&
                                   (2 * K_ <= 32) && (K_ * C4 <= 64);
  // d = 32: four 32-float slices per lane (own Z, own G, neighbour Z, accumulator) need ~170 registers;
  // KEEPA holds three (own G, neighbour Z, accumulator).  KEEPA at d = 16 fits 128 registers (16 warps)
  // without spilling; at 20 warps (96 registers) ptxas keeps loop-invariant values in local memory and
  // reloads them every step, which measured 2.2x slower at mid (DESIGN 4.2)
  static constexpr int MAXW_X = (C4 == 8) ? (FL_MAXW < 12 ? FL_MAXW : 12) : FL_MAXW;
  static constexpr int MAXW_A = (C4 == 8) ? (FL_MAXW_A < 12 ? FL_MAXW_A : 12) : FL_MAXW_A;
  static constexpr int MAXW = KEEPA ? MAXW_A : MAXW_X;
  static constexpr int ROWB = D * 4;
  static constexpr int ROWS = ((ROWB + 127) / 128) * 128;    // staged row stride (128-byte aligned)
  static constexpr int SLB = 128;                             // routed slice slot (d*4 <= 64 used)
  static constexpr int SRB = 128;                             // s[i,:], r[i,:] slot
  // own-row slot: [Z[i]] G[i] (s, r)[i]
  static constexpr int OWN_G = KEEPA ? 0 : ROWS;
  static constexpr int OWN_SR = OWN_G + ROWS;
  static constexpr int OWN_B = OWN_SR + SRB;
  static constexpr int NB_OFF = 0;
  static constexpr int SL_OFF = EPS * ROWS;
  static constexpr int A_OFF = SL_OFF + (HAS_X ? 0 : EPS * SLB);   // KEEPA: a of the step's entries, EPS x 32 bytes
  static constexpr int OWN_OFF = A_OFF + (KEEPA ? EPS * 32 : 0);
  static constexpr int STAGE_B = OWN_OFF + FL_OWN * OWN_B;
  static constexpr int BUDGET = 226 * 1024;
  static constexpr int NW_RAW = BUDGET / (FL_RING * STAGE_B);
  static constexpr bool OK = SHAPE_OK && NW_RAW >= 4;
  static constexpr int NW = NW_RAW >= MAXW ? MAXW : (NW_RAW >= 4 ? NW_RAW : 4);
  static constexpr int THREADS = NW * 32;
  static constexpr size_t SMEM = (size_t)NW * FL_RING * STAGE_B;
  // swizzle key of factor kap: lanes kap, kap' of one 8-lane phase hit the same banks when
  // kap*C4 == kap'*C4 (mod 8); xor-ing the chunk index with kap / (8/C4) separates them
  __device__ static __forceinline__ int key(int kap) { return (kap / (8 / C4)) & (C4 - 1); }
};

struct FMeta {
  int row, col;
  int info;            // kstar << 3 | need << 2 | rank: own-row slot of the entry inside its step, and
                       // whether the lane group that will process it currently holds another row
  float sj, rj, xv;
  unsigned vmask, smask, nmask;   // warp-uniform: valid entries, row starts per step, need flags
};

template <class C>
__device__ __forceinline__ float fl_dot(const float4 (&a)[C::C4], const float4 (&b)[C::C4]) {
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

template <int K_, int d_, int MODE>
__global__ void __launch_bounds__(FlCfg<K_, d_, MODE>::THREADS, 1)
k_bwd_edges_fl(DlGraphDev g, const float* __restrict__ Z, const float* __restrict__ G,
               const unsigned char* __restrict__ kstar, const float* __restrict__ s,
               const float* __restrict__ r, const float* __restrict__ sj, const float2* __restrict__ sr,
               const float* __restrict__ xc, float omb, float T, float* __restrict__ dZ,
               float* __restrict__ carry, float* __restrict__ coef_out) {
  using C = FlCfg<K_, d_, MODE>;
  constexpr bool HAS_X = C::HAS_X;
  constexpr int K = C::K, d = C::d, D = C::D, LPE = C::LPE, EPS = C::EPS, QPC = C::QPC, C4 = C::C4;
  constexpr int FL_RING = C::FL_RING;
  constexpr int ROWS = C::ROWS, STAGE_B = C::STAGE_B, OWN_B = C::OWN_B;
  constexpr int PIECES = K * C4;                       // 16-byte pieces per row (<= 32)
  extern __shared__ __align__(128) unsigned char dl_smem_raw[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const unsigned ring = dl_smem_u32(dl_smem_raw) + (unsigned)warp * FL_RING * STAGE_B;
  const long long gw = (long long)blockIdx.x * C::NW + warp;
  const long long RE = (long long)DL_CH * DL_RANGE;

  const int grp = lane / LPE, kap = lane % LPE, gbase = lane & ~(LPE - 1);
  const bool factive = (K == LPE) || kap < K;
  const bool unit_T = (T == 1.0f);
  // staging: lane t copies piece t of a row to its swizzled slot
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
  // compute: my factor's block inside a staged row; chunk c sits at block ^ (c << 4)
  // (idle factor lanes, kap >= K, read factor 0's block: their own would lie beyond the row and, for wide rows,
  // beyond the stage)
  const unsigned myblk = factive ? ((unsigned)(kap * C4 * 16) | ((unsigned)C::key(kap) << 4)) : 0u;

  DlChunkStream cs;
  cs.init(g.nnz, (long long)gridDim.x * C::NW, g.range_shift);

  // Unconditional loads from a clamped index: a select between a default and the loaded value right
  // here would make the warp wait for the loads at once (ncu: the FSEL / spill store after these loads
  // held 14 % of all stall samples); validity is applied in finish_meta, half a chunk later.
  const float* sjp = sj ? sj : reinterpret_cast<const float*>(g.erow);
  auto load_meta = [&](long long cc, FMeta& m) {
    const long long e = cc * DL_CH + lane;
    const long long ec = (cc >= 0 && e < g.nnz) ? e : 0;
    m.row = __ldg(g.erow + ec); m.col = __ldg(g.col + ec); m.info = __ldg(kstar + ec);
    m.sj = __ldg(sjp + ec);                  // s[col, kstar] as the forward saw it: no gather needed
    if (HAS_X) m.xv = __ldg(xc + ec);        // <G[col,kstar], Z[row,kstar]> as pass 1 computed it
    m.rj = 0.0f;
  };
  // second half of a chunk's metadata, once row / col / kstar have arrived: the s[j,k], r[j,k]
  // gathers and the own-row bookkeeping (prow = per-lane rows of the previous chunk of this warp)
  auto finish_meta = [&](FMeta& m, long long cc, int prow) {
    const int ks = m.info;
    if (!(cc >= 0 && cc * DL_CH + lane < g.nnz)) { m.row = -1; m.sj = 1.0f; }
    if (m.row >= 0) {
      if (sr) {                 // (s, r) interleaved per (node, factor): one 8-byte gather for both
        const float2 v = __ldg(sr + (long long)m.col * K + ks);
        if (!sj) m.sj = v.x;
        m.rj = v.y;
      } else {
        if (!sj) m.sj = fl_ldg_small(s + (long long)m.col * K + ks);
        m.rj = fl_ldg_small(r + (long long)m.col * K + ks);
      }
    }
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
    m.info = (ks << 3) | (need ? 4 : 0) | (rank & 3);
  };
  // cm = the chunk m describes (KEEPA: locates the entries' a)
  auto issue_stage = [&](unsigned st, const FMeta& m, long long cm, int q) {
    const unsigned vq = (m.vmask >> (q * EPS)) & ((1u << EPS) - 1u);
    if (vq == 0) return;
#pragma unroll
    for (int e = 0; e < EPS; ++e) {
      const long long cc = __shfl_sync(DL_FULL, m.col, q * EPS + e);
      if ((vq >> e) & 1u) stage_row(st + C::NB_OFF + e * ROWS, Z + cc * D);
    }
    if (!HAS_X) {   // routed slices G[j, kstar]: lane group e copies the slice of entry e
      const long long cc = __shfl_sync(DL_FULL, m.col, q * EPS + grp);
      const int kk = __shfl_sync(DL_FULL, m.info, q * EPS + grp) >> 3;
      if (((vq >> grp) & 1u) && kap < C4)
        fl_cp16_small(st + C::SL_OFF + grp * C::SLB + kap * 16, G + cc * D + kk * d + kap * 4);
    }
    if (C::KEEPA) {  // a[e, kap]: lane (e, kap) copies its own (EPS consecutive entries: 4 K contiguous floats)
      if (((vq >> grp) & 1u) && factive)
        fl_cp4(st + C::A_OFF + grp * 32 + kap * 4, coef_out + (cm * DL_CH + q * EPS + grp) * K + kap);
    }
    if ((m.nmask >> (q * EPS)) & ((1u << EPS) - 1u)) {
      unsigned starts = (m.smask >> (q * EPS)) & ((1u << EPS) - 1u);
      int o = 0;
      while (starts && o < FL_OWN) {
        const int pos = __ffs(starts) - 1;
        starts &= starts - 1;
        const long long node = g.row_base + __shfl_sync(DL_FULL, m.row, q * EPS + pos);
        const unsigned ow = st + C::OWN_OFF + o * OWN_B;
        if (!C::KEEPA) stage_row(ow, Z + node * D);
        stage_row(ow + C::OWN_G, G + node * D);
        if (lane < K) fl_cp4(ow + C::OWN_SR + lane * 4, s + node * K + lane);
        else if (lane < 2 * K) fl_cp4(ow + C::OWN_SR + lane * 4, r + node * K + (lane - K));
        ++o;
      }
    }
  };

  // own row of the lane group (factor kap) and the per-group row accumulator
  float4 zi[C4], gi[C4], dz[C4];
  float s_own = 1.0f, r_own = 0.0f;
#pragma unroll
  for (int c = 0; c < C4; ++c) zi[c] = gi[c] = dz[c] = dl_zero4();
  int cur_row = -1;
  bool first_run = true, head_open = false, tail_open = false;
  long long cur_range = -1;
  auto flush = [&](bool at_range_end) {
    if (cur_row >= 0) {
      // sum the lane groups in a fixed order
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
          // dZ[i] += row sum.  This warp is the only writer of the row in this kernel (rows cut by a
          // range boundary go through the carries), so a fire-and-forget vector reduction gives the
          // same value as load-add-store in any schedule -- without stalling on the load.  (f32
          // reductions flush subnormals to zero.)
          float* dst = dZ + (g.row_base + cur_row) * D + kap * d;
#ifdef DL_DEBUG_SINGLE_WRITER
          if (kap == 0 && atomicAdd(dl_dbg_claims + cur_row, 1u) != 0u) atomicAdd(&dl_dbg_violations, 1u);
#endif
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

  static_assert(EPS == 4, "info packs the own-row slot in 2 bits");
  static_assert(C::FL_RING - 1 <= QPC / 2, "the next chunk's metadata is completed half a chunk ahead");
  long long c = cs.first(gw);
  FMeta mA, mB;
  load_meta(c, mA);
  finish_meta(mA, c, -1);
#pragma unroll
  for (int pq = 0; pq < FL_RING - 1; ++pq) {
    issue_stage(ring + pq * STAGE_B, mA, c, pq);
    dl_cp_async_commit();
  }
  int rslot = 0;

  while (c >= 0) {
    // the next chunk's ids are requested now, completed (s / r gathers, own-row bookkeeping) half a
    // chunk later and first used by the prefetch at the last step of this chunk
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
      int islot = rslot + (FL_RING - 1);
      if (islot >= FL_RING) islot -= FL_RING;
      const unsigned ist = ring + islot * STAGE_B;
      if (q < QPC - (FL_RING - 1)) issue_stage(ist, mA, c, q + (FL_RING - 1));
      else issue_stage(ist, mB, cn, q + (FL_RING - 1) - QPC);
      dl_cp_async_commit();
      dl_cp_async_wait<FL_RING - 1>();
      __syncwarp();
      const unsigned st = ring + rslot * STAGE_B;
      const unsigned vq = (mA.vmask >> (q * EPS)) & ((1u << EPS) - 1u);
      if (vq) {
        const int src = q * EPS + grp;
        const int row_e = __shfl_sync(DL_FULL, mA.row, src);
        const int info = __shfl_sync(DL_FULL, mA.info, src);
        const int ks = info >> 3;
        const float sjv = __shfl_sync(DL_FULL, mA.sj, src);
        const float rjv = __shfl_sync(DL_FULL, mA.rj, src);
        const int rk = info & 3;
        const bool need = (info & 4) != 0;
        const bool valid = row_e >= 0;
        if (need && factive) {
          if (FL_OWN >= EPS || rk < FL_OWN) {
            const unsigned ow = st + C::OWN_OFF + rk * OWN_B;
#pragma unroll
            for (int cc = 0; cc < C4; ++cc) {
              if (!C::KEEPA) zi[cc] = fl_lds4((ow + myblk) ^ (cc << 4));
              gi[cc] = fl_lds4((ow + C::OWN_G + myblk) ^ (cc << 4));
            }
            s_own = fl_lds1(ow + C::OWN_SR + kap * 4);
            r_own = fl_lds1(ow + C::OWN_SR + (K + kap) * 4);
          } else {
            const long long node = g.row_base + row_e;
#pragma unroll
            for (int cc = 0; cc < C4; ++cc) {
              if (!C::KEEPA) zi[cc] = dl_ldg4(Z + node * D + kap * d + cc * 4);
              gi[cc] = dl_ldg4(G + node * D + kap * d + cc * 4);
            }
            s_own = __ldg(s + node * K + kap);
            r_own = __ldg(r + node * K + kap);
          }
        }
        float4 zj[C4];
#pragma unroll
        for (int cc = 0; cc < C4; ++cc) {
          // (groups without a valid entry and idle factor lanes read stale bytes; they never reach dz)
          zj[cc] = fl_lds4((st + C::NB_OFF + grp * ROWS + myblk) ^ (cc << 4));
        }
        // wv = a[kstar] and a[kap]: KEEPA reads the forward's (IEEE division by the sequential sum) back;
        // otherwise they are recomputed, where the backward only needs a[] to ~1 ulp (kstar is read back,
        // not recomputed), so the 8-lane butterfly and an approximate reciprocal replace the forward's
        // sequential sum and IEEE divisions
        float wv, ev, rsum = 1.0f;                 // a[kap] = ev * rsum (KEEPA: ev = a[kap])
        if (C::KEEPA) {
          ev = fl_lds1(st + C::A_OFF + grp * 32 + kap * 4);
          wv = __shfl_sync(DL_FULL, ev, gbase + ks);
        } else {
          float qv = fl_dot<C>(zi, zj);
          if (!unit_T) qv = __fdiv_rn(qv, T);
          ev = factive ? dl_expf(qv) : 0.0f;
          float sum = ev;
#pragma unroll
          for (int off = 1; off < LPE; off <<= 1) sum = __fadd_rn(sum, __shfl_xor_sync(DL_FULL, sum, off));
          const float eks = __shfl_sync(DL_FULL, ev, gbase + ks);
          rsum = fl_rcp(sum);
          wv = __fmul_rn(eks, rsum);
        }
        const float cij = __fmul_rn(omb, __shfl_sync(DL_FULL, fl_dot<C>(gi, zj), gbase + ks));
        float cji;
        if (HAS_X) {
          cji = __fmul_rn(omb, __shfl_sync(DL_FULL, mA.xv, src));
        } else {
          float4 gje[C4];
#pragma unroll
          for (int cc = 0; cc < C4; ++cc) gje[cc] = fl_lds4(st + C::SL_OFF + grp * C::SLB + cc * 16);
          cji = __fmul_rn(omb, __shfl_sync(DL_FULL, fl_dot<C>(gje, zi), gbase + ks));
        }
        const float siv = __shfl_sync(DL_FULL, s_own, gbase + ks);
        const float riv = __shfl_sync(DL_FULL, r_own, gbase + ks);
        float dws = __fadd_rn(__fmul_rn(cij, fl_rcp(sjv)), __fmul_rn(cji, fl_rcp(siv)));
        dws = __fsub_rn(dws, riv);
        dws = __fsub_rn(dws, rjv);
        float basec = __fmul_rn(dws, wv);
        if (!unit_T) basec = __fdiv_rn(basec, T);
        const float ind = (kap == ks) ? 1.0f : 0.0f;
        float coef = __fmul_rn(basec, __fsub_rn(ind, C::KEEPA ? ev : __fmul_rn(ev, rsum)));
        coef = (valid && factive) ? coef : 0.0f;
        // the coefficients are symmetric in (i, j): the lower-triangle phase reads them back instead of
        // recomputing dots, exponentials and the softmax (32 contiguous bytes per entry at K = 8).  KEEPA:
        // the same element held a[e, kap], staged above, so this overwrites what this lane already read.
        if (MODE >= 2 && valid && factive) coef_out[(c * DL_CH + src) * K + kap] = coef;
        // accumulate: the whole step continues the current row (common), or run by run (entries of
        // a step are consecutive CSR entries)
        unsigned runs = (mA.smask >> (q * EPS)) & ((1u << EPS) - 1u);
        if (!__any_sync(DL_FULL, valid && row_e != cur_row)) {
          if (valid && factive) {
#pragma unroll
            for (int cc = 0; cc < C4; ++cc) dl_fma4(dz[cc], coef, zj[cc]);
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
            for (int cc = 0; cc < C4; ++cc) dl_fma4(dz[cc], coef, zj[cc]);
          }
        }
      }
      __syncwarp();
      rslot = (rslot + 1 == FL_RING) ? 0 : rslot + 1;
    }
    c = cn;
    mA = mB;
  }
  if (cur_range >= 0) flush(true);
  dl_cp_async_wait<0>();
}

template <int K_, int d_, int MODE>
struct FlLaunch {
  static int run(const DlGraphDev& g, const float* Z, const float* G, const unsigned char* kstar,
                 const float* s, const float* r, const float* sj, const float2* sr, const float* x, float omb,
                 float T, float* dZ, float* carry, cudaStream_t st, float* coef_out = nullptr) {
    using C = FlCfg<K_, d_, MODE>;
    int dev = 0, sms = 0;
    DL_CUDA_TRY(cudaGetDevice(&dev));
    DL_CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    DL_CUDA_TRY(cudaFuncSetAttribute(k_bwd_edges_fl<K_, d_, MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     (int)C::SMEM));
    const long long n_chunks = (g.nnz + DL_CH - 1) / DL_CH;
    const long long n_ranges = (n_chunks + DL_RANGE - 1) / DL_RANGE;
    long long grid = (n_ranges + C::NW - 1) / C::NW;
    if (grid > sms) grid = sms;
    if (grid < 1) grid = 1;
#ifdef DL_DEBUG_SINGLE_WRITER
    unsigned int* claims = nullptr;
    const unsigned int zero = 0;
    DL_CUDA_TRY(cudaMalloc(&claims, (size_t)g.N * sizeof(unsigned int)));
    DL_CUDA_TRY(cudaMemsetAsync(claims, 0, (size_t)g.N * sizeof(unsigned int), st));
    DL_CUDA_TRY(cudaMemcpyToSymbolAsync(dl_dbg_claims, &claims, sizeof(claims), 0, cudaMemcpyHostToDevice, st));
    DL_CUDA_TRY(cudaMemcpyToSymbolAsync(dl_dbg_violations, &zero, sizeof(zero), 0, cudaMemcpyHostToDevice, st));
#endif
    k_bwd_edges_fl<K_, d_, MODE><<<(int)grid, C::THREADS, C::SMEM, st>>>(g, Z, G, kstar, s, r, sj, sr, x, omb, T, dZ,
                                                                         carry, coef_out);
    DL_LAUNCH_CHECK();
#ifdef DL_DEBUG_SINGLE_WRITER
    unsigned int bad = 0;
    DL_CUDA_TRY(cudaStreamSynchronize(st));
    DL_CUDA_TRY(cudaMemcpyFromSymbol(&bad, dl_dbg_violations, sizeof(bad)));
    DL_CUDA_TRY(cudaFree(claims));
    if (bad) return DL_EINTERNAL;
#endif
    return DL_OK;
  }
};

}  // namespace

// returns -1000 when (K, d) has no factor-per-lane instantiation; scratch as for bwd_stream.cu
namespace {
// sr[node,k] = (s[node,k], r[node,k]): a streaming pass of 16 bytes per (node, factor) that turns the two
// per-entry 4-byte gathers of pass 2 into one 8-byte gather
__global__ void k_pack_sr(const float* __restrict__ s, const float* __restrict__ r, long long n, float2* __restrict__ sr) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += stride)
    sr[t] = make_float2(__ldg(s + t), __ldg(r + t));
}
}  // namespace

bool dl_bwd_edges_fl_has(int K, int d) {
  return (K == 8 && d == 16) || (K == 8 && d == 8) || (K == 5 && d == 16) || (K == 5 && d == 32) ||
         (K == 3 && d == 32);
}

int dl_launch_bwd_edges_fl(const DlGraphDev& g, const float* Z, const float* G, const unsigned char* kstar,
                           const float* s, const float* r, const float* sj, float* sr_scratch, long long n_nodes,
                           const float* x, int K, int d, float omb, float T, float* dZ, float* scratch,
                           cudaStream_t st) {
  if (!g.erow || g.nnz == 0 || !scratch || !dl_bwd_edges_fl_has(K, d)) return -1000;
  const float2* sr = nullptr;
  if (sr_scratch && n_nodes > 0) {
    k_pack_sr<<<148 * 8, 256, 0, st>>>(s, r, n_nodes * K, reinterpret_cast<float2*>(sr_scratch));
    DL_LAUNCH_CHECK();
    sr = reinterpret_cast<const float2*>(sr_scratch);
  }
  int rc = -1000;
#define FL_CASE(KK, DD)                                                                                             \
  if (K == KK && d == DD)                                                                                           \
    rc = x ? FlLaunch<KK, DD, 1>::run(g, Z, G, kstar, s, r, sj, sr, x, omb, T, dZ, scratch, st)                      \
           : FlLaunch<KK, DD, 0>::run(g, Z, G, kstar, s, r, sj, sr, nullptr, omb, T, dZ, scratch, st);
  FL_CASE(8, 16)
  FL_CASE(8, 8)
  FL_CASE(5, 16)
#undef FL_CASE
  if (rc != DL_OK) return rc;
  return dl_gather_chain_add(g, K, d, scratch, dZ, st);
}

// Symmetric pass 2, phase A: the kernel above on the upper-triangle view gu (entries with col >= row), kstar
// and x in upper-view order (ku, xu); leaves the K coefficients of every upper entry in coef_out [nnz_u, K].
// keep_a: coef_out holds the forward's softmax a [nnz_u, K] of the same entries (MODE 3), else it is recomputed.
// (s, r) must already be packed in sr.  Returns -1000 when (K, d) has no instantiation.
int dl_launch_bwd_sym_upper(const DlGraphDev& gu, const float* Z, const float* G, const unsigned char* ku,
                            const float* s, const float* r, const float2* sr, const float* xu, int K, int d, float omb,
                            float T, float* dZ, float* coef_out, bool keep_a, float* scratch, cudaStream_t st) {
  if (!gu.erow || gu.nnz == 0 || !scratch || !dl_bwd_edges_fl_has(K, d) || !sr || !xu || !ku || !coef_out) return -1000;
  int rc = -1000;
#define FL_CASE(KK, DD)                                                                                   \
  if (K == KK && d == DD)                                                                                 \
    rc = keep_a ? FlLaunch<KK, DD, 3>::run(gu, Z, G, ku, s, r, nullptr, sr, xu, omb, T, dZ, scratch, st, coef_out) \
                : FlLaunch<KK, DD, 2>::run(gu, Z, G, ku, s, r, nullptr, sr, xu, omb, T, dZ, scratch, st, coef_out);
  FL_CASE(8, 16)
  FL_CASE(8, 8)
  FL_CASE(5, 16)
  FL_CASE(5, 32)
  FL_CASE(3, 32)
#undef FL_CASE
  if (rc != DL_OK) return rc;
  return dl_gather_chain_add(gu, K, d, scratch, dZ, st);
}

void dl_pack_sr(const float* s, const float* r, long long n, float* sr_scratch, cudaStream_t st) {
  k_pack_sr<<<148 * 8, 256, 0, st>>>(s, r, n, reinterpret_cast<float2*>(sr_scratch));
}
