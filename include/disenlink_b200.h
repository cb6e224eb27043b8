/*
 * disenlink_b200.h -- C ABI of libdisenlink_b200.so (hand-written sm_100a CUDA kernels).
 *
 * The reference (sjz5202/DisenLink) has no FFI: its hot path is the Python nn.Module API of
 * model.py called by main_disentangled.py.  This ABI is what a binding for that path calls; the
 * Python side (disenlink_b200/model.py, a drop-in for the reference's model.py) reaches it through
 * ctypes.  For every entry point the reference lines it replaces are cited as
 * [ref: file:line] with paths relative to the reference repository root.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes; no torch / C++ types.
 *   - every pointer is a DEVICE pointer unless the name ends in _host.
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).  Calls only
 *     enqueue work; they never synchronise unless stated.
 *   - every function returns 0 on success, a negative DL_E* code for argument errors, or a
 *     positive cudaError_t value when the CUDA runtime reported one.  Nothing throws.
 *   - re-entrant, no global state; outputs are caller-allocated; nothing is freed across the ABI.
 *   - layouts: Z, H, G, dZ, dH are [N, K, d] fp32 row-major (identical in memory to
 *     torch.cat(h_list, dim=1) of model.py:114); rowptr int64 [N+1]; col int32 [nnz] ascending
 *     inside a row; kstar uint8 [nnz]; w fp32 [nnz]; s, r fp32 [N, K].
 */
#ifndef DISENLINK_B200_H
#define DISENLINK_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DL_OK 0
#define DL_EINVAL (-1)      /* bad argument (null pointer, negative size, K or d out of range) */
#define DL_EWORKSPACE (-2)  /* workspace too small */
#define DL_ERANGE (-3)      /* an edge endpoint / pair id is outside [0, N) */
#define DL_EASYM (-4)       /* adjacency pattern is not symmetric */
#define DL_EUNSUPPORTED (-5)
#define DL_EINTERNAL (-6)   /* an internal invariant failed (debug builds only, e.g. -DDL_DEBUG_SINGLE_WRITER) */

#define DL_MAX_K 32         /* kstar is stored in 5 bits of a byte; K-factor count limit */
#define DL_MAX_D 256        /* per-factor width limit */
#define DL_SEG 512          /* edges per work item; rows with more edges are split (hub rows) */
#define DL_N_BUCKETS 33     /* degree classes: bucket b holds rows whose degree has bit length 32-b */
#define DL_HUB_BUCKET_END 23 /* buckets [0,23) hold degree classes 32..10, i.e. degree >= 512 */

typedef void* dl_stream_t;

int dl_abi_version(void);
const char* dl_error_string(int code);

/* ------------------------------------------------------------------------------------------
 * (1) adjacency -> CSR, reverse-edge index, degree buckets and work items.  Integer work.
 * [ref: main_disentangled.py:137-142]  adj = to_dense(train edges); adj[adj!=0]=1;
 *       adj_sym = adj + adj.t(); adj_sym[adj_sym!=0]=1   (duplicates collapse, diagonal kept)
 * ------------------------------------------------------------------------------------------ */

/* Bytes of scratch dl_csr_build needs for E directed input edges. */
size_t dl_csr_build_workspace_bytes(int64_t E, int64_t N);

/* src,dst int64 [E] -> rowptr [N+1], col [capacity >= 2E], *nnz_out (device int64).
 * status_out (device int32): 0, or DL_ERANGE if an endpoint is outside [0,N) (outputs undefined). */
int dl_csr_build(const int64_t* src, const int64_t* dst, int64_t E, int64_t N, int64_t* rowptr,
                 int32_t* col, int64_t* nnz_out, int32_t* status_out, void* ws, size_t ws_bytes,
                 dl_stream_t stream);

/* General form used by node-partitioned runs: rows in [0,n_rows), columns in [0,n_cols); when
 * symmetrize == 0 only (src -> dst) entries are produced (the caller lists both directions of the
 * edges whose row it owns).  dl_csr_build(N) == dl_csr_build_rect(N, N, 1). */
int dl_csr_build_rect(const int64_t* src, const int64_t* dst, int64_t E, int64_t n_rows,
                      int64_t n_cols, int symmetrize, int64_t* rowptr, int32_t* col,
                      int64_t* nnz_out, int32_t* status_out, void* ws, size_t ws_bytes,
                      dl_stream_t stream);

/* Same, from an already dense 0/1 (any non-zero counts) [N,N] fp32 adjacency that is used as is
 * (no symmetrisation): the drop-in path of Disentangle.forward(x, adj).  [ref: model.py:62]
 * Two calls: count (col == NULL) fills rowptr; fill (col != NULL) writes the columns. */
int dl_csr_from_dense(const float* adj, int64_t N, int64_t* rowptr, int32_t* col, void* ws,
                      size_t ws_bytes, dl_stream_t stream);

/* rev[e] = index of entry (j,i) for entry e=(i,j).  status_out = DL_EASYM if some entry has no
 * mirror.  The backward kernels rely on a symmetric pattern (always true for adj_sym). */
int dl_rev_index(const int64_t* rowptr, const int32_t* col, int64_t N, int64_t nnz, int64_t* rev,
                 int32_t* status_out, dl_stream_t stream);

/* Transposed pattern of a square CSR (the in-entries of every node), for the directed backward:
 * trowptr [N+1], tcol [nnz] = source row of each in-entry, tperm [nnz] = CSR index of each in-entry.
 * In-entries of a node are in CSR order (ascending source row for a CSR with sorted rows).  erow = the
 * COO row array of the CSR (dl_entry_rows).  col must lie in [0,N); N, nnz < 2^31 - 1.  Integer work,
 * bit-exact (stable radix sort). */
size_t dl_transpose_index_workspace_bytes(int64_t N, int64_t nnz);
int dl_transpose_index(const int32_t* col, const int32_t* erow, int64_t N, int64_t nnz, int64_t* trowptr,
                       int32_t* tcol, int32_t* tperm, void* ws, size_t ws_bytes, dl_stream_t stream);

/* Degree-sorted row bucketing: perm [N] = row ids ordered by degree class descending (stable),
 * bucket_off [DL_N_BUCKETS+1] (device int64) = start of each class in perm. */
size_t dl_degree_buckets_workspace_bytes(int64_t N);
int dl_degree_buckets(const int64_t* rowptr, int64_t N, int32_t* perm, int64_t* bucket_off,
                      void* ws, size_t ws_bytes, dl_stream_t stream);

/* Work items for hub rows (degree >= DL_SEG, i.e. degree class >= 10), which are the first
 * n_hub = bucket_off[DL_HUB_BUCKET_END] rows of perm.
 * hub_seg_ptr [n_hub+1] (device int64) = running count of DL_SEG-edge segments;
 * item_hub [n_items] = hub index of every segment.  Call once with item_hub == NULL to fill
 * hub_seg_ptr (the caller reads hub_seg_ptr[n_hub] to size item_hub), then again to fill it. */
int dl_hub_items(const int64_t* rowptr, const int32_t* perm, int64_t n_hub, int64_t* hub_seg_ptr,
                 int32_t* item_hub, int64_t n_items, dl_stream_t stream);

/* erow[e] = row of entry e (the COO row array of the CSR).  The streaming kernels cut the entries
 * into equal chunks regardless of row boundaries and read the row id per entry. */
int dl_entry_rows(const int64_t* rowptr, int64_t N, int64_t nnz, int32_t* erow, dl_stream_t stream);

/* Everything a kernel needs to walk the graph.  Plain-old-data, passed by pointer (host memory). */
typedef struct dl_graph {
  int64_t N;                   /* rows held here (all nodes on one GPU; the owned range when the
                                  nodes are partitioned across GPUs) */
  int64_t nnz;
  const int64_t* rowptr;       /* [N+1] */
  const int32_t* col;          /* [nnz] GLOBAL node ids */
  const int32_t* perm;         /* [N] local row ids in degree-class order, hub rows first */
  int64_t n_hub;               /* rows with degree >= DL_SEG */
  int64_t n_hub_items;         /* total segments of hub rows */
  const int64_t* hub_seg_ptr;  /* [n_hub+1] */
  const int32_t* item_hub;     /* [n_hub_items] */
  const int32_t* erow;         /* [nnz] local row id of every entry (COO row array, from
                                  dl_entry_rows); NULL = not built, the row-per-warp kernels are
                                  used instead of the streaming ones */
  int64_t row_base;            /* global node id of local row 0: per-node arrays (Z, H, s, r, G,
                                  dZ) are indexed by row_base + row, i.e. they are full-size
                                  [N_global, ...] arrays of which this call reads every gathered
                                  row and writes only the owned slice */
  uint32_t flags;              /* DL_F_* kernel-path switches; 0 = the fast paths.  Results are
                                  identical up to the stated tolerances whatever the flags (they
                                  exist for A/B measurements and for testing the other paths) */
} dl_graph;

/* dl_graph.flags */
#define DL_F_NO_STREAM 1u     /* row-per-warp / generic kernels instead of the streaming ones */
#define DL_F_NO_FL 2u         /* lane-per-chunk streaming kernels instead of the factor-per-lane ones */
#define DL_F_NO_FL_ATTN 4u    /* ... for the attention kernel only */
#define DL_F_NO_PRESCALE 8u   /* aggregation gathers s[col,k] per entry even when zs_scratch is given */
#define DL_F_NO_SJ 16u        /* backward pass 2 ignores the per-entry s[col,kstar] copy */
#define DL_F_NO_SR 32u        /* backward pass 2 gathers s and r separately instead of packed (s, r) */
#define DL_F_NO_XDOT 64u      /* backward pass 2 re-gathers the G[j,kstar] slice instead of reading the
                                 per-entry dot pass 1 left in x */
#define DL_F_NO_SYM 128u      /* (host side) attention evaluates both directions of every edge even when
                                 the symmetric path (dl_edge_attn_fwd_sym) is available */
#define DL_F_NO_KEEPA 256u    /* the symmetric attention does not store its softmax (a_out is ignored) and the
                                 symmetric backward pass 2 recomputes it (a_valid is ignored) */

/* ------------------------------------------------------------------------------------------
 * (2) per-edge K-factor attention with hard routing.
 * [ref: model.py:56-73]  q_k = z_i^k . z_j^k / T; a = softmax_k(q); kstar = argmax_k a (first
 *       max); w = a[kstar]; s[r,k] = sum of w over row r's entries routed to k, 0 -> 1.
 * hub_ws: fp32 scratch of dl_hub_scratch_floats(g, K) floats (may be NULL when n_hub == 0).
 * ------------------------------------------------------------------------------------------ */
size_t dl_hub_scratch_floats(const dl_graph* g_host, int64_t width);

int dl_edge_attn_fwd(const dl_graph* g_host, const float* Z, int K, int d, float T,
                     uint8_t* kstar, float* w, float* s, float* hub_ws, dl_stream_t stream);

/* (2s) the same, evaluating every undirected edge ONCE.  q_k(i,j) is symmetric and so are, bit for bit,
 * kstar and w (canonical arithmetic), so for a symmetric adjacency that is not row-partitioned the
 * 512-byte row gather is only needed for one entry of every edge -- the PRIMARY one: the entry whose row has
 * the larger degree (ties: the smaller row id; diagonal entries are primary).  Hub rows thereby keep their
 * length and most low-degree rows drop out of the evaluating kernels.
 *   dl_sym_index  (integer, once per graph; two calls like dl_hub_items)
 *       call 1 (ucol == NULL): uptr [N+1] (device int64) = row pointers of the primary view;
 *                              the caller reads uptr[N] = nnz_u to size ucol;
 *       call 2: ucol [nnz_u] = its columns, eidx [nnz] = for every entry of the full CSR its position t in
 *               the primary view (>= 0) or, for a secondary entry, ~t of its mirror (< 0);
 *               lcol / lmirror [nnz - nnz_u] (both or neither, may be NULL) = the secondary view
 *               (row pointers rowptr - uptr): its columns and, per entry, the primary-view position of
 *               the mirror -- used by the symmetric backward pass 2;
 *               status_out (device int32) = DL_EASYM if some entry has no mirror.
 *       erow = dl_entry_rows of the full CSR.  nnz < 2^31.  ws: dl_sym_index_workspace_bytes(N, nnz).
 *       ("upper" / "lower" in argument names = primary / secondary.)
 *   dl_edge_attn_fwd_sym: upper_host = a dl_graph over (uptr, ucol) with its own erow; the factor-per-lane
 *       attention kernel runs on it and leaves packed (w, kstar) records in kw_scratch (2 * nnz_u floats);
 *       a streaming pass expands them through eidx into kstar / w of the full CSR and makes the row
 *       sums s.  Outputs are identical to dl_edge_attn_fwd (kstar, w bit for bit; s up to the order of
 *       the fp32 row sums).  hub_ws: dl_hub_scratch_floats(g, K) floats.  DL_EUNSUPPORTED when (K, d) has
 *       no factor-per-lane instantiation: call dl_edge_attn_fwd instead.
 *       a_out (may be NULL; ignored under DL_F_NO_KEEPA in g_host->flags): nnz_u K floats that receive the
 *       softmax a[t, k] of every primary entry t (the bits w is taken from).  Handed to
 *       dl_factor_bwd_edges_sym as its coef_scratch with a_valid = 1, it spares backward pass 2 the dots,
 *       exponentials and softmax.  [ref: model.py:56-73] */
size_t dl_sym_index_workspace_bytes(int64_t N, int64_t nnz);
int dl_sym_index(const int64_t* rowptr, const int32_t* col, const int32_t* erow, int64_t N, int64_t nnz,
                 int64_t* uptr, int32_t* ucol, int32_t* eidx, int32_t* lcol, int32_t* lmirror, int32_t* status_out,
                 void* ws, size_t ws_bytes, dl_stream_t stream);
int dl_edge_attn_fwd_sym(const dl_graph* g_host, const dl_graph* upper_host, const int32_t* eidx, const float* Z,
                         int K, int d, float T, uint8_t* kstar, float* w, float* s, float* hub_ws,
                         float* kw_scratch, float* a_out, dl_stream_t stream);

/* (3) per-factor gather / segment-sum aggregation with the beta residual.
 * [ref: model.py:75]  H[i,k] = beta Z[i,k] + (1-beta) sum_{j: kstar(i,j)=k} w_ij / s[j,k] Z[j,k]
 * one_minus_beta is passed separately because Python evaluates (1 - beta) in double.
 * sj_out (may be NULL): per-entry copy sj[e] = s[col[e], kstar[e]] of the normaliser the kernel
 * gathers anyway; handing it to dl_factor_bwd(_edges) saves the backward one gather per entry.
 * zs_scratch (may be NULL): zs_rows*K*d floats of scratch, zs_rows = number of rows of Z and s (every
 * column index is below it; 0 = g.N).  When given, Z / s is written there in one streaming pass and the
 * kernel gathers pre-normalised slices: one DRAM transaction per entry instead of two (slice +
 * s[col,k]).  Needs row_base == 0 (one GPU, or the rank-local index space of a partitioned run, where
 * the rows beyond g.N are the halo) and is exclusive with sj_out (DL_EINVAL otherwise).
 * hub_ws: dl_hub_scratch_floats(g, K*d) floats. */
int dl_factor_spmm_fwd(const dl_graph* g_host, const float* Z, const uint8_t* kstar,
                       const float* w, const float* s, int K, int d, float beta,
                       float one_minus_beta, float* H, float* sj_out, float* zs_scratch, int64_t zs_rows,
                       float* hub_ws, dl_stream_t stream);

/* (4) backward of (2)+(3) w.r.t. Z given G = dL/dH.  dZ is ACCUMULATED into (it may already
 * hold the decoder's direct gradient); r [N,K] is scratch/output.  Closed form in DESIGN.md.
 * [ref: autograd of model.py:56-75].  sj (may be NULL): the sj_out of dl_factor_spmm_fwd.
 * sr_scratch (may be NULL): 2 * n_nodes * K floats of scratch, n_nodes = number of rows of s and r
 * (all nodes, not only the local rows): pass 2 packs (s, r) there and gathers both with one access.
 * x_scratch (may be NULL): nnz floats, see dl_factor_bwd_gather.
 * hub_ws: dl_hub_scratch_floats(g, K*d) floats. */
int dl_factor_bwd(const dl_graph* g_host, const float* Z, const float* G, const uint8_t* kstar,
                  const float* w, const float* s, const float* sj, float* sr_scratch, int64_t n_nodes,
                  float* x_scratch, int K, int d, float beta, float one_minus_beta, float T, float* dZ,
                  float* r, float* hub_ws, dl_stream_t stream);
/* The two passes of dl_factor_bwd on their own (a node-partitioned run all-gathers r between
 * them): pass 1 writes r and adds beta*G + T_ to dZ; pass 2 adds the attention-weight terms.
 * x (may be NULL): nnz floats.  Pass 1 holds, per entry e = (i,j), the routed slice G[j,kstar] it
 * gathers and the row's own Z[i]: it leaves x[e] = <G[j,kstar], Z[i,kstar]> there (canonical dot
 * order) and pass 2 reads those 4 bytes instead of gathering the 64-byte slice a second time.
 * x_valid_out (host int, may be NULL) is set to 1 when the pass-1 path taken filled x (the
 * streaming path), else 0; dl_factor_bwd_edges must only be given an x that was filled.
 * x_index (may be NULL): the eidx of dl_sym_index.  When given, only the primary entries (x_index[e] >= 0)
 * are written, at x[x_index[e]] (primary-view order, nnz_u floats), and ku_out [nnz_u] (may be NULL) receives
 * their kstar in the same order -- the layout dl_factor_bwd_edges_sym reads. */
int dl_factor_bwd_gather(const dl_graph* g_host, const float* Z, const float* G,
                         const uint8_t* kstar, const float* w, const float* s, int K, int d,
                         float beta, float one_minus_beta, float* dZ, float* r, float* x,
                         const int32_t* x_index, uint8_t* ku_out, int* x_valid_out, float* hub_ws,
                         dl_stream_t stream);
/* Pass 2 evaluating every undirected edge once (csrc/bwd_sym.cu): the coefficients
 * coef_e[kap] = dwsum_e w_e / T ((kap == kstar_e) - a_e[kap]) are the same numbers for (i,j) and (j,i), so the
 * dots, exponentials, softmax and (s, r) gathers run on the upper-triangle view only (phase A, which stores
 * coef [nnz_u, K] in coef_scratch) and the strictly-lower view gathers Z[j] and its mirror's coefficients
 * (phase B).  upper_host / lower_host / lmirror: dl_sym_index views (each with its own erow); ku, xu: kstar and
 * <G[j,k*], Z[i,k*]> in upper-view order (dl_factor_bwd_gather with x_index); sr_scratch: 2 n_nodes K floats;
 * coef_scratch: nnz_u K floats; hub_ws: dl_hub_scratch_floats(full graph, K*d) floats.  dZ is accumulated
 * into.  Equal to dl_factor_bwd_edges up to fp32 rounding (the two directions of an edge associate dwsum and
 * the row sums differently).  DL_EUNSUPPORTED when (K, d) has no factor-per-lane instantiation.
 * a_valid != 0: coef_scratch holds the softmax dl_edge_attn_fwd_sym stored through a_out for the same Z, T
 * and views; phase A reads it instead of recomputing it (and without the rows Z[i]), and overwrites it with
 * the coefficients, so the caller clears its record of a valid softmax after this call.  Ignored under
 * DL_F_NO_KEEPA in upper_host->flags. */
int dl_factor_bwd_edges_sym_supported(int K, int d);     /* 1 when (K, d) has the kernels, else 0 */
int dl_factor_bwd_edges_sym(const dl_graph* upper_host, const dl_graph* lower_host, const int32_t* lmirror,
                            const float* Z, const float* G, const uint8_t* ku, const float* s, const float* r,
                            float* sr_scratch, int64_t n_nodes, const float* xu, float* coef_scratch, int K, int d,
                            float one_minus_beta, float T, int a_valid, float* dZ, float* hub_ws, dl_stream_t stream);
int dl_factor_bwd_edges(const dl_graph* g_host, const float* Z, const float* G,
                        const uint8_t* kstar, const float* w, const float* s, const float* r,
                        const float* sj, float* sr_scratch, int64_t n_nodes, const float* x, int K,
                        int d, float one_minus_beta, float T, float* dZ, float* hub_ws,
                        dl_stream_t stream);
/* Backward of the attention + aggregation for ANY 0/1 pattern (csrc/bwd_dir.cu): the autograd of
 * model.py:56-75 when adj is not symmetric (e.g. the directed train adjacency).  Given G = dL/dH, with
 * e = (i,j), k = kstar[e]:  T_[j,k] = (1-beta)/s[j,k] sum_{in-entries e of j, kstar=k} w[e] G[i,k];
 * r[j,k] = <Z[j,k], T_[j,k]>/s[j,k], or 0 when row j has no entry routed to k (the reference's clamped
 * s[j,k] = 1 passes no gradient); dZ[j] += beta G[j] + T_[j];  dw[e] = (1-beta)<G[i,k],Z[j,k]>/s[j,k] - r[i,k];
 * coef[e,kk] = dw[e] w[e]/T ((kk==k) - a[e,kk]);  dZ[i,kk] += coef Z[j,kk];  dZ[j,kk] += coef Z[i,kk].
 * g_host: the CSR (row_base 0, one GPU); gt_host, tperm: its transposed pattern as a dl_graph of its own
 * (dl_transpose_index) and the CSR index of every in-entry.  dZ is accumulated into; r [N,K] is written.
 * dw_scratch: nnz floats; routed_scratch: N uint32 (K <= 32); hub_ws / hub_ws_t:
 * dl_hub_scratch_floats(g / gt, K*d) floats.  Gathers only, no floating-point atomics, deterministic. */
int dl_factor_bwd_directed(const dl_graph* g_host, const dl_graph* gt_host, const int32_t* tperm,
                           const float* Z, const float* G, const uint8_t* kstar, const float* w, const float* s,
                           int K, int d, float beta, float one_minus_beta, float T, float* dZ, float* r,
                           float* dw_scratch, uint32_t* routed_scratch, float* hub_ws, float* hub_ws_t,
                           dl_stream_t stream);
/* One phase of dl_factor_bwd_directed, for the rank-local graphs of a node-partitioned step
 * (disenlink_b200/partition.py, DirectedPartitionedLinkStep), which exchanges data between the phases:
 *   phase 1: routed mask of the rows of g, pass 1 over gt (T_, r, dZ += beta G + T_), in-hub finish;
 *   phase 2: pass 2 out-side over g (writes dw[0, g.nnz)), hub fixup;
 *   phase 3: pass 2 in-side over gt (reads dw and kstar through tperm), hub fixup.
 * dl_factor_bwd_directed is phases 1, 2, 3 in order (the same launches).  Rank-local shapes are accepted:
 * g and gt have the same N (the owned rows) and row_base 0, gt->nnz may differ from g->nnz, every column of
 * g and gt is below n_tot (the rows of Z, G, s: owned + halo) and every tperm value below n_rec (the length
 * of the per-entry arrays kstar, w, dw: the own entries [0, g.nnz) followed by records pushed by the owners
 * of remote in-entries), n_rec >= g->nnz.  Arguments, columns and tperm are checked (DL_EINVAL otherwise);
 * the index check is one pass over the phase's columns / tperm and one stream synchronisation.
 * routed_scratch: phase 1 only; r: written by phase 1, read by phase 2; hub_ws: phase 2; hub_ws_t:
 * phases 1 and 3. */
int dl_factor_bwd_directed_phase(const dl_graph* g_host, const dl_graph* gt_host, const int32_t* tperm,
                                 const float* Z, const float* G, const uint8_t* kstar, const float* w,
                                 const float* s, int K, int d, float beta, float one_minus_beta, float T,
                                 int64_t n_tot, int64_t n_rec, float* dZ, float* r, float* dw,
                                 uint32_t* routed_scratch, float* hub_ws, float* hub_ws_t, int phase,
                                 dl_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * (5) factor-weighted link-pair scoring over explicit (u,v) batches.
 * [ref: model.py:109-113]  logit = sum_k exp(z_u^k.z_v^k/T) (h_u^k.h_v^k); prob = sigmoid(logit)
 * logit / prob may each be NULL (not both).  Ids must lie in [0,N); the caller validates them once
 * per batch (dl_pair_incidence reports DL_ERANGE-free lists only for valid ids).
 * ------------------------------------------------------------------------------------------ */
int dl_pair_score_fwd(const int32_t* u, const int32_t* v, int64_t P, const float* Z,
                      const float* H, int64_t N, int K, int d, float T, float* logit, float* prob,
                      dl_stream_t stream);

/* Node-major incidence lists of a pair batch (built once per batch, integer work):
 * inc_ptr [N+1] int64, inc_other [2P] int32 (the other endpoint), inc_pair [2P] int32 (pair id),
 * in pair order inside a node.  Needed by the atomic-free backward. */
size_t dl_pair_incidence_workspace_bytes(int64_t P, int64_t N);
int dl_pair_incidence(const int32_t* u, const int32_t* v, int64_t P, int64_t N, int64_t* inc_ptr,
                      int32_t* inc_other, int32_t* inc_pair, void* ws, size_t ws_bytes,
                      dl_stream_t stream);

/* Incidence lists of the nodes in [row_lo, row_hi) only (a rank's owned range); inc_ptr has
 * row_hi-row_lo+1 entries and inc_ptr[last] is the number of incidences kept. */
int dl_pair_incidence_range(const int32_t* u, const int32_t* v, int64_t P, int64_t row_lo,
                            int64_t row_hi, int64_t* inc_ptr, int32_t* inc_other, int32_t* inc_pair,
                            void* ws, size_t ws_bytes, dl_stream_t stream);

/* Backward of the decoder given dS = dL/dlogit [P].  `inc_host` is the incidence structure seen
 * as a graph (rowptr = inc_ptr, col = inc_other, plus perm / hub items from dl_degree_buckets and
 * dl_hub_items, so nodes that take part in many pairs are split like hub rows).  dZ, dH [N,K,d]
 * are OVERWRITTEN (every node's row is written exactly once; no atomics).
 * hub_ws: dl_hub_scratch_floats(inc, 2*K*d) floats.  [ref: autograd of model.py:109-113] */
int dl_pair_score_bwd(const dl_graph* inc_host, const int32_t* inc_pair, const float* Z,
                      const float* H, const float* dS, int K, int d, float T, float* dZ, float* dH,
                      float* hub_ws, dl_stream_t stream);

/* Dense all-pairs decoder for the small-N drop-in contract: out [N,N] = sigmoid(logit(u,v)).
 * [ref: model.py:109-113, consumed by main_disentangled.py:195,202,217 via boolean masks] */
int dl_allpairs_score_fwd(const float* Z, const float* H, int64_t N, int K, int d, float T,
                          float* prob, dl_stream_t stream);
/* dSsym [N,N] = dS + dS^T with dS = dL/dlogit (dense; zeros are skipped) -> dZ, dH overwritten. */
int dl_allpairs_score_bwd(const float* Z, const float* H, const float* dSsym, int64_t N, int K,
                          int d, float T, float* dZ, float* dH, dl_stream_t stream);

/* Dense [K,N,N] views of the layer's internals for API parity with Disentangle_layer.forward's
 * second and third returns (alpha0 = exp(zz^T/T); att).  Small N only.  [ref: model.py:57,74,77] */
int dl_dense_alpha0(const float* Z, int64_t N, int K, int d, float T, float* alpha0,
                    dl_stream_t stream);
int dl_dense_att(const dl_graph* g_host, const uint8_t* kstar, const float* w, const float* s,
                 int K, float* att, dl_stream_t stream);

/* ---- weighted BCE over a pair list, forward + backward fused ------------------------------
 * [ref: main_disentangled.py:195 -- F.binary_cross_entropy(a_pred[mask == 1], target) summed over the
 * positive mask and the m negative masks; the per-pair weights fold the means and the 1/m.]
 *   loss[0] = sum_p weights[p] * -( y log p + (1 - y) log(1 - p) ),  logs clamped at -100 (torch)
 *   dS[p]   = weights[p] (p - y) / max(p (1 - p), 1e-12) * (1 - p) p      (dL/dlogit; NULL: skipped)
 * weights may be NULL (all ones).  ws: >= dl_link_bce_workspace_bytes() bytes of device scratch.
 * Deterministic: partial sums are combined in a fixed order. */
int64_t dl_link_bce_workspace_bytes(void);
int dl_link_bce(const float* prob, const float* labels, const float* weights, int64_t P, float* dS,
                float* loss, void* ws, int64_t ws_bytes, dl_stream_t stream);

/* The loss of dl_link_bce on every segment [seg_ptr[r], seg_ptr[r+1]) of one pair list, r < R: the independent
 * runs of the script trained as one union (disenlink_b200/runs.py), each run's pairs one segment.
 * [ref: main_disentangled.py:131,195 -- one loss per run of the `for run in range(args.run)` loop]
 *   loss[r] = sum over the segment of weights[p] * -( y log p + (1 - y) log(1 - p) )   (dl_link_bce's terms)
 * Loss only (the gradient of the union comes from dl_link_bce).  seg_ptr: int64 [R+1] on the device,
 * 0 = seg_ptr[0] <= ... <= seg_ptr[R] = P (reads are clamped to [0, P) whatever it holds); an empty segment
 * gives 0.  Deterministic: double partial sums combined in a fixed order.
 * ws: >= dl_link_bce_segments_workspace_bytes(R) bytes of device scratch. */
int64_t dl_link_bce_segments_workspace_bytes(int64_t R);
int dl_link_bce_segments(const float* prob, const float* labels, const float* weights, int64_t P,
                         const int64_t* seg_ptr, int64_t R, float* loss, void* ws, int64_t ws_bytes,
                         dl_stream_t stream);

/* ---- ROC-AUC of a score list ----------------------------------------------------------------
 * [ref: main_disentangled.py:202-204,217-219 -- sklearn.metrics.roc_auc_score(y, a_pred[mask == 1])]
 * labels: 0 / non-zero floats.  out: 5 doubles on the device = { auc, n_pos, n_neg, n_nan, 2U } where
 * 2U = sum over positives of 2 * #(negatives below) + #(negatives tied) (an exact integer) and
 * auc = 2U / (2 n_pos n_neg); auc is NaN when a class is empty or a score is NaN (sklearn raises).
 * P < 2^31.  ws: >= dl_roc_auc_workspace_bytes(P) bytes of device scratch. */
int64_t dl_roc_auc_workspace_bytes(int64_t P);
int dl_roc_auc(const float* score, const float* labels, int64_t P, double* out, void* ws, int64_t ws_bytes,
               dl_stream_t stream);

/* dl_roc_auc on every segment [seg_ptr[r], seg_ptr[r+1]) of one score list, r < R: out[5r .. 5r+4] =
 * { auc, n_pos, n_neg, n_nan, 2U } of that segment alone, equal bit for bit to dl_roc_auc on it (an empty,
 * one-class or NaN segment gives NaN in its own row only).  Equal scores in different segments never tie.
 * [ref: main_disentangled.py:131,202-204,217-219 -- roc_auc_score per run of the `for run in range(args.run)` loop]
 * seg_ptr: int64 [R+1] on the device with 0 = seg_ptr[0] <= ... <= seg_ptr[R] = P.  P < 2^31, 1 <= R < 2^31.
 * ws: >= dl_roc_auc_segments_workspace_bytes(P, R) bytes of device scratch. */
int64_t dl_roc_auc_segments_workspace_bytes(int64_t P, int64_t R);
int dl_roc_auc_segments(const float* score, const float* labels, int64_t P, const int64_t* seg_ptr, int64_t R,
                        double* out, void* ws, int64_t ws_bytes, dl_stream_t stream);

/* ---- first layer of the factor MLPs from sparse features (csrc/feat_proj.cu) ----------------
 * [ref: model.py:24-27,106]  A = act(x W1^T + b1) of the K factors (all runs of a union) at once, x [N, F] sparse
 * bag-of-words features.  x is given as CSR (rowptr int64 [N+1], col int32, val fp32, rows sorted by column) for
 * the forward and as CSC (row int32, cval fp32, rows ascending inside a column) for the weight gradient.
 * Wt = W1^T is [F, J] row-major, b [J]; relu = 1: act = ReLU (Factor2), 0: the identity (Factor, nhid == 1).
 *   forward:   A[n, j] = act( (sum over row n's entries p, in CSR order, of val[p] Wt[col[p], j]) + b[j] )
 *   backward:  G' = G * 1[A > 0] (relu only);  dWt[f, j] = sum over column f's entries p, in CSC order, of
 *              cval[p] G'[row[p], j];  db[j] = sum_n G'[n, j].  dWt (contiguous [F, J]) and db are overwritten.
 * Each sum is one fixed-order chain that depends on neither J nor the launch shape; no atomics, so the results
 * are bitwise reproducible and a run's block of a union's Wt gives that run's A and dWt on its own.
 * A and G are addressed as element (n, j) at n * row_stride + (j / blk) * blk_stride + j % blk (blk = nhid,
 * J % blk == 0): the [B, N, nhid] view of [N, J] the second layer reads and the gradient its backward returns.
 * The CSC entries are cut into items: items [0, n_slots) are the chunks of the n_heavy columns longer than the
 * caller's chunk length, in column order, chunks in order (heavy_col [n_heavy], heavy_ptr [n_heavy+1] = their
 * item ranges); items [n_slots, n_items) are the other columns, one whole (possibly empty) column each.  Item t
 * covers CSC entries [item_lo[t], item_hi[t]) of column item_col[t]; n_items = F + n_slots - n_heavy.
 * ws: dl_feat_proj_bwd_workspace_bytes(N, J, n_slots) bytes (G', db partials, chunk partial rows).
 * Any J >= 1 (float4 access when J, blk, the strides and the pointers allow it).  DL_EINVAL on bad sizes. */
int dl_feat_proj_fwd(const int64_t* rowptr, const int32_t* col, const float* val, int64_t N, int64_t F,
                     const float* Wt, const float* b, int64_t J, int relu, float* A, int64_t a_row_stride,
                     int64_t a_blk_stride, int64_t blk, dl_stream_t stream);
size_t dl_feat_proj_bwd_workspace_bytes(int64_t N, int64_t J, int64_t n_slots);
int dl_feat_proj_bwd(const int32_t* row, const float* cval, const int32_t* item_col, const int64_t* item_lo,
                     const int64_t* item_hi, int64_t n_items, int64_t n_slots, const int32_t* heavy_col,
                     const int64_t* heavy_ptr, int64_t n_heavy, int64_t N, int64_t F, const float* A,
                     int64_t a_row_stride, int64_t a_blk_stride, const float* G, int64_t g_row_stride,
                     int64_t g_blk_stride, int64_t blk, int64_t J, int relu, float* dWt, float* db, void* ws,
                     size_t ws_bytes, dl_stream_t stream);

/* ---- structured negative sampling ---------------------------------------------------------
 * [ref: main_disentangled.py:160 -- torch_geometric.utils.structured_negative_sampling(edge_index)]
 * For every edge e with source src[e]: k_out[e] ~ U[0, num_nodes) redrawn while (src[e], k) is an
 * entry of g (the CSR of the DIRECTED edge columns, dl_csr_build_rect with symmetrize = 0).  Draw t of
 * edge e is Philox4x32-10(key = seed, counter = (e, t)) -> r = (c1 << 32 | c0), k = (r * num_nodes) >> 64.
 * After max_tries rejected draws the first non-neighbour of the row is used; a row adjacent to every
 * node yields -1 and is counted in n_failed[0] (device int). */
int dl_structured_negative_sampling(const dl_graph* g_host, const int64_t* src, int64_t E, int64_t num_nodes,
                                    uint64_t seed, int max_tries, int64_t* k_out, int* n_failed,
                                    dl_stream_t stream);

/* ---- all-gather of a node-partitioned array as a push over NVLink peer memory ---------------
 * The owner of a slice writes it into the same position of every peer's copy of the array:
 * peer_dst[q] (host array of n_peers <= 15 device pointers, already offset to the slice, mapped into
 * this process with CUDA IPC) receives the n_bytes at src.  All pointers 16-byte aligned.  The call
 * only enqueues the kernel; the caller orders the ranks (a barrier after it, and none of the peers
 * may still be reading the previous contents). */
int dl_push_slice(const void* src, void* const* peer_dst, int n_peers, int64_t n_bytes, dl_stream_t stream);
/* The two kernels whose output is exchanged right after them, with the exchange fused in: every owned
 * row they finish is stored into the local array AND into the same row of each peer's copy
 * (H_peers / dH_peers: host arrays of n_peers <= 15 device pointers to the peers' full-size arrays,
 * mapped with dl_ipc_open), so the all-gather overlaps the kernel instead of following it.  The
 * caller still orders the ranks with a barrier afterwards.  Otherwise identical to
 * dl_factor_spmm_fwd (without the zs_scratch path) and dl_pair_score_bwd.  The same for the two small
 * per-node arrays: dl_edge_attn_fwd_push stores s, dl_factor_bwd_gather_push stores r. */
int dl_factor_spmm_fwd_push(const dl_graph* g_host, const float* Z, const uint8_t* kstar,
                            const float* w, const float* s, int K, int d, float beta,
                            float one_minus_beta, float* H, float* sj_out, float* hub_ws,
                            float* const* H_peers, int n_peers, dl_stream_t stream);
int dl_edge_attn_fwd_push(const dl_graph* g_host, const float* Z, int K, int d, float T,
                          uint8_t* kstar, float* w, float* s, float* hub_ws, float* const* s_peers, int n_peers,
                          dl_stream_t stream);
int dl_factor_bwd_gather_push(const dl_graph* g_host, const float* Z, const float* G,
                              const uint8_t* kstar, const float* w, const float* s, int K, int d,
                              float beta, float one_minus_beta, float* dZ, float* r, float* x,
                              int* x_valid_out, float* hub_ws, float* const* r_peers, int n_peers,
                              dl_stream_t stream);
int dl_pair_score_bwd_push(const dl_graph* inc_host, const int32_t* inc_pair, const float* Z,
                           const float* H, const float* dS, int K, int d, float T, float* dZ, float* dH,
                           float* hub_ws, float* const* dH_peers, int n_peers, dl_stream_t stream);
/* ---- halo exchange of a node-partitioned run ------------------------------------------------
 * Rank-local storage: a rank keeps its own rows [0, n_own) of every per-node array followed by the halo
 * rows [n_own, n_own + n_halo) -- the remote nodes its CSR columns and pair lists reference, grouped by
 * owner -- and its CSR columns are local indices (dl_graph.N = n_own, row_base = 0).  Before a kernel
 * reads halo rows their OWNERS push them: exactly the rows (or, for dH, the routed factor slices) the
 * peer reads, straight into the peer's array over NVLink peer memory.  No collective library call, no
 * reduction; the caller orders the ranks with a barrier after the pushes.
 *
 * dl_push_rows: for every peer q (descs_host[q], host array) and t in [0, n):
 *     dst_q[(dst_idx ? dst_idx[t] : t)] = src[(src_idx ? src_idx[t] : t)]     rows of row_bytes bytes
 * dst = device pointer into the peer's array (mapped with dl_ipc_open), already offset to the block that
 * receives this rank's rows when dst_idx == NULL.  vec_per_factor > 0 (a power of two) and desc.mask != NULL: a row is
 * K = row_bytes / (16 vec_per_factor) factor slices and only the slices k with bit k of mask[source row]
 * set are sent (the routed slices of dH the peer's backward pass 1 gathers; the others are never read).
 * row_bytes % 16 == 0, pointers 16-byte aligned, n_peers <= 15.  One launch for all peers. */
typedef struct dl_push_desc {
  void* dst;
  const int32_t* src_idx;
  const int32_t* dst_idx;
  const uint32_t* mask;
  int64_t n;
} dl_push_desc;
int dl_push_rows(const void* src, int64_t row_bytes, int vec_per_factor, const dl_push_desc* descs_host,
                 int n_peers, dl_stream_t stream);
/* dl_push_entries: the per-entry records of the directed step (kstar: 1 byte, w and dw: 4 bytes).  For every
 * peer q and t in [0, n):  dst_q[(dst_idx ? dst_idx[t] : t)] = src[(src_idx ? src_idx[t] : t)], elements of
 * elem_bytes (1 or 4) bytes.  dst = the peer's array, already offset to the block that receives this rank's
 * records; desc.mask must be NULL; a descriptor with n = 0 is allowed.  Plain stores, one launch for all
 * peers, n_peers <= 15. */
int dl_push_entries(const void* src, int elem_bytes, const dl_push_desc* descs_host, int n_peers,
                    dl_stream_t stream);
/* Which factor slices of an owned row does each peer read?  By the symmetry of adjacency and routing, peer p
 * gathers G[j, k] (j owned here) exactly when this rank holds an entry (j, i) routed to k with i owned by p.
 * masks [n_parts][g.N] (device uint32, overwritten): bit k of masks[p][j] set accordingly.  halo_off
 * [n_parts + 1] (device int32) = boundaries of the owners' blocks in the local column index space
 * (halo_off[0] = n_own; an empty block for this rank itself).  Integer work (atomicOr), n_parts <= 16. */
int dl_need_masks(const dl_graph* g_host, const uint8_t* kstar, const int32_t* halo_off, int n_parts,
                  uint32_t* masks, dl_stream_t stream);
/* cudaDeviceEnablePeerAccess(peer_device) for the current device; DL_EINVAL if the pair has no P2P path. */
int dl_enable_peer_access(int peer_device);
/* Map / unmap a peer process's allocation for kernels of the CURRENT device: handle = the 64 bytes of the
 * owner's cudaIpcMemHandle_t; base_out receives the base address of that allocation in this process. */
int dl_ipc_open(const void* handle, void** base_out);
int dl_ipc_close(void* base);

#ifdef __cplusplus
}
#endif
#endif /* DISENLINK_B200_H */
