/*
 * lstep_b200.h — C ABI of the B200-native (sm_100a) L-STEP positional-encoding hot path.
 *
 * The reference (kthrn22/L-STEP) has no FFI layer: its hot path is Python/PyTorch code
 * (SURVEY.md §8(b)). Each entry point below names the reference code it replaces, relative to
 * /root/reference. A host binds these with ctypes (INTEGRATION.md); the in-tree Python host is
 * l-step_b200/_lib.py.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in _host;
 *   - every function enqueues work on `stream` (a cudaStream_t passed as void*) and returns
 *     without synchronising; nothing allocates device memory — scratch comes from a caller
 *     owned workspace whose size lstep_workspace_bytes() reports — so a call sequence can be
 *     captured in a CUDA graph;
 *   - the return value is an lstep_status; functions never throw; asynchronous data errors
 *     (an out-of-range node id) are reported through a caller supplied device flag word;
 *   - node / edge ids cross the ABI as int64 (the reference's numpy longlong), times as
 *     float64, PE values and neighbour times as float32, exactly as in the reference.
 */
#ifndef LSTEP_B200_H
#define LSTEP_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LSTEP_ABI_VERSION 2

typedef enum lstep_status {
  LSTEP_OK = 0,
  LSTEP_ERR_INVALID_ARG = 1,   /* null pointer, negative size, K <= 0 (utils/utils.py:156 assert) */
  LSTEP_ERR_UNSUPPORTED = 2,   /* shape outside what the kernels were built for */
  LSTEP_ERR_WORKSPACE = 3,     /* workspace too small */
  LSTEP_ERR_CUDA = 4,          /* a CUDA runtime call failed; see lstep_last_cuda_error() */
  LSTEP_ERR_ID_RANGE = 5       /* id outside the table, or not representable in the int32 device encoding */
} lstep_status;

/* bits set in the device `err_flag` word by kernels */
#define LSTEP_FLAG_NODE_OUT_OF_RANGE 1u /* utils/utils.py:140 would raise IndexError (SURVEY Q8) */
#define LSTEP_FLAG_UNSORTED_STREAM 2u
#define LSTEP_FLAG_CHANGELOG_FULL 4u /* a step changed more rows than the change-log history has event capacity for */
#define LSTEP_FLAG_PEER_TIMEOUT 8u   /* a peer GPU did not reach a step barrier within the time limit (peer group step) */
#define LSTEP_FLAG_CSR_FULL 16u      /* an append to a growable CSR found no room in a row; nothing was written to that row */
/* Phase B of update_pe adds its contributions in 32.32 fixed point (int64). A call with n rows of K slots raises this flag
 * when a contribution it adds that way is non-finite or has |x| >= 2^31 / (n*K + 1) (fp32, rounded toward zero): below that
 * bound every column sum provably fits in int64, at or above it the sum may wrap and the updated rows are not the
 * reference's. The push form checks every batch row's phase-A values and time features; the pull form checks the
 * contributions to lists longer than 4 slots (shorter lists and the padding row are fp32 sums there). */
#define LSTEP_FLAG_FIXED_POINT_RANGE 32u

const char* lstep_strerror(int status);
const char* lstep_last_cuda_error(void);
int lstep_abi_version(void);
/* 1 when a CUDA device of compute capability 10.x is current; the library has no other path */
int lstep_device_ok(void);

/* ------------------------------------------------------------------------------------------
 * a1 — time-sorted CSR of the undirected temporal adjacency.
 * Replaces get_neighbor_sampler + NeighborSampler.__init__ (utils/utils.py:282-301, 72-109):
 * entry order per node = stable sort by time of the insertion order (edge order, source side
 * before destination side).
 * ------------------------------------------------------------------------------------------ */
typedef struct lstep_csr {
  const int64_t* indptr; /* [num_rows + 1] */
  const int32_t* nbr;    /* [nnz] neighbour node id */
  const int32_t* eid;    /* [nnz] edge id */
  const double* t;       /* [nnz] interaction time, ascending within a row */
  int64_t num_rows;      /* max node id + 1 (row 0 = padding node, empty) */
  int64_t nnz;
} lstep_csr;

/* Bytes of scratch lstep_csr_build_* needs for `n_entries` adjacency entries. */
size_t lstep_csr_build_workspace_bytes(int64_t n_entries, int64_t num_rows);

/* Edge stream (src,dst,eid,t)[E] -> CSR with 2E entries. Outputs are caller allocated:
 * indptr[num_rows+1], nbr/eid[2E], t[2E]. */
int lstep_csr_build_from_edges(const int64_t* src, const int64_t* dst, const int64_t* eid, const double* t,
                               int64_t num_edges, int64_t num_rows, int64_t* out_indptr, int32_t* out_nbr,
                               int32_t* out_eid, double* out_t, void* workspace, size_t workspace_bytes,
                               uint32_t* err_flag, void* stream);

/* Flattened adjacency lists (owner node, neighbour, edge id, time)[n] in list order -> CSR
 * (the NeighborSampler(adj_list=...) constructor form). */
int lstep_csr_build_from_entries(const int64_t* owner, const int64_t* nbr, const int64_t* eid, const double* t,
                                 int64_t n_entries, int64_t num_rows, int64_t* out_indptr, int32_t* out_nbr,
                                 int32_t* out_eid, double* out_t, void* workspace, size_t workspace_bytes,
                                 uint32_t* err_flag, void* stream);

/* ------------------------------------------------------------------------------------------
 * Growable CSR (csrc/csr_grow.cu): an lstep_csr whose rows end in padding, plus int32 fill[num_rows]. Row v holds its
 * real entries at [indptr[v], indptr[v] + fill[v]); the rest of [indptr[v], indptr[v+1]) is padding (t = +inf, nbr = 0,
 * eid = 0), which no lookup selects (every reader counts entries with t < tq, strict, and none reads nnz). Every entry
 * point that takes an lstep_csr reads a growable one unchanged and returns what it returns on the exact CSR of the
 * same edges.
 * lstep_csr_relayout copies each row's real entries (src_fill NULL: src is exact, every entry is real) to
 * [new_indptr[v], ...) of the output arrays, pads the rest of each new row and writes out_fill. Output arrays must not
 * alias src's. A row whose new capacity is below its fill keeps its first entries and raises LSTEP_FLAG_CSR_FULL.
 * lstep_csr_ingest appends a batch of edges in the reference's order (utils/utils.py:292-299): for edge i, (dst, eid, t)
 * to row src, then (src, eid, t) to row dst (a self-loop gives two entries); eid NULL: eid_base + i. Times must be
 * non-decreasing across the batch and not earlier than any real entry of a row they go to (else
 * LSTEP_FLAG_UNSORTED_STREAM); a row without room for its entries of a chunk of 2048 edges gets none of them
 * (LSTEP_FLAG_CSR_FULL); an edge with an id outside the rows or an eid outside int32 is dropped
 * (LSTEP_FLAG_NODE_OUT_OF_RANGE).
 * ------------------------------------------------------------------------------------------ */
int lstep_csr_relayout(const lstep_csr* src, const int32_t* src_fill, const int64_t* new_indptr, int32_t* out_nbr,
                       int32_t* out_eid, double* out_t, int32_t* out_fill, uint32_t* err_flag, void* stream);
int lstep_csr_ingest(const lstep_csr* csr, int32_t* fill, const int64_t* src, const int64_t* dst, const int64_t* eid,
                     int64_t eid_base, const double* t, int64_t n_edges, uint32_t* err_flag, void* stream);
/* Row capacity of a growable CSR: indptr has row_cap + 1 entries, csr->num_rows counts the LIVE rows (every lookup's
 * bound), and the arrays end in a padded tail [indptr[num_rows], nnz) that new rows take their entries from.
 * lstep_csr_relayout_rows is lstep_csr_relayout for a regrow that may add rows: rows [src->num_rows, new_rows) are new
 * (all padding, fill 0), out_fill[new_rows .. row_cap) = 0, new_indptr holds new_rows + 1 entries (the caller may fill the
 * rest), and the tail [new_indptr[new_rows], total) is padded (total < 0: no tail). lstep_csr_relayout(src, ...) is
 * lstep_csr_relayout_rows(src, ..., src->num_rows, src->num_rows, ..., -1, ...).
 * lstep_csr_add_rows makes n_rows more rows live without moving any entry: row csr->num_rows + i gets cap[i] (device
 * int64 [n_rows]) entries of the tail, i.e. indptr[num_rows + 1 + i] = indptr[num_rows] + cap[0] + ... + cap[i], and fill 0;
 * then csr->num_rows += n_rows (host side). The caller guarantees room: num_rows + n_rows <= row_cap and the caps fit the
 * tail. One CTA; stream-ordered after lookups already enqueued, which never read rows at or above their num_rows. */
int lstep_csr_relayout_rows(const lstep_csr* src, const int32_t* src_fill, int64_t new_rows, int64_t row_cap, const int64_t* new_indptr,
                            int64_t total, int32_t* out_nbr, int32_t* out_eid, double* out_t, int32_t* out_fill, uint32_t* err_flag,
                            void* stream);
int lstep_csr_add_rows(lstep_csr* csr, int32_t* fill, int64_t n_rows, const int64_t* cap, void* stream);

/* ------------------------------------------------------------------------------------------
 * a2 — most-recent-K temporal neighbour lookup (kernel K1).
 * Replaces NeighborSampler.get_historical_neighbors, 'recent' strategy, and
 * find_neighbors_before (utils/utils.py:129-146, 148-213). Row i < n_valid: c = #entries of
 * q_node[i] with t < q_time[i] (strict, fp64), the last min(K,c) are written right-aligned into
 * columns [K-len, K), the rest are 0. Rows n_valid <= i < n_rows are all zero (the reference's
 * zip() truncation, SURVEY Q1). Outputs [n_rows, K]; out_eid may be NULL.
 * ------------------------------------------------------------------------------------------ */
int lstep_sample_recent(const lstep_csr* csr, const int64_t* q_node, const double* q_time, int64_t n_rows,
                        int64_t n_valid, int K, int64_t* out_nbr, int64_t* out_eid, float* out_t,
                        uint32_t* err_flag, void* stream);

/* Device-internal compact form consumed by the aggregation kernels: int32 ids, no edge ids. */
int lstep_sample_recent_compact(const lstep_csr* csr, const int64_t* q_node, const double* q_time, int64_t n_rows,
                                int64_t n_valid, int K, int32_t* out_nbr, float* out_t, uint32_t* err_flag,
                                void* stream);

/* ------------------------------------------------------------------------------------------
 * a3 — learnable DFT filter over each node's PE history (kernel K3).
 * Replaces LSTEP.fourier_transform_pe (models/LSTEP.py:104-137). FFT -> mask -> complex filter
 * -> mask -> iFFT -> mask -> real -> Linear(T->1) is linear in the history, so it collapses to
 *     out[n,c] = sum_{s < Th} G[s,c] * hist[ids[n], s, c]
 * with a real table G[T,d] that depends on the parameters and on min(batch_idx, T) only.
 * lstep_dft_collapse computes G (fp64 accumulation) from fft_filter.weight (complex64 [T,d],
 * interleaved re/im) and fft_agg.weight ([T]); `b` is the mask length (T when unmasked).
 * History element (node v, step s, column c) lives at
 *     hist[v*node_stride + ((s0 + s) % ring) * time_stride + c]
 * (reference layout [V1,Th,d]: node_stride=Th*d, time_stride=d, s0=0, ring=Th).
 * ------------------------------------------------------------------------------------------ */
int lstep_dft_collapse(const float* fft_filter_weight_c64, const float* fft_agg_weight, int T, int d, int b, float* G,
                       void* stream);
int lstep_dft_filter(const float* hist, int64_t node_stride, int64_t time_stride, int s0, int ring, int Th, int d,
                     const int64_t* ids, int64_t n_ids, const float* G, float* out, int64_t out_stride, void* stream);
/* dG[s,c] = sum_n hist[ids[n],s,c] * dout[n,c]  (s < Th; rows Th..T-1 of dG are left untouched) */
int lstep_dft_filter_bwd(const float* hist, int64_t node_stride, int64_t time_stride, int s0, int ring, int Th, int d,
                         const int64_t* ids, int64_t n_ids, const float* dout, float* dG, void* stream);

/* ------------------------------------------------------------------------------------------
 * PE MLP parameters, packed for the kernels: every Linear weight transposed and zero padded to
 * [in_pad][ldo] (in_pad = lstep_packed_rows(in), ldo = lstep_packed_ld(out)) so that a tile of 16
 * input rows is one contiguous block a bulk async copy can stream; biases padded to ldo.
 * lstep_pack_linear does one layer.
 * ------------------------------------------------------------------------------------------ */
int lstep_packed_ld(int out_features);
int lstep_packed_rows(int in_features);
size_t lstep_packed_tc_floats(int out_features, int in_features);
int lstep_pack_linear_tc(const float* weight /* [out,in] row major (torch) */, int out_features, int in_features,
                         float* packed /* lstep_packed_tc_floats() floats */, void* stream);
int lstep_pack_linear(const float* weight /* [out,in] row major (torch) */, const float* bias /* [out] or NULL */,
                      int out_features, int in_features, float* packed_w /* [in_pad][ldo] */,
                      float* packed_b /* [ldo] */, void* stream);

typedef struct lstep_pe_mlp {
  const float* w1; /* packed [rows(d+t)][ldo]  pe_mlp_1 / pe_neighbor_mlp_1 */
  const float* b1;
  const float* w2; /* packed [rows(d)][ldo]    pe_mlp_2 / pe_neighbor_mlp_2 */
  const float* b2;
  const float* ws; /* packed [rows(d)][ldo]    self_update_pe / self_update_neighbor_pe; NULL = no self term */
  const float* bs;
  const float* tw; /* [t] TimeEncoder frequencies (models/modules.py:20), fp32 */
  int d;
  int t;
  /* the same three weight matrices packed for the tensor-core kernel (lstep_pack_linear_tc: B-fragment
   * order, TF32 hi / lo split); all NULL = fp32 SIMT kernel only */
  const float* w1_tc;
  const float* w2_tc;
  const float* ws_tc;
} lstep_pe_mlp;

/* ------------------------------------------------------------------------------------------
 * a5 — TimeEncoder.forward (models/modules.py:27-39, frozen at models/LSTEP.py:50):
 *   out[i, j] = cos(dt[i] * w[j])   — the fp32 product rounded on its own (what Linear(1 -> t) with a zero bias
 * computes), then the accurate cosine the gather / update kernels use (time_feature() in csrc/common.cuh; all
 * three argument ranges: |x| < 2^14 Cody-Waite, < 2^32 fixed-point Payne-Hanek, beyond: general window).
 * In the step this is fused into the K2 kernels; the stand-alone entry point exists so that the encoder can be
 * pinned on its own against a float64 cosine.
 * ------------------------------------------------------------------------------------------ */
int lstep_time_features(const float* dt, int64_t n, const float* w, int t, float* out, void* stream);

/* ------------------------------------------------------------------------------------------
 * f2 — edge / time mixer of LSTEP.aggregated_node_embeddings (models/LSTEP.py:146-167), collapsed: edge_mlp_1 (Linear)
 * followed by edge_agg (Linear over the K axis) equals W1 (sum_k a_k C[i,k,:]) + (sum_k a_k) b1 + b_agg, so one pass
 * forms X[i] = sum_k a_k [ (nbr_k != 0) cos(fp32(t_i - t_k) tw) || edge_feats[eid_k] ]  (row pitch t + Fe; the lookup
 * of the K most recent neighbours and their edge ids happens inside). Rows >= n_valid are all-padding (zip truncation).
 * ------------------------------------------------------------------------------------------ */
int lstep_feature_aggregate(const lstep_csr* csr, const int64_t* q_node, const double* q_time, int64_t n_rows, int64_t n_valid,
                            int K, const float* edge_feats, int64_t n_edge_rows, int Fe, const float* tw, int t,
                            const float* agg_w /* [K] = edge_agg.weight */, float* X, uint32_t* err_flag, void* stream);

/* ------------------------------------------------------------------------------------------
 * a6 — neighbourhood PE aggregate (kernel K2, gather side) + MLP.
 * Replaces LSTEP.compute_neighborhood_pe (models/LSTEP.py:222-249) after the sampler call:
 *   S[i] = sum_k [ pe[nbr[i,k]] || mask_k * cos(fp32(q_time[i] - nbr_t[i,k]) * tw) ]
 *   out[i] = pe[q_node[i]] + tanh(Ws pe[q_node[i]] + bs + W2 relu(W1 S[i] + b1) + b2)
 * lstep_nbr_aggregate writes S only (training path: the MLP then runs under autograd);
 * lstep_nbr_aggregate_bwd scatters dS[:, :d] back into dpe (dpe[nbr[i,k]] += dS[i,:d]).
 * ------------------------------------------------------------------------------------------ */
int lstep_nbr_aggregate(const float* pe, int64_t pe_rows, const double* q_time, const int32_t* nbr,
                        const float* nbr_t, int64_t n_rows, int K, const float* tw, int d, int t, float* S,
                        void* stream);
/* Lookup + aggregate in one launch (the streaming step's form): row i looks up the K most recent neighbours of
 * (q_node[i], q_time[i]) itself, as lstep_sample_recent would, and writes S[i] (row pitch d + t). */
int lstep_nbr_lookup_aggregate(const lstep_csr* csr, const int64_t* q_node, const double* q_time, int64_t n_rows, int K,
                               const float* pe, int64_t pe_rows, const float* tw, int d, int t, float* S,
                               uint32_t* err_flag, void* stream);
int lstep_nbr_aggregate_bwd(const float* dS, const int32_t* nbr, int64_t n_rows, int K, int d, int t, float* dpe,
                            int64_t pe_rows, void* stream);
int lstep_neighborhood_pe(const float* pe, int64_t pe_rows, const int64_t* q_node, const double* q_time,
                          const int32_t* nbr, const float* nbr_t, int64_t n_rows, int K, const lstep_pe_mlp* mlp,
                          float* out, void* workspace, size_t workspace_bytes, void* stream);

/* out[i] = base[i] + tanh(Ws base[i] + bs + W2 relu(W1 A[i] + b1) + b2) for n_rows rows of A [n, d+t];
 * base[i] = pe[base_ids[i]]; result row i is written to out + i*out_stride, or, when out is NULL,
 * back into pe[base_ids[i]] (in place). Exposed for tests. */
int lstep_pe_mlp_apply(const float* A, const float* pe, const int64_t* base_ids, int64_t n_rows,
                       const lstep_pe_mlp* mlp, float* out, int64_t out_stride, float* pe_inplace, void* stream);

/* ------------------------------------------------------------------------------------------
 * a7 + a8 — PE update with ordered write-back (kernels K2 scatter side + K4).
 * Replaces LSTEP.update_pe (models/LSTEP.py:268-341), including its sampler call, on the
 * caller's pe[pe_rows, d] table, in place:
 *   phase A  every batch node gets the sum over its batch edges of [pe[other endpoint] || tf]
 *            (source-side contributions first, then destination-side, edge order) -> MLP with
 *            self term -> pe[ids] written;
 *   pe[0] = 0;
 *   phase B  most-recent-K lookup for (ids[i], times[i]), i < min(n_ids, n_edges) (Q1/Q1b);
 *            every sampled neighbour u accumulates [pe[ids[i]] || tf] from the phase-A table;
 *            all gathers complete before any row is written; MLP without self term (Q3);
 *            pe[u] written for every distinct u, including u = 0 when any slot was padding.
 * current_time is rounded to fp32 first (torch.Tensor([current_time]), Q4).
 * ------------------------------------------------------------------------------------------ */
size_t lstep_update_pe_workspace_bytes(int64_t n_ids, int64_t n_edges, int K, int d, int t, int64_t pe_rows);
int lstep_update_pe(float* pe, int64_t pe_rows, const lstep_csr* csr, const int64_t* ids, int64_t n_ids,
                    const int64_t* src, const int64_t* dst, const double* times, int64_t n_edges,
                    double current_time, int K, const lstep_pe_mlp* mlp, void* workspace, size_t workspace_bytes,
                    uint32_t* err_flag, void* stream);
/* The same update as separate phases, for a node-id sharded table (l-step_b200/shard.py): rank r owns
 * the rows v with v % G == r, runs phase A for the batch nodes it owns, then the aggregation half of
 * phase B for the (node, time) pairs it owns (csr_ids index the rank's local CSR, row_ids the table),
 * ships the partial aggregate rows to the owners of the destinations, which combine them
 * (lstep_segment_sum_rows, fixed order) and apply the MLP (lstep_pe_mlp_apply without self term).
 * lstep_update_pe_workspace_layout reports where phase B left its results inside the workspace:
 * offsets[0] counters int32[8] (0: #distinct non-zero destinations M, 1: padding seen), offsets[1] U
 * int64[M (+1)], offsets[2] A float[M (+1)][lda], offsets[3] = lda. */
int lstep_update_pe_phase_a(float* pe, int64_t pe_rows, const int64_t* ids, int64_t n_ids, const int64_t* src,
                            const int64_t* dst, const double* times, int64_t n_edges, double current_time, int K,
                            const lstep_pe_mlp* mlp, void* workspace, size_t workspace_bytes, void* stream);
int lstep_update_pe_phase_b_partial(float* pe, int64_t pe_rows, const lstep_csr* csr, const int64_t* csr_ids,
                                    const int64_t* row_ids, int64_t n_ids, const double* q_times, int64_t n_valid,
                                    int64_t n_edges_layout, double current_time, int K, const lstep_pe_mlp* mlp,
                                    void* workspace, size_t workspace_bytes, uint32_t* err_flag, void* stream);
int lstep_update_pe_workspace_layout(int64_t n_ids, int64_t n_edges, int K, int d, int t, int64_t pe_rows, int64_t* offsets);
int lstep_segment_sum_rows(const float* rows, int64_t ld, const int64_t* seg_off, int64_t n_seg, int width, float* out,
                           int64_t ldo, void* stream);
int lstep_dft_filter_scatter(const float* hist, int64_t node_stride, int64_t time_stride, int s0, int ring, int Th, int d,
                             const int64_t* ids, const int64_t* out_ids, int64_t n_ids, const float* G, float* out,
                             int64_t out_stride, void* stream);
int lstep_ring_copy_rows(float* ring, float* cur, int64_t ring_rows, int T, int d, int slot, int64_t row_mul,
                         int64_t row_add, int to_ring, void* stream);

/* The update keeps a per-node int32 scratch map inside the workspace that must be zero on
 * entry and is zero again on exit; call once after allocating the workspace. */
int lstep_update_pe_workspace_init(void* workspace, size_t workspace_bytes, int64_t pe_rows, void* stream);

/* ------------------------------------------------------------------------------------------
 * f1 — streaming PE step on device-resident state (an addition to the reference API; the loops'
 * trim / clone / cat of the history, train_LSTEP_link_prediction.py:205,224-230,301-306 and
 * evaluate_model_utils.py:57-63,131-135, become one ring-slot write).
 *   ring  [V1][T][d] node-major history ring; logical step j lives in slot (head + j) % T, j < len
 *   cur   [V1][d]    current table; equals the newest ring slot between steps (lstep_ring_load
 *                    initialises it after an import)
 * lstep_pe_step runs, for the batch of edges [lo, lo + n_edges) of the resident stream:
 *   the DFT filter of the batch nodes `ids` (G = collapsed filter for this step's mask) scattered into
 *   cur; compute_neighborhood_pe for n_queries id sets (host array of device pointers, each
 *   [n_edges], queried at the batch's edge times) -> nbr_out [n_queries][n_edges][d]; update_pe on
 *   cur; cur -> ring[:, append_slot].
 * The workspace starts with the update_pe workspace: initialise it with
 * lstep_update_pe_workspace_init.
 * ------------------------------------------------------------------------------------------ */
typedef struct lstep_pe_stream {
  const int64_t* src; /* [E] whole edge stream, resident */
  const int64_t* dst;
  const double* t;
  float* ring;
  float* cur;
  int64_t V1; /* live rows: every bound check and every full-table pass covers [0, V1) */
  int T;
  int d;
  int64_t row_cap; /* rows allocated in ring / cur (>= V1) and covered by the update workspace's per-node maps; 0 = V1 */
} lstep_pe_stream;

size_t lstep_pe_step_workspace_bytes(int64_t max_ids, int64_t max_edges, int n_queries, int K, int d, int t, int64_t V1);
int lstep_ring_load(const float* ring, float* cur, int64_t V1, int T, int d, int slot, void* stream);
/* New nodes [r0, r1) of a stream that grows its node set: writes rows[(v - r0) * rows_stride .. + d) (rows_stride 0: one
 * broadcast row [d]; device memory) to table row v (table != NULL), to all T slots of ring row v (ring != NULL; node-major,
 * one contiguous T*d block per node) and, when v % world == rank, to change-log base row (v - rank) / world (base != NULL).
 * d % 4 == 0 and 16-byte aligned pointers. Enqueued on `stream` behind the steps already there, which touch only rows
 * below r0: a node no edge has touched holds its initial row in the table, in every ring slot and as its base row. */
int lstep_pe_rows_init(float* table, float* ring, int T, int d, float* base, int64_t world, int64_t rank, int64_t r0, int64_t r1,
                       const float* rows, int64_t rows_stride, void* stream);
int lstep_pe_step(const lstep_pe_stream* s, const lstep_csr* csr, int64_t lo, int64_t n_edges, const int64_t* ids,
                  int64_t n_ids, double current_time, int head, int len, int append_slot, const float* G,
                  const int64_t* const* query_ids_host, int n_queries, float* nbr_out, int K,
                  const lstep_pe_mlp* mlp_nbr, const lstep_pe_mlp* mlp_upd, void* workspace, size_t workspace_bytes,
                  uint32_t* err_flag, void* stream);

/* n_steps consecutive batches of the resident stream in one call (steady state, ring full): host arrays lo / n_edges /
 * ids_off[n_steps+1] / tmax / q_off describe the batches, `ids` (device) holds all their sorted unique node ids. Outputs of
 * step i at nbr_out + i * out_step_stride. *head_io advances by one slot per step. */
int lstep_pe_steps(const lstep_pe_stream* s, const lstep_csr* csr, int64_t n_steps, const int64_t* lo_host,
                   const int64_t* n_edges_host, const int64_t* ids, const int64_t* ids_off_host, const double* tmax_host,
                   int* head_io, int* len_io, const float* G, const int64_t* const* query_ids_host, const int64_t* q_off_host,
                   int n_queries, float* nbr_out, int64_t out_step_stride, int K, const lstep_pe_mlp* mlp_nbr,
                   const lstep_pe_mlp* mlp_upd, void* workspace, size_t workspace_bytes, uint32_t* err_flag, void* stream);

/* One rank's share of a step on a node-id sharded group with a replicated table and CSR and a sharded history ring: lstep_pe_step
 * without the DFT filter and the ring append (both owner-local, done by the caller around an all-gather of the filtered rows);
 * the a6 query sets cover edges [q_off, q_off + q_rows) of the batch, query_ids_host[c] pointing at the first of those ids. */
int lstep_pe_step_sharded(const lstep_pe_stream* s, const lstep_csr* csr, int64_t lo, int64_t n_edges, const int64_t* ids,
                          int64_t n_ids, double current_time, const int64_t* const* query_ids_host, int n_queries, int64_t q_off,
                          int64_t q_rows, float* nbr_out, int K, const lstep_pe_mlp* mlp_nbr, const lstep_pe_mlp* mlp_upd,
                          void* workspace, size_t workspace_bytes, uint32_t* err_flag, void* stream);

/* ------------------------------------------------------------------------------------------
 * Change-log PE history (csrc/changelog.cu): the history [V1, T, d] of the loops (a4 / f1) stored as base rows + the rows
 * every step changed, instead of T full snapshots — V1 + T * (rows changed per step) rows: 7.8 GB instead of 688 GB for
 * the 10 M-node graph at T = 100, and 9 MB instead of 13.8 GB written per step. x[v, f] = the row of the latest event of v
 * at a window index <= f, else base[v]: the same function of time, so the collapsed DFT filter becomes
 * out[n] = sum_versions (sum of G over the span a version covers) * version row.
 *   base     [rows][d]        value at the window's oldest step            ev_cnt  [T]     events per window slot
 *   ev_node  [T][cap]         node of an event                             ev_hash [T][H]  open addressing: node << 32 | index
 *   ev_row   [T][cap][d]      its row                                      ev_mask [rows][4] bit s: the node has an event in slot s
 * All zero-initialised except ev_hash (all ones). H = power of two >= 2 * cap; T <= 128. Node-id sharded groups: a rank
 * holds the nodes v with v % row_mul == row_add at local row (v - row_add) / row_mul (1, 0: everything).
 * ------------------------------------------------------------------------------------------ */
typedef struct lstep_changelog {
  float* base;
  int32_t* ev_node;
  float* ev_row;
  int32_t* ev_cnt;
  unsigned long long* ev_hash;
  uint32_t* ev_mask;
  int64_t rows;
  int T, cap, H, d;
  int64_t row_mul, row_add;
} lstep_changelog;

/* out[out_ids ? out_ids[i] : i] = filtered history of node ids[i] over the window (head = slot of its oldest step, len steps) */
int lstep_changelog_filter(const lstep_changelog* cl, int head, int len, const int64_t* ids, int64_t n_ids, const float* G,
                           float* out, int64_t out_stride, const int64_t* out_ids, void* stream);
/* retire (optional) the events of `slot` into the base rows, then record table[v] for v in U[0 .. min(n_u, *n_u_dev)) and for
 * the ids whose stamp_map entry differs from `stamp` (U == NULL: every id) as the slot's new events */
int lstep_changelog_append(const lstep_changelog* cl, int slot, int retire, const float* table, const int64_t* U,
                           const int32_t* n_u_dev, int64_t n_u, const int64_t* ids, int64_t n_ids, const int32_t* stamp_map, int stamp,
                           int with_row0 /* also the padding row 0, which every update_pe call zeroes */, uint32_t* err_flag, void* stream);
/* lstep_pe_step on a change-log history (s->ring unused). phase 0: filter + step + append; 1: filter only; 2: step + append
 * (sharded groups filter with lstep_changelog_filter, all-gather, scatter, then call phase 2). q_off / q_rows as in
 * lstep_pe_step_sharded (q_rows < 0: all edges). */
int lstep_pe_step_changelog(const lstep_pe_stream* s, const lstep_changelog* cl, const lstep_csr* csr, int64_t lo, int64_t n_edges,
                            const int64_t* ids, int64_t n_ids, double current_time, int head, int len, const float* G,
                            const int64_t* const* query_ids_host, int n_queries, int64_t q_off, int64_t q_rows, float* nbr_out, int K,
                            const lstep_pe_mlp* mlp_nbr, const lstep_pe_mlp* mlp_upd, void* workspace, size_t workspace_bytes,
                            uint32_t* err_flag, void* stream, int phase);

/* ------------------------------------------------------------------------------------------
 * Peer group: the scale-out step over NVLink peer memory (csrc/peer.cu; BASELINE config 5, SURVEY §8(e)).
 * One process per GPU. Every rank keeps a REPLICA of the current PE table and of the temporal CSR and OWNS the nodes
 * v with v % world == rank: their PE history (change log), their share of every phase of the step, and the duty to
 * make every row it changes available. A step on rank r:
 *     filter      DFT filter of the owned batch nodes into the local table and, at the node's position in the batch's id list,
 *                 into every other rank's filt buffer
 *     barrier 1   (flag exchange through peer memory, no host, no NCCL) + refresh of the replica in the same launch: the rows
 *                 the previous step changed on the other ranks (this rank's inbox) and the other owners' filtered rows
 *     gather      a6 for this rank's 1/world share of the query rows || a7 edge aggregate of the OWNED batch nodes
 *     MLP pair    neighbourhood MLP of the share || phase-A MLP of the owned batch nodes; the phase-A rows are stored
 *                 into every rank's new_rows buffer at the node's position in the batch's id list
 *     barrier 2
 *     push        most-recent-K lookup of ALL batch nodes (replicated, cheap), accumulation only for the OWNED
 *                 destinations (u % world == rank); the owned batch nodes' phase-A rows are applied to the local table
 *     MLP (B)     over the owned destinations
 *     append      the owned changed rows (owned batch nodes + owned destinations + row 0 on rank 0) become events of
 *                 the change log
 *     publish     ... and are copied, as one contiguous block, into every other rank's inbox.
 * Nothing a rank reads between two barriers is written by another rank in that interval (csrc/peer.cu states the
 * argument), so the replicas agree after every refresh and the results are those of the single-GPU step, bit for bit
 * (phase B's sums are exact fixed point, hence independent of which rank adds them).
 * Memory that peers write (inbox, filt, new_rows, flags) is allocated with lstep_ipc_alloc (cudaMalloc) and shared
 * with the CUDA IPC handles of lstep_ipc_export / lstep_ipc_open; in a single process (tests) plain device pointers of
 * several rank states can be used instead.
 * ------------------------------------------------------------------------------------------ */
#define LSTEP_MAX_PEERS 16
typedef struct lstep_peer_group {
  int rank, world;
  float* table[LSTEP_MAX_PEERS];     /* table[rank] = this rank's table replica (== s->cur); the other entries are unused */
  /* WRITTEN by the other ranks — small, fixed regions only (scattered accesses to a multi-GB peer mapping, and reads of peer
   * memory, are slow: profiles/r02_peer_bw.txt, profiles/r02_scaleout_history.md): */
  float* new_rows[LSTEP_MAX_PEERS];  /* phase-A row buffer of every rank, [max batch nodes, d], row p = the node at position p of
                                        the batch's id list, written by its owner */
  float* filt[LSTEP_MAX_PEERS];      /* filtered-row buffer of every rank, same indexing, written by the owners' filter kernels */
  void* inbox[LSTEP_MAX_PEERS];      /* inbox of every rank, lstep_peer_inbox_bytes(world, cap, d) bytes: one block per SOURCE rank =
                                        { int32 count, pad[3]; int32 node[cap]; float row[cap][d] } — the rows that rank changed
                                        in the previous step, copied there by its publish kernel */
  uint32_t* flags[LSTEP_MAX_PEERS];  /* flag block of every rank, uint32[LSTEP_MAX_PEERS]: flags[g][r] = last barrier epoch
                                        rank r has announced to rank g (zero-initialised, epochs start at 1) */
  int64_t cap;                       /* rows per inbox block (>= the change logs' event capacity; the same on every rank) */
} lstep_peer_group;
size_t lstep_peer_inbox_bytes(int world, int64_t cap, int d);
int lstep_ipc_alloc(size_t bytes, void** ptr);                         /* cudaMalloc + zero fill */
int lstep_ipc_free(void* ptr);
int lstep_ipc_export(void* ptr, unsigned char handle_out[64]);         /* cudaIpcGetMemHandle */
int lstep_ipc_open(const unsigned char handle[64], void** ptr);        /* cudaIpcOpenMemHandle (enables peer access) */
int lstep_ipc_close(void* ptr);
/* announce `epoch` to every rank / wait until every rank has announced it (bounded: after ~timeout_ms the wait gives up
 * and raises LSTEP_FLAG_PEER_TIMEOUT in *err_flag instead of hanging the device) */
int lstep_peer_signal(const lstep_peer_group* g, uint32_t epoch, void* stream);
int lstep_peer_wait(const lstep_peer_group* g, uint32_t epoch, int timeout_ms, uint32_t* err_flag, void* stream);
/* announce `epoch`, wait for every rank, then apply the inbox (the rows the last step changed on the other ranks): afterwards, in
 * stream order, this rank's replica equals every other one (what a caller does before it reads the table after the last step) */
int lstep_peer_sync_tables(const lstep_peer_group* g, uint32_t epoch, int timeout_ms, uint32_t* err_flag, int d, int64_t V1, void* stream);
/* dst[g][dst_rows[i]][0..d) = src[i][0..d) for every rank g whose bit is set in rank_mask (dst_rows NULL: row i); which = 0: the
 * table replicas, 1: the new_rows buffers. The building block of the step's row publication (also used to measure the
 * peer-store bandwidth, profiles/peer_bw.py). */
int lstep_peer_rows_bcast(const float* src, int64_t n_rows, int d, const int64_t* dst_rows, const lstep_peer_group* grp, int which,
                          uint32_t rank_mask, void* stream);
/* One step of this rank (see above). ids = the batch's sorted unique node ids (all of them, replicated); ids_mine = the owned
 * ones, pos_mine[i] = index of ids_mine[i] in ids. The a6 query sets cover edges [q_off, q_off + q_rows) of the batch,
 * query_ids_host[c] pointing at the first of those ids; outputs [n_queries, q_rows, d]. epoch_base: barrier 1 uses
 * epoch_base + 1, barrier 2 epoch_base + 2 (the caller advances it by 2 per step, identically on every rank).
 * phases: bit 0 = filter + signal 1; bit 1 = wait 1 .. signal 2; bit 2 = wait 2 .. append (7 = the whole step; a
 * single-process group of several rank states runs each bit for every rank before the next). */
int lstep_pe_step_peer(const lstep_pe_stream* s, const lstep_changelog* cl, const lstep_csr* csr, const lstep_peer_group* grp,
                       int64_t lo, int64_t n_edges, const int64_t* ids, int64_t n_ids, const int64_t* ids_mine,
                       const int64_t* pos_mine, int64_t n_mine, double current_time, int head, int len, const float* G,
                       const int64_t* const* query_ids_host, int n_queries, int64_t q_off, int64_t q_rows, float* nbr_out, int K,
                       const lstep_pe_mlp* mlp_nbr, const lstep_pe_mlp* mlp_upd, void* workspace, size_t workspace_bytes,
                       uint32_t* err_flag, uint32_t epoch_base, int timeout_ms, int phases, void* stream);
/* A run of consecutive steady-state steps (len == T) in one call: the host only pays the launches. Arrays indexed by step i:
 * lo / n_edges / tmax; ids + ids_off[i] .. ids_off[i+1]; ids_mine / pos_mine + mine_off[i] .. mine_off[i+1]; query set c of
 * step i = query_ids_host[c] + q_base[i] (n_edges[i] ids; this rank's share of them is taken here:
 * [rank * n / world, (rank+1) * n / world)); outputs of step i at nbr_out + i * out_step_stride floats. *head_io and
 * *epoch_io are advanced. */
int lstep_pe_steps_peer(const lstep_pe_stream* s, const lstep_changelog* cl, const lstep_csr* csr, const lstep_peer_group* grp,
                        int64_t n_steps, const int64_t* lo_host, const int64_t* n_edges_host, const double* tmax_host,
                        const int64_t* ids, const int64_t* ids_off_host, const int64_t* ids_mine, const int64_t* pos_mine,
                        const int64_t* mine_off_host, int* head_io, const float* G, const int64_t* const* query_ids_host,
                        const int64_t* q_base_host, int n_queries, float* nbr_out, int64_t out_step_stride, int K,
                        const lstep_pe_mlp* mlp_nbr, const lstep_pe_mlp* mlp_upd, void* workspace, size_t workspace_bytes,
                        uint32_t* err_flag, uint32_t* epoch_io, int timeout_ms, void* stream);

/* ------------------------------------------------------------------------------------------
 * Host-fed streaming step (csrc/host_step.cu): what a loop that holds the batch as HOST arrays calls
 * per batch (the hand-over train_LSTEP_link_prediction.py:204-313 / evaluate_model_utils.py:38-142 do
 * with numpy arrays and .cpu() reads). A stepper owns `slots` pinned input/result slots and their
 * device mirrors (allocated once by _create: the only entry points that allocate).
 * lstep_pe_step_host packs (src, dst, t, sorted unique batch nodes, the query id sets) into a pinned
 * slot, moves them with one async copy, enqueues lstep_pe_step's kernels on the staged batch
 * (current_time = max t, LSTEP.update_pe's caller passes that), reduces nbr_out to per-query row sums
 * [n_queries][n_edges] and copies them to the slot's pinned result, all on `stream`, without
 * synchronising; *ticket identifies the step. ids_host may be NULL (computed here by sort + unique).
 * nbr_out may be NULL (the stepper's own [n_queries][n_edges][d] buffer is used).
 * lstep_host_step_result waits for the ticket's event and returns the pinned result (valid until the
 * slot is reused `slots` steps later).
 * ------------------------------------------------------------------------------------------ */
typedef struct lstep_host_stepper lstep_host_stepper;
int lstep_host_stepper_create(int slots, int64_t max_edges, int max_queries, int d, lstep_host_stepper** out);
void lstep_host_stepper_destroy(lstep_host_stepper* h);
int lstep_pe_step_host(lstep_host_stepper* h, const lstep_pe_stream* s, const lstep_csr* csr, int64_t n_edges,
                       const int64_t* src_host, const int64_t* dst_host, const double* t_host, const int64_t* ids_host,
                       int64_t n_ids, int head, int len, int append_slot, const float* G,
                       const int64_t* const* query_ids_host_arrays, int n_queries, float* nbr_out, int K,
                       const lstep_pe_mlp* mlp_nbr, const lstep_pe_mlp* mlp_upd, void* workspace, size_t workspace_bytes,
                       uint32_t* err_flag, void* stream, int64_t* ticket);
int lstep_host_step_result(lstep_host_stepper* h, int64_t ticket, const float** result_host, int64_t* n_floats);
/* Arms the stepper to grow a growable CSR (see lstep_csr_ingest; `fill` its fill array, the csr being the one each call
 * passes): every later lstep_pe_step_host / lstep_pe_steps_host call first appends its batch, with edge ids next_eid + i,
 * then runs its step on the grown CSR. Before anything is enqueued a call rejects a batch whose times are not finite, decrease,
 * or start before last_t (LSTEP_ERR_INVALID_ARG), or whose ids or edge ids fall outside the CSR's rows or int32
 * (LSTEP_ERR_ID_RANGE). The append runs on the copy-in path, between the batch's copy-in and its hand-over to the
 * compute stream, on a stream of the highest priority (created by the first arming). The first append after arming, or after the CSR's arrays change, also waits for the work enqueued on
 * the compute stream so far (a relayout, or appends made there). The append of batch b+1 is not ordered after work the caller
 * enqueues on the compute stream after step b: a lookup there is exact at times <= the times of batch b only. fill = NULL
 * disarms. */
int lstep_host_stepper_set_ingest(lstep_host_stepper* h, int32_t* fill, int64_t next_eid, double last_t);
void lstep_host_stepper_bytes(const lstep_host_stepper* h, uint64_t* h2d_bytes, uint64_t* d2h_bytes);
/* lstep_pe_step_host on a change-log history (lstep_pe_step_changelog; cl->row_mul == 1): the same staging, host checks,
 * optional append (lstep_host_stepper_set_ingest) and result path, around the change-log step: filter of the batch nodes into
 * the table, the step's kernels, retire + append. Its events go to slot (head + len) % T while the log fills, to `head` (after
 * retiring it) once len == T. s->src / s->dst / s->t are never read, so a descriptor over an empty edge stream serves it. */
int lstep_pe_step_changelog_host(lstep_host_stepper* h, const lstep_pe_stream* s, const lstep_changelog* cl, const lstep_csr* csr,
                                 int64_t n_edges, const int64_t* src_host, const int64_t* dst_host, const double* t_host,
                                 const int64_t* ids_host, int64_t n_ids, int head, int len, const float* G,
                                 const int64_t* const* query_ids_host_arrays, int n_queries, float* nbr_out, int K,
                                 const lstep_pe_mlp* mlp_nbr, const lstep_pe_mlp* mlp_upd, void* workspace, size_t workspace_bytes,
                                 uint32_t* err_flag, void* stream, int64_t* ticket);
/* A run of consecutive batches in one call (an evaluation split, evaluate_model_utils.py:38-142): the loop over
 * lstep_pe_step_host / lstep_host_step_result is done natively, results read one step behind. Full history ring only
 * (*len_io == T, one collapsed filter G); batch b = edges [b*batch_size, min((b+1)*batch_size, n_total)) of the host
 * arrays; results_host [n_batches][n_queries][batch_size]; *head_io is advanced. Synchronous on return.
 * On an error in batch k (e.g. LSTEP_ERR_ID_RANGE) batches [0, k) HAVE been applied: *head_io and *n_done_out (may be
 * NULL) report the ring position reached and the number of batches applied, so the caller's state stays consistent. */
int lstep_pe_steps_host(lstep_host_stepper* h, const lstep_pe_stream* s, const lstep_csr* csr, int64_t n_total,
                        int64_t batch_size, const int64_t* src_host, const int64_t* dst_host, const double* t_host,
                        const int64_t* const* query_ids_host_arrays, int n_queries, int* head_io, int* len_io,
                        const float* G, int K, const lstep_pe_mlp* mlp_nbr, const lstep_pe_mlp* mlp_upd, void* workspace,
                        size_t workspace_bytes, uint32_t* err_flag, void* stream, float* results_host, int64_t* n_done_out);
/* lstep_pe_steps_host on a change-log history: every batch through lstep_pe_step_changelog_host. Full log only (*len_io == T,
 * else LSTEP_ERR_UNSUPPORTED); results one step behind; on an error in batch k batches [0, k) stay applied and *head_io /
 * *n_done_out report the position reached. */
int lstep_pe_steps_changelog_host(lstep_host_stepper* h, const lstep_pe_stream* s, const lstep_changelog* cl, const lstep_csr* csr,
                                  int64_t n_total, int64_t batch_size, const int64_t* src_host, const int64_t* dst_host,
                                  const double* t_host, const int64_t* const* query_ids_host_arrays, int n_queries, int* head_io,
                                  int* len_io, const float* G, int K, const lstep_pe_mlp* mlp_nbr, const lstep_pe_mlp* mlp_upd,
                                  void* workspace, size_t workspace_bytes, uint32_t* err_flag, void* stream, float* results_host,
                                  int64_t* n_done_out);
/* One rank's peer-group step (lstep_pe_step_peer) fed from HOST arrays: the same staging, host checks, optional append into the
 * rank's own CSR replica (lstep_host_stepper_set_ingest) and result path as lstep_pe_step_host. The rank's owned ids of the batch
 * and their positions are derived on the device from the staged ids, on the copy-in path. s->src / s->dst / s->t are never read.
 * phases as in lstep_pe_step_peer; a single-process group issues each bit for every rank before the next:
 *   - the call with bit 0 stages the batch and keeps it as the stepper's pending batch;
 *   - later calls of the same step (bits 1, 2) use the pending batch: their n_edges, host arrays and n_queries are not read
 *     (may be 0 / NULL), and nbr_out must be the one the staging call passed;
 *   - the call with bit 2 finishes the step: row sums of this rank's share [n_queries][q_rows] (q_off = rank * n / world,
 *     q_rows = (rank + 1) * n / world - q_off) into the pinned result, and *ticket.
 * LSTEP_ERR_INVALID_ARG for a later phase with no pending batch and for staging while a batch is pending. Every check comes
 * before anything is enqueued and depends only on the batch and the arguments, so the ranks of a group given the same batch
 * all accept or all reject it. n_edges must not exceed the batch size the group's new_rows / filt buffers are sized for
 * (2 * n_edges rows). */
int lstep_pe_step_peer_host(lstep_host_stepper* h, const lstep_pe_stream* s, const lstep_changelog* cl, const lstep_csr* csr,
                            const lstep_peer_group* grp, int64_t n_edges, const int64_t* src_host, const int64_t* dst_host,
                            const double* t_host, const int64_t* ids_host, int64_t n_ids, int head, int len, const float* G,
                            const int64_t* const* query_ids_host_arrays, int n_queries, float* nbr_out, int K,
                            const lstep_pe_mlp* mlp_nbr, const lstep_pe_mlp* mlp_upd, void* workspace, size_t workspace_bytes,
                            uint32_t* err_flag, uint32_t epoch_base, int timeout_ms, int phases, void* stream, int64_t* ticket);
/* lstep_pe_steps_host for one rank of a peer group: every batch through lstep_pe_step_peer_host (phases 7), full log only
 * (*len_io == T, else LSTEP_ERR_UNSUPPORTED), results read one step behind into results_host [n_batches][n_queries][batch_size]
 * (the first q_rows of each row: this rank's share), each step's publication on a side stream as in lstep_pe_steps_peer.
 * *head_io and *epoch_io are advanced; on an error in batch k batches [0, k) stay applied and *head_io / *epoch_io /
 * *n_done_out report the position reached. */
int lstep_pe_steps_peer_host(lstep_host_stepper* h, const lstep_pe_stream* s, const lstep_changelog* cl, const lstep_csr* csr,
                             const lstep_peer_group* grp, int64_t n_total, int64_t batch_size, const int64_t* src_host,
                             const int64_t* dst_host, const double* t_host, const int64_t* const* query_ids_host_arrays, int n_queries,
                             int* head_io, int* len_io, const float* G, int K, const lstep_pe_mlp* mlp_nbr, const lstep_pe_mlp* mlp_upd,
                             void* workspace, size_t workspace_bytes, uint32_t* err_flag, uint32_t* epoch_io, int timeout_ms,
                             void* stream, float* results_host, int64_t* n_done_out);

/* ------------------------------------------------------------------------------------------
 * Measurement / A-B plumbing (no reference counterpart).
 * lstep_set_option: switches of the launch paths ("pdl", "phaseb_push", "gather_pipe", "mlp_umma", "mlp_umma_min_rows",
 * "profile"), each selecting a shipped path or its reference on the same inputs; defaults are the shipped paths, the LSTEP_*
 * environment variables of DESIGN.md set them once at first use. None changes results beyond fp32 summation order.
 * An unknown name returns LSTEP_ERR_INVALID_ARG.
 * lstep_step_profile(1): every streaming step records CUDA events around its kernels; lstep_step_profile_read returns
 * the six durations (ms) of the last step: DFT filter, fused gather, paired MLP, phase-B push, phase-B MLP, ring append.
 * ------------------------------------------------------------------------------------------ */
int lstep_set_option(const char* name, int value);
int lstep_get_option(const char* name, int* value);
int lstep_step_profile(int enable);
int lstep_step_profile_read(float* ms6);
/* every mark of the last profiled step, peer-group marks included (n >= 9): DFT filter (+ barrier-1 announcement), wait on
 * barrier 1, fused gather, paired MLP, phase-A row broadcast (+ barrier-2 announcement), wait on barrier 2, phase-B push,
 * phase-B MLP, append; -1 where no mark was recorded */
int lstep_step_profile_read_all(float* ms, int n);

#ifdef __cplusplus
}
#endif
#endif /* LSTEP_B200_H */
