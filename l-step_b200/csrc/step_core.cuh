// Internal interface of the streaming step's core (csrc/step.cu), shared with the host-fed stepper and the change-log history.
#pragma once
#include "common.cuh"

namespace lstep {

// Rows the update workspace's per-node maps cover: the stream's row capacity, so that the workspace layout stays put while
// the live row count V1 grows inside it (lstep_pe_stream.row_cap, 0 = V1).
inline int64_t pe_ws_rows(const lstep_pe_stream* s) { return s->row_cap > s->V1 ? s->row_cap : s->V1; }

// Owner-computes step of a peer group (csrc/peer.cu): phase A runs for the OWNED batch nodes only and its rows are stored
// into every rank's new_rows buffer; phase B runs for the owned destinations only. `phases` bit 1: everything up to the
// announcement of barrier 2; bit 2: from the wait on barrier 2 on (a single-process group runs bit 1 of every rank first).
struct PeerPlan {
  const lstep_peer_group* grp = nullptr;
  const int64_t* ids_mine = nullptr;  // owned batch nodes (ascending)
  const int64_t* pos_mine = nullptr;  // their positions in the batch's id list
  int64_t n_mine = 0;
  uint32_t epoch2 = 0;
  int timeout_ms = 2000;
  int phases = 6;
};
// Variations of the step for callers that own the history themselves (node-id sharded groups, the change-log history): the DFT
// filter and the ring append are then done by the caller, and the a6 queries may cover only a share [q_off, q_off + q_rows)
// of the batch's edges. stamp_out receives the step's stamp (the value the push kernel wrote into the per-node stamp map
// for every row phase B changed).
struct StepOpts {
  bool skip_dft = false, skip_append = false;
  int64_t q_off = 0, q_rows = -1;  // -1: all n_edges
  int* stamp_out = nullptr;
  const PeerPlan* peer = nullptr;
};
// csrc/peer.cu
int peer_rows_bcast(const float* src, int64_t n_rows, int d, const int64_t* dst_rows, const lstep_peer_group* grp, int which, cudaStream_t st);
int peer_signal(const lstep_peer_group* g, uint32_t epoch, cudaStream_t st);
int peer_wait(const lstep_peer_group* g, uint32_t epoch, int timeout_ms, uint32_t* err_flag, cudaStream_t st, bool announce = false);
// Side stream of a native multi-step peer call: the publication of a step's rows runs next to the NEXT step's filter (neither
// touches what the other writes); the next barrier-1 launch waits for it. open creates the stream and events; close makes the
// caller's stream wait for a pending publication and releases them.
struct SideLane {
  cudaStream_t stream = nullptr;
  cudaEvent_t appended = nullptr, published = nullptr;
  bool pending = false;  // a publication has been enqueued and not yet waited for
};
int side_lane_open(SideLane* lane);
void side_lane_close(SideLane* lane, cudaStream_t st);
// The peer step's checks of everything but the batch (callers make them before they enqueue anything), and the step itself on
// explicit batch pointers (src / dst / tq: n_edges device entries; s->src / s->dst / s->t are never read). q_off / q_rows: this
// rank's share of the batch's edges for the a6 queries, query_ids[c] pointing at the first of them.
int peer_step_check(const lstep_pe_stream* s, const lstep_changelog* cl, const lstep_csr* csr, const lstep_peer_group* grp, int64_t n_edges,
                    int head, int len, const lstep_pe_mlp* mlp_nbr, const lstep_pe_mlp* mlp_upd, int phases, int64_t q_rows);
int peer_step_core(const lstep_pe_stream* s, const lstep_changelog* cl, const lstep_csr* csr, const lstep_peer_group* grp, const int64_t* src,
                   const int64_t* dst, const double* tq, int64_t n_edges, const int64_t* ids, int64_t n_ids, const int64_t* ids_mine,
                   const int64_t* pos_mine, int64_t n_mine, double current_time, int head, int len, const float* G,
                   const int64_t* const* query_ids, int n_queries, int64_t q_off, int64_t q_rows, float* nbr_out, int K,
                   const lstep_pe_mlp* mlp_nbr, const lstep_pe_mlp* mlp_upd, void* workspace, size_t workspace_bytes, uint32_t* err_flag,
                   uint32_t epoch_base, int timeout_ms, int phases, void* stream, SideLane* side);
// A rank's owned plan of a batch on the device: ids_mine = the ids[0 .. n_ids) with v % world == rank, in order, and pos_mine =
// their positions in ids (one CTA; an ordered compaction). The host-fed peer step runs it on its copy-in stream.
int peer_plan_mine(const int64_t* ids, int64_t n_ids, int world, int rank, int64_t* ids_mine, int64_t* pos_mine, cudaStream_t st);

int pe_step_core_ex(const lstep_pe_stream* s, const lstep_csr* csr, const int64_t* src, const int64_t* dst, const double* tq,
                    int64_t n_edges, const int64_t* ids, int64_t n_ids, double current_time, int head, int len, int append_slot,
                    const float* G, const int64_t* const* query_ids_host, int n_queries, float* nbr_out, int K,
                    const lstep_pe_mlp* mlp_nbr, const lstep_pe_mlp* mlp_upd, void* workspace, size_t workspace_bytes,
                    uint32_t* err_flag, void* stream, const StepOpts& opt);
int pe_step_core(const lstep_pe_stream* s, const lstep_csr* csr, const int64_t* src, const int64_t* dst, const double* tq,
                 int64_t n_edges, const int64_t* ids, int64_t n_ids, double current_time, int head, int len, int append_slot,
                 const float* G, const int64_t* const* query_ids_host, int n_queries, float* nbr_out, int K,
                 const lstep_pe_mlp* mlp_nbr, const lstep_pe_mlp* mlp_upd, void* workspace, size_t workspace_bytes,
                 uint32_t* err_flag, void* stream);
// lists phase B leaves in an update workspace: U (distinct destinations), their count (device), the per-node stamp map
void update_ws_phase_b_lists(void* workspace, int64_t n_ids, int64_t n_edges, int K, int d, int t, int64_t pe_rows, const int64_t** U,
                             const int32_t** n_dest_dev, const int32_t** stamp_map);
bool update_push_available(const lstep_pe_mlp* mlp);
// csrc/changelog.cu: the change-log step on explicit batch pointers (never reads s->src / s->dst / s->t), and its checks of
// everything but the batch, which callers make before they enqueue anything
int changelog_step_check(const lstep_pe_stream* s, const lstep_changelog* cl, int head, int len, const lstep_pe_mlp* mlp_upd);
int changelog_step_core(const lstep_pe_stream* s, const lstep_changelog* cl, const lstep_csr* csr, const int64_t* src, const int64_t* dst,
                        const double* tq, int64_t n_edges, const int64_t* ids, int64_t n_ids, double current_time, int head, int len,
                        const float* G, const int64_t* const* query_ids_host, int n_queries, int64_t q_off, int64_t q_rows, float* nbr_out,
                        int K, const lstep_pe_mlp* mlp_nbr, const lstep_pe_mlp* mlp_upd, void* workspace, size_t workspace_bytes,
                        uint32_t* err_flag, void* stream, int phase);
// The change-log close of a step (changelog_step_core, peer_step_core): the step's kernels after the filter (`peer`: a peer
// rank's plan, else NULL), then its events appended into *slot: `head`, retired first, once the window is full, else the next
// free slot. A peer rank appends only with bit 2 of peer->phases.
int changelog_step_close(const lstep_pe_stream* s, const lstep_changelog* cl, const lstep_csr* csr, const int64_t* src, const int64_t* dst,
                         const double* tq, int64_t n_edges, const int64_t* ids, int64_t n_ids, double current_time, int head, int len,
                         const int64_t* const* query_ids_host, int n_queries, int64_t q_off, int64_t q_rows, float* nbr_out, int K,
                         const lstep_pe_mlp* mlp_nbr, const lstep_pe_mlp* mlp_upd, void* workspace, size_t workspace_bytes,
                         uint32_t* err_flag, void* stream, const PeerPlan* peer, int* slot);

}  // namespace lstep
