// Host-fed streaming step: the per-batch call a loop holding HOST (numpy) batches makes.
//
// The reference's loops hand every batch to the model as host arrays and read the predictions back
// (train_LSTEP_link_prediction.py:204-313, evaluate_model_utils.py:38-142). lstep_pe_step_host is the
// native form of that hand-over for the PE path: one call packs the batch (endpoints, times, the sorted
// unique batch nodes, the C query id sets) into a pinned slot, moves it with ONE async copy, enqueues the
// whole step (pe_step_core, csrc/step.cu), reduces the [C][n][d] neighbourhood PEs to the per-query row
// sums a caller reads back, and copies those to a pinned result slot, all on the caller's stream, without
// synchronising. lstep_host_step_result waits for a ticket's event and hands out the pinned result, so a
// loop can keep `slots - 1` steps in flight (results read one step behind hide the host's own time).
// lstep_pe_step_changelog_host is the same hand-over around the change-log step (changelog_step_core, csrc/changelog.cu):
// host_stage and host_finish below are the two halves both share, the step between them is the only difference.
// lstep_pe_step_peer_host puts one rank's peer-group step (peer_step_core, csrc/peer.cu) between them, with the rank's owned plan
// of the batch derived on the device while the batch is staged.
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <new>
#include <vector>

#include "common.cuh"
#include "step_core.cuh"

namespace lstep {

// The batch moves in and the result moves out through KERNELS that read / write the pinned slots directly
// (pinned host memory is device-addressable under unified virtual addressing): a copy-engine transfer between
// two kernels costs a stream hand-over in each direction (~6-8 us each for these 14 KB / 3 KB payloads) and
// is slower than a 4-CTA copy kernel. The copy-in runs on a side stream (it overlaps the previous step; the
// compute stream waits on its event), the result kernel on another (the next step does not queue behind it).
__global__ void __launch_bounds__(256) stage_in_kernel(const uint4* __restrict__ host_slot, uint4* __restrict__ dev_slot, int64_t n16) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n16; i += (int64_t)gridDim.x * blockDim.x)
    dev_slot[i] = __ldcv(host_slot + i);  // the host rewrites the pinned slot between launches: never cached
}

// res[row] = sum_c x[row][c]: one warp per row, lanes stride the columns, fixed-order shuffle tree
__global__ void __launch_bounds__(256) row_sum_kernel(const float* __restrict__ x, int64_t n_rows, int d, float* __restrict__ res) {
  pdl_launch_dependents();
  pdl_wait();
  const int64_t row = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (row >= n_rows) return;
  const float* p = x + row * d;
  float acc = 0.f;
  for (int c = lane; c < d; c += 32) acc += ld_dep(p + c);
  acc = warp_sum(acc);
  if (lane == 0) res[row] = acc;
}

constexpr int kMaxSlots = 8;

}  // namespace lstep

using namespace lstep;

// A batch staged by host_stage: its slot and, in the slot's device copy, src | dst | t | ids | query sets.
struct HostBatch {
  int slot;
  int64_t n_ids;
  double tmax;
  const int64_t* dp;
  const int64_t* qdev[8];
};

struct lstep_host_stepper {
  int slots;
  int64_t max_edges;
  int max_queries;
  int d;
  size_t in_bytes;   // capacity of one input slot
  size_t res_floats; // capacity of one result slot
  char* h_in[kMaxSlots];
  char* d_in[kMaxSlots];
  float* h_res[kMaxSlots];
  cudaEvent_t done[kMaxSlots];       // result of the slot's step is in the pinned result slot
  cudaEvent_t in_ready[kMaxSlots];   // the slot's batch is on the device
  cudaEvent_t step_done[kMaxSlots];  // the slot's step has written nbr_out
  float* d_nbr[kMaxSlots];           // [max_queries][max_edges][d] per slot: the result kernel of step i reads it while step i+1 runs
  cudaStream_t in_stream, out_stream;  // side streams: copy-in overlaps the previous step, the result path leaves the critical path
  int64_t res_n[kMaxSlots];
  int64_t ticket_of[kMaxSlots];  // ticket currently held by the slot, -1 = none
  float* d_nbr_out;              // [max_queries][max_edges][d] when the caller keeps no copy of its own
  int64_t next_ticket;
  uint64_t h2d_bytes, d2h_bytes;
  // lstep_host_stepper_set_ingest: append each batch to a growable CSR before its step (ing_fill NULL: disarmed)
  int32_t* ing_fill;
  int64_t ing_next_eid;
  double ing_last_t;
  bool ing_wait;              // the next append waits for the compute stream (just armed, or the CSR's arrays changed)
  const void* ing_arrays[4];  // indptr, nbr, eid, t of the CSR the last append wrote
  cudaEvent_t ing_ev;         // compute stream -> append (ing_wait)
  cudaEvent_t ing_staged;     // copy-in -> append
  cudaStream_t ing_stream;    // the appends: highest priority, so that the append CTA gets the first free SM slot
  // lstep_pe_step_peer_host: per slot, the rank's owned ids of the staged batch and their positions (ids_mine | pos_mine,
  // 2 x 2 * max_edges int64, allocated by the first peer call), and the batch a call with phase bit 0 staged for the later
  // phases of the same step
  int64_t* d_mine[kMaxSlots];
  bool peer_pending;
  HostBatch peer_hb;
  int64_t peer_n_edges, peer_n_mine;
  int peer_n_queries;
};

// sorted unique ids of src[0..n) U dst[0..n) -> out[<= 2n]. Small id spaces: a bitmap over [0, V1) scanned in
// order (1 us for 11 k nodes); otherwise (or when an id is out of range, which the device lookup reports) sort.
static int64_t unique_sorted_ids(const int64_t* src, const int64_t* dst, size_t n, int64_t V1, int64_t* out) {
  static thread_local std::vector<uint64_t> bits;
  if (V1 > 0 && V1 <= (1 << 18)) {
    const size_t words = (size_t)(V1 + 63) / 64;
    if (bits.size() < words) bits.assign(words, 0);
    bool ok = true;
    for (size_t i = 0; i < n && ok; ++i) {
      const int64_t a = src[i], b = dst[i];
      if (a < 0 || a >= V1 || b < 0 || b >= V1) {
        ok = false;
        break;
      }
      bits[(size_t)a >> 6] |= 1ull << (a & 63);
      bits[(size_t)b >> 6] |= 1ull << (b & 63);
    }
    if (ok) {
      int64_t m = 0;
      for (size_t w = 0; w < words; ++w) {
        uint64_t x = bits[w];
        if (!x) continue;
        bits[w] = 0;
        while (x) {
          out[m++] = (int64_t)(w * 64 + (size_t)__builtin_ctzll(x));
          x &= x - 1;
        }
      }
      return m;
    }
    std::fill(bits.begin(), bits.begin() + words, 0);
  }
  memcpy(out, src, 8 * n);
  memcpy(out + n, dst, 8 * n);
  std::sort(out, out + 2 * n);
  return std::unique(out, out + 2 * n) - out;
}

static int cuda_fail(cudaError_t e, const char* where) {
  set_cuda_error(e, where);
  return LSTEP_ERR_CUDA;
}

extern "C" void lstep_host_stepper_destroy(lstep_host_stepper* h) {
  if (!h) return;
  for (int i = 0; i < h->slots; ++i) {
    if (h->done[i]) cudaEventDestroy(h->done[i]);
    if (h->in_ready[i]) cudaEventDestroy(h->in_ready[i]);
    if (h->step_done[i]) cudaEventDestroy(h->step_done[i]);
    if (h->d_nbr[i]) cudaFree(h->d_nbr[i]);
    if (h->h_in[i]) cudaFreeHost(h->h_in[i]);
    if (h->h_res[i]) cudaFreeHost(h->h_res[i]);
    if (h->d_in[i]) cudaFree(h->d_in[i]);
    if (h->d_mine[i]) cudaFree(h->d_mine[i]);
  }
  if (h->d_nbr_out) cudaFree(h->d_nbr_out);
  if (h->ing_ev) cudaEventDestroy(h->ing_ev);
  if (h->ing_staged) cudaEventDestroy(h->ing_staged);
  if (h->ing_stream) cudaStreamDestroy(h->ing_stream);
  if (h->in_stream) cudaStreamDestroy(h->in_stream);
  if (h->out_stream) cudaStreamDestroy(h->out_stream);
  delete h;
}

extern "C" int lstep_host_stepper_create(int slots, int64_t max_edges, int max_queries, int d, lstep_host_stepper** out) {
  if (!out || slots < 1 || slots > kMaxSlots || max_edges <= 0 || max_queries < 0 || max_queries > 8 || d <= 0)
    return LSTEP_ERR_INVALID_ARG;
  lstep_host_stepper* h = new (std::nothrow) lstep_host_stepper();
  if (!h) return LSTEP_ERR_INVALID_ARG;
  h->slots = slots;
  h->max_edges = max_edges;
  h->max_queries = max_queries;
  h->d = d;
  // src | dst | t | ids (<= 2n) | C query sets, 8 bytes each
  h->in_bytes = align_up(sizeof(int64_t) * (size_t)max_edges * (size_t)(5 + max_queries), 16);
  h->res_floats = (size_t)std::max(1, max_queries) * (size_t)max_edges;
  h->next_ticket = 0;
  h->h2d_bytes = h->d2h_bytes = 0;
  h->d_nbr_out = nullptr;
  h->in_stream = h->out_stream = nullptr;
  h->ing_fill = nullptr;
  h->ing_next_eid = 0;
  h->ing_last_t = 0.0;
  h->ing_wait = false;
  for (int k = 0; k < 4; ++k) h->ing_arrays[k] = nullptr;
  h->ing_ev = h->ing_staged = nullptr;
  h->ing_stream = nullptr;
  h->peer_pending = false;
  h->peer_hb = HostBatch{};
  h->peer_n_edges = h->peer_n_mine = 0;
  h->peer_n_queries = 0;
  for (int i = 0; i < kMaxSlots; ++i) {
    h->h_in[i] = h->d_in[i] = nullptr;
    h->h_res[i] = nullptr;
    h->done[i] = h->in_ready[i] = h->step_done[i] = nullptr;
    h->d_nbr[i] = nullptr;
    h->d_mine[i] = nullptr;
    h->ticket_of[i] = -1;
    h->res_n[i] = 0;
  }
  cudaError_t e = cudaSuccess;
  for (int i = 0; i < slots && e == cudaSuccess; ++i) {
    if ((e = cudaHostAlloc((void**)&h->h_in[i], h->in_bytes, cudaHostAllocDefault)) != cudaSuccess) break;
    if ((e = cudaHostAlloc((void**)&h->h_res[i], sizeof(float) * h->res_floats, cudaHostAllocDefault)) != cudaSuccess) break;
    if ((e = cudaMalloc((void**)&h->d_in[i], h->in_bytes)) != cudaSuccess) break;
    if ((e = cudaEventCreateWithFlags(&h->done[i], cudaEventDisableTiming)) != cudaSuccess) break;
    if ((e = cudaEventCreateWithFlags(&h->in_ready[i], cudaEventDisableTiming)) != cudaSuccess) break;
    if ((e = cudaEventCreateWithFlags(&h->step_done[i], cudaEventDisableTiming)) != cudaSuccess) break;
    if ((e = cudaMalloc((void**)&h->d_nbr[i], sizeof(float) * h->res_floats * (size_t)d)) != cudaSuccess) break;
  }
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&h->in_stream, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&h->out_stream, cudaStreamNonBlocking);
  if (e != cudaSuccess) {
    lstep_host_stepper_destroy(h);
    return cuda_fail(e, "host_stepper_create");
  }
  *out = h;
  return LSTEP_OK;
}

// A peer rank's owned plan of the batch being staged (into the slot's d_mine): world and rank in, n_mine out.
struct PeerStage {
  int world, rank;
  int64_t n_mine;
};

// The first half of a host-fed step: slot wait, pack, the host id-range and ingest checks, copy-in, the optional owned plan of a
// peer rank and append, both on the copy-in path, and the hand-over to the compute stream (in_ready). A call rejected by a check
// has enqueued nothing.
static int host_stage(lstep_host_stepper* h, const lstep_pe_stream* s, const lstep_csr* csr, int64_t n_edges, const int64_t* src_host,
                      const int64_t* dst_host, const double* t_host, const int64_t* ids_host, int64_t n_ids,
                      const int64_t* const* query_ids_host_arrays, int n_queries, uint32_t* err_flag, cudaStream_t st, HostBatch* hb,
                      PeerStage* peer = nullptr) {
  if (!h || !s || n_edges <= 0 || n_edges > h->max_edges || n_queries < 0 || n_queries > h->max_queries) return LSTEP_ERR_INVALID_ARG;
  if (!src_host || !dst_host || !t_host || (n_queries > 0 && !query_ids_host_arrays)) return LSTEP_ERR_INVALID_ARG;
  if (ids_host && (n_ids < 0 || n_ids > 2 * n_edges)) return LSTEP_ERR_INVALID_ARG;
  for (int c = 0; c < n_queries; ++c)
    if (!query_ids_host_arrays[c]) return LSTEP_ERR_INVALID_ARG;
  if (s->d != h->d) return LSTEP_ERR_INVALID_ARG;
  const int slot = (int)(h->next_ticket % h->slots);
  cudaError_t e;
  if (h->ticket_of[slot] >= 0) {  // the slot's previous step (copy in, kernels, copy out) must have drained
    if ((e = cudaEventSynchronize(h->done[slot])) != cudaSuccess) return cuda_fail(e, "pe_step_host slot wait");
  }
  const size_t n = (size_t)n_edges;
  int64_t* hp = reinterpret_cast<int64_t*>(h->h_in[slot]);
  int64_t* h_src = hp;
  int64_t* h_dst = hp + n;
  double* h_t = reinterpret_cast<double*>(hp + 2 * n);
  int64_t* h_ids = hp + 3 * n;  // room for 2n
  int64_t* h_q = hp + 5 * n;
  memcpy(h_src, src_host, 8 * n);
  memcpy(h_dst, dst_host, 8 * n);
  memcpy(h_t, t_host, 8 * n);
  double tmax = t_host[0];
  for (size_t i = 1; i < n; ++i) tmax = t_host[i] > tmax ? t_host[i] : tmax;
  if (ids_host) {
    memcpy(h_ids, ids_host, 8 * (size_t)n_ids);
  } else {  // sorted unique endpoints (evaluate_model_utils.py:54-55 does this with torch.unique on the host)
    n_ids = unique_sorted_ids(src_host, dst_host, n, s->V1, h_ids);
  }
  for (int c = 0; c < n_queries; ++c) memcpy(h_q + (size_t)c * n, query_ids_host_arrays[c], 8 * n);
  {
    // every id indexes the [V1, d] table and the ring on the device: reject out-of-range ids here (the reference
    // raises IndexError on them, utils.py:140 / LSTEP.py:303; the Python host maps this status to IndexError)
    const int64_t V1 = s->V1;
    bool ok = n_ids == 0 || (h_ids[0] >= 0 && h_ids[n_ids - 1] < V1);  // sorted
    if (ids_host)
      for (int64_t i = 0; i < n_ids && ok; ++i) ok = h_ids[i] >= 0 && h_ids[i] < V1;
    for (size_t i = 0; i < n && ok; ++i) ok = src_host[i] >= 0 && src_host[i] < V1 && dst_host[i] >= 0 && dst_host[i] < V1;
    for (size_t i = 0; i < (size_t)n_queries * n && ok; ++i) ok = h_q[i] >= 0 && h_q[i] < V1;
    if (!ok) return LSTEP_ERR_ID_RANGE;
  }
  const bool ingest = h->ing_fill != nullptr;
  if (ingest) {  // the batch goes into the growable CSR: the same conditions lstep_csr_ingest's guards check, on the host
    if (!csr) return LSTEP_ERR_INVALID_ARG;
    double prev = h->ing_last_t;
    for (size_t i = 0; i < n; ++i) {
      if (!std::isfinite(t_host[i]) || t_host[i] < prev) return LSTEP_ERR_INVALID_ARG;
      prev = t_host[i];
    }
    for (size_t i = 0; i < n; ++i)
      if (src_host[i] >= csr->num_rows || dst_host[i] >= csr->num_rows) return LSTEP_ERR_ID_RANGE;  // (>= 0: checked above)
    if (h->ing_next_eid < 0 || h->ing_next_eid + n_edges - 1 > 0x7fffffffLL) return LSTEP_ERR_ID_RANGE;
  }
  const size_t bytes = 8 * n * (size_t)(5 + n_queries);
  // copy-in on its own stream: it only has to wait for the slot's previous use (synchronised above), so it runs
  // while the previous step is still computing; the compute stream picks it up through an event
  stage_in_kernel<<<4, 256, 0, h->in_stream>>>(reinterpret_cast<const uint4*>(h->h_in[slot]), reinterpret_cast<uint4*>(h->d_in[slot]),
                                               (int64_t)((bytes + 15) / 16));
  int rc0 = check_launch("stage_in");
  if (rc0 != LSTEP_OK) return rc0;
  if (peer) {
    // the rank's owned ids of the batch and their positions, from the staged ids, on the copy-in stream: off the compute stream's
    // chain like the append. The filter launch is sized by n_mine, counted here from the same ids.
    int64_t m = 0;
    for (int64_t i = 0; i < n_ids; ++i) m += h_ids[i] % peer->world == peer->rank;
    int64_t* mine = h->d_mine[slot];
    const int64_t* ids_dev = reinterpret_cast<const int64_t*>(h->d_in[slot]) + 3 * n;
    if ((rc0 = peer_plan_mine(ids_dev, n_ids, peer->world, peer->rank, mine, mine + 2 * h->max_edges, h->in_stream)) != LSTEP_OK) return rc0;
    peer->n_mine = m;
  }
  if (ingest) {
    // The batch is appended to the CSR from the staged slot, on the copy-in path: on a high-priority stream that waits for
    // the copy-in and records in_ready, so the compute stream sees the grown CSR and the step's launch chain is unchanged.
    // (The step's kernels, launched ahead with programmatic dependent launch, keep the SMs occupied; at default priority the
    // append CTA only found room between two steps.) The append of batch b+1 may run while step b still reads the
    // CSR. That is safe: step b queries at times <= tmax_b (a6 at its edge times, phase B at its edge times), every time
    // being written is >= the last time ingested >= tmax_b, and every slot being written held padding (t = +inf). Each
    // reader counts the entries of a row with t < tq (strict) and reads nothing at or after that count, so the written
    // slots count as "not earlier" both before and after the write (an aligned 8-byte store is seen whole or not at all),
    // and step b selects the same entries whichever it sees. fill[] is read by the appends only.
    // The change-log step (lstep_pe_step_changelog_host) reads the CSR in the same two places only, the a6 gather and
    // phase B's push, through the same strict-< counts; its filter, retire and append kernels read the change log and the
    // table, never the CSR. So the same argument covers it and its appends overlap the same way.
    // A peer rank's step (lstep_pe_step_peer_host) appends to the rank's own CSR replica and reads it in the same two places:
    // the a6 gather of its share of the query rows and the push kernel's lookups of all batch nodes, both through strict-<
    // counts. Its owned-plan kernel, filter, barrier refresh, phase-A broadcast, change-log append and publication never read
    // the CSR. So the append of batch b+1 overlaps step b there too.
    const void* arrays[4] = {csr->indptr, csr->nbr, csr->eid, csr->t};
    bool changed = false;
    for (int k = 0; k < 4; ++k) changed |= arrays[k] != h->ing_arrays[k];
    if ((e = cudaEventRecord(h->ing_staged, h->in_stream)) != cudaSuccess) return cuda_fail(e, "pe_step_host ingest event");
    if ((e = cudaStreamWaitEvent(h->ing_stream, h->ing_staged, 0)) != cudaSuccess) return cuda_fail(e, "pe_step_host ingest wait");
    if (h->ing_wait || changed) {  // a relayout or an append enqueued on the compute stream must land first
      if ((e = cudaEventRecord(h->ing_ev, st)) != cudaSuccess) return cuda_fail(e, "pe_step_host ingest event");
      if ((e = cudaStreamWaitEvent(h->ing_stream, h->ing_ev, 0)) != cudaSuccess) return cuda_fail(e, "pe_step_host ingest wait");
    }
    const int64_t* dp_in = reinterpret_cast<const int64_t*>(h->d_in[slot]);
    const int rc1 = lstep_csr_ingest(csr, h->ing_fill, dp_in, dp_in + n, nullptr, h->ing_next_eid,
                                     reinterpret_cast<const double*>(dp_in + 2 * n), n_edges, err_flag, h->ing_stream);
    if (rc1 != LSTEP_OK) return rc1;
    h->ing_wait = false;
    for (int k = 0; k < 4; ++k) h->ing_arrays[k] = arrays[k];
    h->ing_next_eid += n_edges;
    h->ing_last_t = t_host[n - 1];
  }
  if ((e = cudaEventRecord(h->in_ready[slot], ingest ? h->ing_stream : h->in_stream)) != cudaSuccess)
    return cuda_fail(e, "pe_step_host event");
  if ((e = cudaStreamWaitEvent(st, h->in_ready[slot], 0)) != cudaSuccess) return cuda_fail(e, "pe_step_host wait");
  h->h2d_bytes += bytes;
  const int64_t* dp = reinterpret_cast<const int64_t*>(h->d_in[slot]);
  for (int c = 0; c < n_queries; ++c) {
    // the same host array passed twice (negative sources == sources under random negative sampling) becomes the same
    // device pointer, which is what pe_step_core recognises as an identical query set
    int u = 0;
    while (u < c && query_ids_host_arrays[u] != query_ids_host_arrays[c]) ++u;
    hb->qdev[c] = dp + 5 * n + (size_t)u * n;
  }
  hb->slot = slot;
  hb->n_ids = n_ids;
  hb->tmax = tmax;
  hb->dp = dp;
  return LSTEP_OK;
}

// The second half: the per-query row sums of outp into the slot's pinned result, the slot's done event and the ticket.
// rows_per_query: n_edges, or a peer rank's share q_rows of them.
static int host_finish(lstep_host_stepper* h, const HostBatch& hb, int64_t rows_per_query, int n_queries, float* nbr_out, const float* outp,
                       cudaStream_t st, int64_t* ticket) {
  const int slot = hb.slot;
  cudaError_t e;
  int rc;
  const int64_t rows = (int64_t)n_queries * rows_per_query;
  // result path on its own stream, behind the step: the next step does not queue behind it. (A caller-owned
  // nbr_out is reused by the caller's next step, so in that case the result kernel stays on the compute stream.)
  cudaStream_t rs = nbr_out ? st : h->out_stream;
  if (!nbr_out) {
    if ((e = cudaEventRecord(h->step_done[slot], st)) != cudaSuccess) return cuda_fail(e, "pe_step_host event");
    if ((e = cudaStreamWaitEvent(rs, h->step_done[slot], 0)) != cudaSuccess) return cuda_fail(e, "pe_step_host wait");
  }
  if (rows > 0) {
    // the row sums go straight into the pinned result slot (visible to the host once the event below has fired)
    row_sum_kernel<<<(unsigned)ceil_div(rows * 32, 256), 256, 0, rs>>>(outp, rows, h->d, h->h_res[slot]);
    if ((rc = check_launch("row_sum")) != LSTEP_OK) return rc;
    h->d2h_bytes += sizeof(float) * (size_t)rows;
  }
  if ((e = cudaEventRecord(h->done[slot], rs)) != cudaSuccess) return cuda_fail(e, "pe_step_host event");
  h->res_n[slot] = rows;
  h->ticket_of[slot] = h->next_ticket;
  *ticket = h->next_ticket++;
  return LSTEP_OK;
}

extern "C" int lstep_pe_step_host(lstep_host_stepper* h, const lstep_pe_stream* s, const lstep_csr* csr, int64_t n_edges,
                                  const int64_t* src_host, const int64_t* dst_host, const double* t_host,
                                  const int64_t* ids_host, int64_t n_ids, int head, int len, int append_slot, const float* G,
                                  const int64_t* const* query_ids_host_arrays, int n_queries, float* nbr_out, int K,
                                  const lstep_pe_mlp* mlp_nbr, const lstep_pe_mlp* mlp_upd, void* workspace,
                                  size_t workspace_bytes, uint32_t* err_flag, void* stream, int64_t* ticket) {
  if (!ticket) return LSTEP_ERR_INVALID_ARG;
  const cudaStream_t st = as_stream(stream);
  HostBatch hb;
  int rc = host_stage(h, s, csr, n_edges, src_host, dst_host, t_host, ids_host, n_ids, query_ids_host_arrays, n_queries, err_flag, st, &hb);
  if (rc != LSTEP_OK) return rc;
  const int64_t* dp = hb.dp;
  float* outp = nbr_out ? nbr_out : h->d_nbr[hb.slot];
  rc = pe_step_core(s, csr, dp, dp + n_edges, reinterpret_cast<const double*>(dp + 2 * n_edges), n_edges, dp + 3 * n_edges, hb.n_ids, hb.tmax,
                    head, len, append_slot, G, hb.qdev, n_queries, outp, K, mlp_nbr, mlp_upd, workspace, workspace_bytes, err_flag, stream);
  if (rc != LSTEP_OK) return rc;
  return host_finish(h, hb, n_edges, n_queries, nbr_out, outp, st, ticket);
}

extern "C" int lstep_pe_step_changelog_host(lstep_host_stepper* h, const lstep_pe_stream* s, const lstep_changelog* cl, const lstep_csr* csr,
                                            int64_t n_edges, const int64_t* src_host, const int64_t* dst_host, const double* t_host,
                                            const int64_t* ids_host, int64_t n_ids, int head, int len, const float* G,
                                            const int64_t* const* query_ids_host_arrays, int n_queries, float* nbr_out, int K,
                                            const lstep_pe_mlp* mlp_nbr, const lstep_pe_mlp* mlp_upd, void* workspace,
                                            size_t workspace_bytes, uint32_t* err_flag, void* stream, int64_t* ticket) {
  if (!h || !s || !cl || !csr || !G || !mlp_nbr || K <= 0 || !ticket) return LSTEP_ERR_INVALID_ARG;
  int rc = changelog_step_check(s, cl, head, len, mlp_upd);
  if (rc != LSTEP_OK) return rc;
  if (cl->row_mul != 1) return LSTEP_ERR_INVALID_ARG;  // one GPU's whole history (a peer group steps through lstep_pe_step_peer)
  const cudaStream_t st = as_stream(stream);
  HostBatch hb;
  rc = host_stage(h, s, csr, n_edges, src_host, dst_host, t_host, ids_host, n_ids, query_ids_host_arrays, n_queries, err_flag, st, &hb);
  if (rc != LSTEP_OK) return rc;
  const int64_t* dp = hb.dp;
  float* outp = nbr_out ? nbr_out : h->d_nbr[hb.slot];
  rc = changelog_step_core(s, cl, csr, dp, dp + n_edges, reinterpret_cast<const double*>(dp + 2 * n_edges), n_edges, dp + 3 * n_edges, hb.n_ids,
                           hb.tmax, head, len, G, hb.qdev, n_queries, 0, -1, outp, K, mlp_nbr, mlp_upd, workspace, workspace_bytes, err_flag,
                           stream, 0);
  if (rc != LSTEP_OK) return rc;
  return host_finish(h, hb, n_edges, n_queries, nbr_out, outp, st, ticket);
}

extern "C" int lstep_host_step_result(lstep_host_stepper* h, int64_t ticket, const float** result_host, int64_t* n_floats) {
  if (!h || ticket < 0 || ticket >= h->next_ticket) return LSTEP_ERR_INVALID_ARG;
  const int slot = (int)(ticket % h->slots);
  if (h->ticket_of[slot] != ticket) return LSTEP_ERR_INVALID_ARG;  // the slot has been reused: result gone
  cudaError_t e = cudaEventSynchronize(h->done[slot]);
  if (e != cudaSuccess) return cuda_fail(e, "host_step_result");
  if (result_host) *result_host = h->h_res[slot];
  if (n_floats) *n_floats = h->res_n[slot];
  return LSTEP_OK;
}

extern "C" int lstep_host_stepper_set_ingest(lstep_host_stepper* h, int32_t* fill, int64_t next_eid, double last_t) {
  if (!h) return LSTEP_ERR_INVALID_ARG;
  if (fill && (next_eid < 0 || next_eid > 0x7fffffffLL || std::isnan(last_t))) return LSTEP_ERR_INVALID_ARG;
  if (fill && !h->ing_stream) {
    int least = 0, greatest = 0;
    cudaError_t e = cudaDeviceGetStreamPriorityRange(&least, &greatest);
    if (e == cudaSuccess && !h->ing_ev) e = cudaEventCreateWithFlags(&h->ing_ev, cudaEventDisableTiming);
    if (e == cudaSuccess && !h->ing_staged) e = cudaEventCreateWithFlags(&h->ing_staged, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaStreamCreateWithPriority(&h->ing_stream, cudaStreamNonBlocking, greatest);
    if (e != cudaSuccess) return cuda_fail(e, "host_stepper_set_ingest");
  }
  h->ing_fill = fill;
  h->ing_next_eid = next_eid;
  h->ing_last_t = last_t;
  h->ing_wait = fill != nullptr;
  return LSTEP_OK;
}

extern "C" void lstep_host_stepper_bytes(const lstep_host_stepper* h, uint64_t* h2d_bytes, uint64_t* d2h_bytes) {
  if (!h) return;
  if (h2d_bytes) *h2d_bytes = h->h2d_bytes;
  if (d2h_bytes) *d2h_bytes = h->d2h_bytes;
}

// The loop of a multi-batch host-fed call: batch b = edges [b*batch_size, min((b+1)*batch_size, n_total)), stepped by
// step(lo, n, query sets, head, &ticket) with the full window (the oldest slot, head, is overwritten and becomes the newest),
// its result read one step behind into results_host [n_batches][n_queries][batch_size] (the first rows of each query set's
// row when a step's result covers only a share of the batch).
template <class Step>
static int steps_host_loop(lstep_host_stepper* h, int T, int64_t n_total, int64_t batch_size, const int64_t* const* query_ids_host_arrays,
                           int n_queries, int* head_io, float* results_host, int64_t* n_done_out, Step&& step) {
  int head = *head_io;
  int64_t pending = -1, pending_b = -1, pending_n = 0;
  auto collect = [&](int64_t ticket, int64_t b, int64_t n) -> int {
    const float* r = nullptr;
    int64_t nf = 0;
    const int rc = lstep_host_step_result(h, ticket, &r, &nf);
    if (rc != LSTEP_OK) return rc;
    // rows per query: n, or a peer rank's share of the batch (the row sums of query set c are at r + c * rows)
    const int64_t rows = n_queries > 0 ? nf / n_queries : 0;
    float* dst = results_host + (size_t)b * n_queries * batch_size;
    for (int c = 0; c < n_queries; ++c) memcpy(dst + (size_t)c * batch_size, r + (size_t)c * rows, sizeof(float) * (size_t)rows);
    return LSTEP_OK;
  };
  int64_t b = 0;
  for (int64_t lo = 0; lo < n_total; lo += batch_size, ++b) {
    const int64_t n = n_total - lo < batch_size ? n_total - lo : batch_size;
    const int64_t* q[8];
    for (int c = 0; c < n_queries; ++c) q[c] = query_ids_host_arrays[c] + lo;
    int64_t ticket = -1;
    int rc = step(lo, n, q, head, &ticket);
    if (rc != LSTEP_OK) {
      // batches [0, b) HAVE been applied to the history: report the position reached (head, and the count in *len_io's place is
      // not possible — len stays T — so the caller derives it from the returned head and n_done below) and drain the pending result
      if (pending >= 0) (void)collect(pending, pending_b, pending_n);
      *head_io = head;
      if (n_done_out) *n_done_out = b;
      return rc;
    }
    head = (head + 1) % T;
    if (pending >= 0 && (rc = collect(pending, pending_b, pending_n)) != LSTEP_OK) {
      *head_io = head;
      if (n_done_out) *n_done_out = b + 1;
      return rc;
    }
    pending = ticket;
    pending_b = b;
    pending_n = n;
  }
  *head_io = head;
  if (n_done_out) *n_done_out = b;
  if (pending >= 0) {
    const int rc = collect(pending, pending_b, pending_n);
    if (rc != LSTEP_OK) return rc;
  }
  return LSTEP_OK;
}

// A whole run of consecutive batches in one call (an evaluation split: evaluate_model_utils.py:38-142 loops over
// batches of the split): the loop of lstep_pe_step_host + lstep_host_step_result lives here, results read one step
// behind, so the host cost per batch is the CUDA launches alone. Steady-state regime only (the history ring is full:
// *len_io == T, one collapsed filter G for every step); batch b is edges [b*batch_size, min((b+1)*batch_size, n_total)).
// results_host: [n_batches][n_queries][batch_size] floats (the tail of a ragged last batch is left untouched).
// Synchronous: every result has been read when the call returns.
extern "C" int lstep_pe_steps_host(lstep_host_stepper* h, const lstep_pe_stream* s, const lstep_csr* csr, int64_t n_total,
                                   int64_t batch_size, const int64_t* src_host, const int64_t* dst_host, const double* t_host,
                                   const int64_t* const* query_ids_host_arrays, int n_queries, int* head_io, int* len_io,
                                   const float* G, int K, const lstep_pe_mlp* mlp_nbr, const lstep_pe_mlp* mlp_upd,
                                   void* workspace, size_t workspace_bytes, uint32_t* err_flag, void* stream,
                                   float* results_host, int64_t* n_done_out) {
  if (n_done_out) *n_done_out = 0;
  if (!h || !s || !head_io || !len_io || !results_host || n_total < 0 || batch_size <= 0 || batch_size > h->max_edges)
    return LSTEP_ERR_INVALID_ARG;
  if (n_queries < 0 || n_queries > 8 || (n_queries > 0 && !query_ids_host_arrays)) return LSTEP_ERR_INVALID_ARG;
  if (*len_io != s->T) return LSTEP_ERR_UNSUPPORTED;  // masked regime: the filter changes every step, use the per-step call
  return steps_host_loop(h, s->T, n_total, batch_size, query_ids_host_arrays, n_queries, head_io, results_host, n_done_out,
                         [&](int64_t lo, int64_t n, const int64_t* const* q, int head, int64_t* ticket) {
                           return lstep_pe_step_host(h, s, csr, n, src_host + lo, dst_host + lo, t_host + lo, nullptr, 0, head, s->T, head, G,
                                                     q, n_queries, nullptr, K, mlp_nbr, mlp_upd, workspace, workspace_bytes, err_flag,
                                                     stream, ticket);
                         });
}

// lstep_pe_steps_host on a change-log history: every batch through lstep_pe_step_changelog_host with the full window (its
// events retire slot head and take its place). Same contract: steady state only, results one step behind, and on an error in
// batch k batches [0, k) stay applied, with *head_io / *n_done_out reporting the position reached.
extern "C" int lstep_pe_steps_changelog_host(lstep_host_stepper* h, const lstep_pe_stream* s, const lstep_changelog* cl, const lstep_csr* csr,
                                             int64_t n_total, int64_t batch_size, const int64_t* src_host, const int64_t* dst_host,
                                             const double* t_host, const int64_t* const* query_ids_host_arrays, int n_queries, int* head_io,
                                             int* len_io, const float* G, int K, const lstep_pe_mlp* mlp_nbr, const lstep_pe_mlp* mlp_upd,
                                             void* workspace, size_t workspace_bytes, uint32_t* err_flag, void* stream, float* results_host,
                                             int64_t* n_done_out) {
  if (n_done_out) *n_done_out = 0;
  if (!h || !s || !cl || !head_io || !len_io || !results_host || n_total < 0 || batch_size <= 0 || batch_size > h->max_edges)
    return LSTEP_ERR_INVALID_ARG;
  if (n_queries < 0 || n_queries > 8 || (n_queries > 0 && !query_ids_host_arrays)) return LSTEP_ERR_INVALID_ARG;
  const int rc = changelog_step_check(s, cl, *head_io, *len_io, mlp_upd);
  if (rc != LSTEP_OK) return rc;
  if (*len_io != cl->T) return LSTEP_ERR_UNSUPPORTED;  // the log is still filling: the filter changes every step, use the per-step call
  return steps_host_loop(h, cl->T, n_total, batch_size, query_ids_host_arrays, n_queries, head_io, results_host, n_done_out,
                         [&](int64_t lo, int64_t n, const int64_t* const* q, int head, int64_t* ticket) {
                           return lstep_pe_step_changelog_host(h, s, cl, csr, n, src_host + lo, dst_host + lo, t_host + lo, nullptr, 0, head,
                                                               cl->T, G, q, n_queries, nullptr, K, mlp_nbr, mlp_upd, workspace,
                                                               workspace_bytes, err_flag, stream, ticket);
                         });
}

// One rank's peer step between host_stage and host_finish (see the header). The checks that depend on the batch (host_stage's)
// and those that do not (peer_step_check) come before anything is enqueued, and every rank makes the same ones on the same
// batch: either every rank enqueues the step, or none does, and no rank waits at a barrier for a peer that rejected it.
static int step_peer_host(lstep_host_stepper* h, const lstep_pe_stream* s, const lstep_changelog* cl, const lstep_csr* csr, const lstep_peer_group* grp,
                          int64_t n_edges, const int64_t* src_host, const int64_t* dst_host, const double* t_host, const int64_t* ids_host,
                          int64_t n_ids, int head, int len, const float* G, const int64_t* const* query_ids_host_arrays, int n_queries,
                          float* nbr_out, int K, const lstep_pe_mlp* mlp_nbr, const lstep_pe_mlp* mlp_upd, void* workspace,
                          size_t workspace_bytes, uint32_t* err_flag, uint32_t epoch_base, int timeout_ms, int phases, void* stream,
                          int64_t* ticket, SideLane* side) {
  if (!h || !s || !cl || !csr || !grp || !G || K <= 0 || phases <= 0 || (phases & ~7) || ((phases & 4) && !ticket)) return LSTEP_ERR_INVALID_ARG;
  const bool stage = (phases & 1) != 0;
  if (stage == h->peer_pending) return LSTEP_ERR_INVALID_ARG;  // staging over a pending batch, or a later phase with none
  const int64_t n = stage ? n_edges : h->peer_n_edges;
  const int C = stage ? n_queries : h->peer_n_queries;
  if (grp->world < 1 || grp->world > LSTEP_MAX_PEERS || grp->rank < 0 || grp->rank >= grp->world) return LSTEP_ERR_INVALID_ARG;
  const int64_t q_off = grp->rank * n / grp->world, q_rows = (grp->rank + 1) * n / grp->world - q_off;
  int rc = peer_step_check(s, cl, csr, grp, n, head, len, mlp_nbr, mlp_upd, phases, q_rows);
  if (rc != LSTEP_OK) return rc;
  const cudaStream_t st = as_stream(stream);
  if (stage) {
    if (!h->d_mine[0]) {
      for (int i = 0; i < h->slots; ++i) {
        const cudaError_t e = cudaMalloc((void**)&h->d_mine[i], sizeof(int64_t) * 4 * (size_t)h->max_edges);
        if (e != cudaSuccess) return cuda_fail(e, "pe_step_peer_host plan buffer");
      }
    }
    PeerStage ps{grp->world, grp->rank, 0};
    HostBatch hb;
    rc = host_stage(h, s, csr, n_edges, src_host, dst_host, t_host, ids_host, n_ids, query_ids_host_arrays, n_queries, err_flag, st, &hb, &ps);
    if (rc != LSTEP_OK) return rc;
    h->peer_hb = hb;
    h->peer_n_edges = n_edges;
    h->peer_n_queries = n_queries;
    h->peer_n_mine = ps.n_mine;
    h->peer_pending = true;
  }
  const HostBatch& hb = h->peer_hb;
  const int64_t* dp = hb.dp;
  const int64_t* mine = h->d_mine[hb.slot];
  float* outp = nbr_out ? nbr_out : h->d_nbr[hb.slot];
  const int64_t* q[8] = {};
  for (int c = 0; c < C; ++c) q[c] = hb.qdev[c] + q_off;
  rc = peer_step_core(s, cl, csr, grp, dp, dp + n, reinterpret_cast<const double*>(dp + 2 * n), n, dp + 3 * n, hb.n_ids, mine,
                      mine + 2 * h->max_edges, h->peer_n_mine, hb.tmax, head, len, G, q, C, q_off, q_rows, outp, K, mlp_nbr, mlp_upd, workspace,
                      workspace_bytes, err_flag, epoch_base, timeout_ms, phases, stream, side);
  if (rc != LSTEP_OK || (phases & 4)) h->peer_pending = false;
  if (rc != LSTEP_OK || !(phases & 4)) return rc;
  return host_finish(h, hb, q_rows, C, nbr_out, outp, st, ticket);
}

extern "C" int lstep_pe_step_peer_host(lstep_host_stepper* h, const lstep_pe_stream* s, const lstep_changelog* cl, const lstep_csr* csr,
                                       const lstep_peer_group* grp, int64_t n_edges, const int64_t* src_host, const int64_t* dst_host,
                                       const double* t_host, const int64_t* ids_host, int64_t n_ids, int head, int len, const float* G,
                                       const int64_t* const* query_ids_host_arrays, int n_queries, float* nbr_out, int K,
                                       const lstep_pe_mlp* mlp_nbr, const lstep_pe_mlp* mlp_upd, void* workspace, size_t workspace_bytes,
                                       uint32_t* err_flag, uint32_t epoch_base, int timeout_ms, int phases, void* stream, int64_t* ticket) {
  return step_peer_host(h, s, cl, csr, grp, n_edges, src_host, dst_host, t_host, ids_host, n_ids, head, len, G, query_ids_host_arrays, n_queries,
                        nbr_out, K, mlp_nbr, mlp_upd, workspace, workspace_bytes, err_flag, epoch_base, timeout_ms, phases, stream, ticket,
                        nullptr);
}

// lstep_pe_steps_host for one rank of a peer group: every batch through the whole host-fed peer step (phases 7) with the full
// window, results (this rank's share) read one step behind, the publication of each step on a side stream next to the next
// step's filter, as in lstep_pe_steps_peer. On an error in batch k batches [0, k) stay applied: *head_io, *epoch_io and
// *n_done_out report the position reached.
extern "C" int lstep_pe_steps_peer_host(lstep_host_stepper* h, const lstep_pe_stream* s, const lstep_changelog* cl, const lstep_csr* csr,
                                        const lstep_peer_group* grp, int64_t n_total, int64_t batch_size, const int64_t* src_host,
                                        const int64_t* dst_host, const double* t_host, const int64_t* const* query_ids_host_arrays,
                                        int n_queries, int* head_io, int* len_io, const float* G, int K, const lstep_pe_mlp* mlp_nbr,
                                        const lstep_pe_mlp* mlp_upd, void* workspace, size_t workspace_bytes, uint32_t* err_flag,
                                        uint32_t* epoch_io, int timeout_ms, void* stream, float* results_host, int64_t* n_done_out) {
  if (n_done_out) *n_done_out = 0;
  if (!h || !s || !cl || !csr || !grp || !head_io || !len_io || !epoch_io || !results_host || n_total < 0 || batch_size <= 0 ||
      batch_size > h->max_edges)
    return LSTEP_ERR_INVALID_ARG;
  if (n_queries < 0 || n_queries > 8 || (n_queries > 0 && !query_ids_host_arrays)) return LSTEP_ERR_INVALID_ARG;
  if (h->peer_pending) return LSTEP_ERR_INVALID_ARG;
  int rc = peer_step_check(s, cl, csr, grp, batch_size, *head_io, *len_io, mlp_nbr, mlp_upd, 7, 0);
  if (rc != LSTEP_OK) return rc;
  if (*len_io != cl->T) return LSTEP_ERR_UNSUPPORTED;  // the log is still filling: the filter changes every step, use the per-step call
  uint32_t epoch = *epoch_io;
  SideLane lane;
  const bool overlap = grp->world > 1 && n_total > batch_size;
  if (overlap && (rc = side_lane_open(&lane)) != LSTEP_OK) return rc;
  rc = steps_host_loop(h, cl->T, n_total, batch_size, query_ids_host_arrays, n_queries, head_io, results_host, n_done_out,
                       [&](int64_t lo, int64_t n, const int64_t* const* q, int head, int64_t* ticket) {
                         const int r = step_peer_host(h, s, cl, csr, grp, n, src_host + lo, dst_host + lo, t_host + lo, nullptr, 0, head, cl->T,
                                                      G, q, n_queries, nullptr, K, mlp_nbr, mlp_upd, workspace, workspace_bytes, err_flag,
                                                      epoch, timeout_ms, 7, stream, ticket, overlap ? &lane : nullptr);
                         if (r == LSTEP_OK) epoch += 2;
                         return r;
                       });
  if (overlap) side_lane_close(&lane, as_stream(stream));
  *epoch_io = epoch;
  return rc;
}
