// Streaming PE step (SURVEY §8(f) f1): the whole per-batch sequence of the eval loop
// (evaluate_model_utils.py:54-135) as one C call on device-resident state:
//
//   a3   cur[ids] <- sum_s G[s] * ring[ids, (head+s) % T]            (DFT filter, scattered into the table)
//   a6   out[c]   <- neighbourhood PE of query set c at the batch's edge times, all C sets in ONE
//                    sampler / aggregate / MLP launch (C*B rows)
//   a7/8 cur      <- update_pe(cur)                                   (in place)
//        ring[:, slot] <- cur                                          (append: overwrite the oldest slot)
//
// `cur` always equals the newest ring slot between steps, so the loops' clone(hist[:, -1]) disappears,
// and the history is never trimmed or concatenated: one [V1, d] table copy per step remains (the H term
// of SURVEY §8(d)) instead of ~3 GB of clone + cat at Reddit size.
#include <algorithm>
#include <atomic>
#include <cstdlib>

#include "common.cuh"
#include "gather_bodies.cuh"
#include "mlp_job.cuh"
#include "step_core.cuh"

namespace lstep {

template <typename IdT, bool kWithEid>
int launch_sample(const lstep_csr* csr, RowIds q_node, const double* q_time, int64_t n_rows, int64_t n_valid, int K,
                  IdT* out_nbr, IdT* out_eid, float* out_t, uint32_t* err_flag, void* stream);
int launch_nbr_lookup_aggregate(const lstep_csr* csr, RowIds q_node, const float* pe, const double* q_time, int64_t n_rows, int K,
                                const float* tw, int d, int t, float* S, int64_t ldS, uint32_t* err_flag, cudaStream_t st);
void update_ws_phase_a(void* workspace, int64_t n_ids, int64_t n_edges, int K, int d, int t, int64_t pe_rows, float** A, int64_t* lda,
                       int32_t** counters, float** new_rows);

int update_pe_impl(float* pe, int64_t pe_rows, const lstep_csr* csr, const int64_t* ids, int64_t n_ids, const int64_t* src,
                   const int64_t* dst, const double* times, int64_t n_edges, double current_time, int K, const lstep_pe_mlp* mlp,
                   void* workspace, size_t workspace_bytes, uint32_t* err_flag, void* stream, bool edges_done, int32_t** dirty_out, int stamp, bool phase_a_in_new_rows,
                   float* ring_slot, int64_t ring_stride, const PushOwner* owner = nullptr);
int launch_phase_a_to_new_rows(const float* pe, void* workspace, int64_t ws_ids, int64_t ws_edges, int K, int64_t pe_rows, const int64_t* ids,
                               int64_t n_ids, const int64_t* src, const int64_t* dst, const double* times, int64_t n_edges, float tc,
                               const lstep_pe_mlp* mlp, bool aggregate_done, cudaStream_t st);

// a6's neighbourhood aggregate (blocks [0, grid_q)) and a7's edge aggregate (the rest) in ONE launch: both only
// read the current table and neither depends on the other, so the short edge kernel (and its hub chain) hides
// behind the cosine-bound neighbourhood rows instead of being a link of the step's dependency chain.
__global__ void __launch_bounds__(512) gather_ab_kernel(const float* __restrict__ pe, const double* __restrict__ q_time, int64_t n_rows,
                                                        int K, const float* __restrict__ tw_q, int d, int t, int t_pad,
                                                        float* __restrict__ S, int64_t ldS, int64_t period, LookupArgs lk, int grid_q,
                                                        const int64_t* __restrict__ ids, int64_t n_ids,
                                                        const int64_t* __restrict__ src, const int64_t* __restrict__ dst,
                                                        const double* __restrict__ times, int64_t n_edges, float tc,
                                                        const float* __restrict__ tw_u, float* __restrict__ A, int64_t lda,
                                                        int32_t* __restrict__ counters, int lk_base) {
  // The kernel in front (the DFT filter, launched with a late trigger: this kernel is resident only after
  // everything before the filter has completed) writes the table and nothing else this kernel touches. Lookups,
  // edge scans and all cosines therefore run BEFORE the dependency wait, next to the HBM-bound filter; only the
  // threads that gather table rows wait (inside the bodies).
  TL_ENTRY(1);
  pdl_launch_dependents();
#ifdef LSTEP_TIMELINE
  if (threadIdx.x == 0) atomicMax(&g_timeline[((int)blockIdx.x < grid_q ? 9 : 10) * 4 + 2], gtimer());  // last CTA START (nbr / edge)
#endif
  // lk_base > 0: the CTAs walk several query rows each; the warp at threads [lk_base, lk_base + 32) looks one row ahead
  if ((int)blockIdx.x < grid_q) {
    if (lk_base > 0)
      nbr_aggregate_rows_piped(blockIdx.x, grid_q, true, pe, q_time, n_rows, K, tw_q, d, t, t_pad, S, ldS, period, lk, lk_base);
    else
      nbr_aggregate_rows<4, true>(blockIdx.x, grid_q, true, pe, q_time, nullptr, nullptr, n_rows, K, tw_q, d, t, t_pad, S, ldS, period, lk);
  } else
    edge_aggregate_rows((int64_t)blockIdx.x - grid_q, (int64_t)gridDim.x - grid_q, (int)blockIdx.x == grid_q, true, pe, ids, n_ids, src, dst,
                        times, n_edges, tc, tw_u, d, t, t_pad, A, lda, counters);
#ifdef LSTEP_TIMELINE
  if (threadIdx.x == 0) atomicMax(&g_timeline[((int)blockIdx.x < grid_q ? 11 : 12) * 4 + 2], gtimer());  // last CTA EXIT (nbr / edge)
#endif
  TL_EXIT(1);
}
int launch_pe_mlp(const float* A, int64_t lda, const float* pe, RowIds base_ids, int64_t n_rows, int64_t expected_rows,
                  const int32_t* n_rows_dev, const lstep_pe_mlp* m, float* out, int64_t out_stride, float* pe_inplace,
                  cudaStream_t st, bool late_trigger = false);
int launch_dft_filter(const float* hist, int64_t node_stride, int64_t time_stride, int s0, int ring, int Th, int d,
                      const int64_t* ids, int64_t n_ids, const float* G, float* out, int64_t out_stride,
                      const int64_t* out_ids, void* stream, bool prefetch_old_rows);

// ring[v][slot][:] = cur[v][:]  (node-major ring: 688-byte rows at a 68.8 KB pitch)
// table row of ring row v is v*row_mul + row_add (1, 0 for a single GPU; G, rank for a node-id sharded ring)
// dirty != NULL (streaming step, push form of phase B): the kernel in front is the phase-B MLP, launched with a late
// trigger, so this kernel is resident only after the push kernel has completed: the set of rows the MLP is changing
// (dirty[v] == stamp) is final, and all other rows of `cur` are. Every thread copies its elements BEFORE the
// dependency wait, next to the MLP, and copies the elements of the changed rows again after it (same thread, same
// address: program order). 14 of the 15.1 MB move off the step's critical path.
__global__ void __launch_bounds__(256) ring_append_kernel(const float* __restrict__ cur, float* __restrict__ ring,
                                                          int64_t V1, int T, int d, int slot, int64_t row_mul, int64_t row_add,
                                                          const int32_t* dirty, int stamp) {
  TL_ENTRY(5);
  pdl_launch_dependents();
  const int dvec = d >> 2;
  const int64_t total = V1 * dvec;
  if (dirty) {
    // Rows carrying `stamp` are being rewritten by the phase-B MLP, which writes them into the ring slot itself; this
    // kernel copies all other rows, all of it before the dependency wait (the flags are final: the push kernel has
    // completed). kPer loads in flight per thread and sweep.
    constexpr int kPer = 8;
    const int64_t nthr = (int64_t)gridDim.x * blockDim.x, gtid = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    for (int64_t base = 0; base < total; base += nthr * kPer) {
      int flag[kPer];
      float4 val[kPer];
#pragma unroll
      for (int e = 0; e < kPer; ++e) {
        const int64_t i = base + gtid + e * nthr;
        flag[e] = i < total ? ld_dep(dirty + i / dvec) : stamp;
        if (i < total) val[e] = ld_dep(reinterpret_cast<const float4*>(cur + (i / dvec) * (int64_t)d) + (int)(i % dvec));
      }
#pragma unroll
      for (int e = 0; e < kPer; ++e) {
        const int64_t i = base + gtid + e * nthr;
        if (flag[e] != stamp) reinterpret_cast<float4*>(ring + ((i / dvec) * T + slot) * (int64_t)d)[i % dvec] = val[e];
      }
    }
    pdl_wait();  // (completion order only: the kernel must not finish before its predecessor)
    TL_WAITED(5);
    TL_EXIT(5);
    return;
  }
  pdl_wait();
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t v = i / dvec;
    const int c = (int)(i % dvec);
    reinterpret_cast<float4*>(ring + (v * T + slot) * (int64_t)d)[c] =
        ld_dep(reinterpret_cast<const float4*>(cur + (v * row_mul + row_add) * (int64_t)d) + c);
  }
}

__global__ void __launch_bounds__(256) ring_load_kernel(const float* __restrict__ ring, float* __restrict__ cur, int64_t V1,
                                                        int T, int d, int slot, int64_t row_mul, int64_t row_add) {
  const int dvec = d >> 2;
  const int64_t total = V1 * dvec;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t v = i / dvec;
    const int c = (int)(i % dvec);
    reinterpret_cast<float4*>(cur + (v * row_mul + row_add) * (int64_t)d)[c] =
        reinterpret_cast<const float4*>(ring + (v * T + slot) * (int64_t)d)[c];
  }
}

struct StepWs {
  void* update;  // lstep_update_pe workspace (first: its per-node counter map sits at offset 0)
  size_t update_bytes;
  int32_t* nbrQ;  // [C*B*K]
  float* ntQ;     // [C*B*K]
  float* S;       // [C*B][lda]
  int64_t lda;
  size_t bytes;
};

static StepWs carve_step(void* base, int64_t max_ids, int64_t max_edges, int C, int K, int d, int t, int64_t V1) {
  StepWs w;
  size_t o = 0;
  auto take = [&](size_t bytes) {
    void* p = base ? static_cast<char*>(base) + o : nullptr;
    o = align_up(o + bytes, 256);
    return p;
  };
  w.update_bytes = lstep_update_pe_workspace_bytes(max_ids, max_edges, K, d, t, V1);
  w.update = take(w.update_bytes);
  const size_t rows = (size_t)C * max_edges;
  w.nbrQ = (int32_t*)take(4 * rows * K);
  w.ntQ = (float*)take(4 * rows * K);
  w.lda = (int64_t)align_up((size_t)(d + t), 4);
  w.S = (float*)take(4 * rows * w.lda);
  w.bytes = o;
  return w;
}

}  // namespace lstep

using namespace lstep;

extern "C" size_t lstep_pe_step_workspace_bytes(int64_t max_ids, int64_t max_edges, int n_queries, int K, int d, int t,
                                                int64_t V1) {
  if (max_ids < 0 || max_edges < 0 || n_queries < 0 || n_queries > 8 || K <= 0 || d <= 0 || t < 0 || V1 <= 0) return 0;
  return carve_step(nullptr, max_ids, max_edges, n_queries, K, d, t, V1).bytes;
}

extern "C" int lstep_ring_load(const float* ring, float* cur, int64_t V1, int T, int d, int slot, void* stream) {
  if (!ring || !cur || V1 <= 0 || T <= 0 || d <= 0 || d % 4 != 0 || slot < 0 || slot >= T) return LSTEP_ERR_INVALID_ARG;
  ring_load_kernel<<<num_sms() * 8, 256, 0, as_stream(stream)>>>(ring, cur, V1, T, d, slot, 1, 0);
  return check_launch("ring_load");
}

namespace lstep {
// Rows [r0, r1) of new nodes: table row, every ring slot (node-major, so one contiguous T*d block per node) and, for the owned
// nodes (v % world == rank), the change-log base row at (v - rank) / world, from rows[(v - r0) * rows_stride] (stride 0: one
// broadcast row). One float4 per thread-iteration, grid-stride over the nodes' blocks.
__global__ void __launch_bounds__(256) pe_rows_init_kernel(float* __restrict__ table, float* __restrict__ ring, int T, int d,
                                                           float* __restrict__ base, int64_t world, int64_t rank, int64_t r0,
                                                           int64_t r1, const float* __restrict__ rows, int64_t rows_stride) {
  const int dvec = d / 4;
  const int64_t per_node = (int64_t)(1 + (ring ? T : 0)) * dvec;  // table row, then the T ring slots
  const int64_t total = (r1 - r0) * per_node;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += stride) {
    const int64_t k = i / per_node, j = i - k * per_node;
    const int64_t v = r0 + k;
    const int c = (int)(j % dvec);
    const float4 x = reinterpret_cast<const float4*>(rows + k * rows_stride)[c];
    if (j < dvec) {
      if (table) reinterpret_cast<float4*>(table + v * d)[c] = x;
      if (base && v % world == rank) reinterpret_cast<float4*>(base + ((v - rank) / world) * d)[c] = x;
    } else {
      reinterpret_cast<float4*>(ring + v * (int64_t)T * d)[j - dvec] = x;
    }
  }
}
}  // namespace lstep

extern "C" int lstep_pe_rows_init(float* table, float* ring, int T, int d, float* base, int64_t world, int64_t rank, int64_t r0, int64_t r1,
                                  const float* rows, int64_t rows_stride, void* stream) {
  if (!rows || d <= 0 || d % 4 != 0 || r0 < 0 || r1 < r0 || rows_stride < 0 || rows_stride % 4 != 0) return LSTEP_ERR_INVALID_ARG;
  if ((ring && T <= 0) || (base && (world <= 0 || rank < 0 || rank >= world))) return LSTEP_ERR_INVALID_ARG;
  if (reinterpret_cast<uintptr_t>(rows) % 16 || reinterpret_cast<uintptr_t>(table) % 16 || reinterpret_cast<uintptr_t>(ring) % 16 ||
      reinterpret_cast<uintptr_t>(base) % 16)
    return LSTEP_ERR_INVALID_ARG;
  if (r1 == r0 || (!table && !ring && !base)) return LSTEP_OK;
  const int64_t work = (r1 - r0) * (int64_t)(1 + (ring ? T : 0)) * (d / 4);
  const int64_t grid = std::min<int64_t>(ceil_div(work, 256), (int64_t)num_sms() * 8);
  pe_rows_init_kernel<<<(unsigned)grid, 256, 0, as_stream(stream)>>>(table, ring, T, d, base, world, rank, r0, r1, rows, rows_stride);
  return check_launch("pe_rows_init");
}

/* Sharded ring (rows v of the local ring <-> table rows v*row_mul + row_add): load / append one slot. */
extern "C" int lstep_ring_copy_rows(float* ring, float* cur, int64_t ring_rows, int T, int d, int slot, int64_t row_mul,
                                    int64_t row_add, int to_ring, void* stream) {
  if (!ring || !cur || ring_rows < 0 || T <= 0 || d <= 0 || d % 4 != 0 || slot < 0 || slot >= T || row_mul <= 0 || row_add < 0)
    return LSTEP_ERR_INVALID_ARG;
  if (ring_rows == 0) return LSTEP_OK;
  if (to_ring)
    launch_k(ring_append_kernel, dim3(num_sms() * 8), dim3(256), 0, as_stream(stream), cur, ring, ring_rows, T, d, slot, row_mul, row_add,
             nullptr, 0);
  else
    ring_load_kernel<<<num_sms() * 8, 256, 0, as_stream(stream)>>>(ring, cur, ring_rows, T, d, slot, row_mul, row_add);
  return check_launch("ring_copy_rows");
}

namespace lstep {
// The step on explicit batch pointers (src/dst/tq = the batch's n_edges endpoints and times on the device).
int pe_step_core(const lstep_pe_stream* s, const lstep_csr* csr, const int64_t* src, const int64_t* dst, const double* tq,
                 int64_t n_edges, const int64_t* ids, int64_t n_ids, double current_time, int head, int len, int append_slot,
                 const float* G, const int64_t* const* query_ids_host, int n_queries, float* nbr_out, int K,
                 const lstep_pe_mlp* mlp_nbr, const lstep_pe_mlp* mlp_upd, void* workspace, size_t workspace_bytes,
                 uint32_t* err_flag, void* stream) {
  return pe_step_core_ex(s, csr, src, dst, tq, n_edges, ids, n_ids, current_time, head, len, append_slot, G, query_ids_host, n_queries, nbr_out,
                         K, mlp_nbr, mlp_upd, workspace, workspace_bytes, err_flag, stream, StepOpts{});
}

int pe_step_core_ex(const lstep_pe_stream* s, const lstep_csr* csr, const int64_t* src, const int64_t* dst, const double* tq,
                    int64_t n_edges, const int64_t* ids, int64_t n_ids, double current_time, int head, int len, int append_slot,
                    const float* G, const int64_t* const* query_ids_host, int n_queries, float* nbr_out, int K,
                    const lstep_pe_mlp* mlp_nbr, const lstep_pe_mlp* mlp_upd, void* workspace, size_t workspace_bytes,
                    uint32_t* err_flag, void* stream, const StepOpts& opt) {
  if (!s || !csr || !mlp_nbr || !mlp_upd || (!G && !opt.skip_dft) || n_edges < 0 || n_ids < 0 || K <= 0 || n_queries < 0 || n_queries > 8)
    return LSTEP_ERR_INVALID_ARG;
  const int64_t q_rows = opt.q_rows < 0 ? n_edges : opt.q_rows;
  if (opt.q_off < 0 || opt.q_off + q_rows > n_edges) return LSTEP_ERR_INVALID_ARG;
  const double* tq_q = tq + opt.q_off;  // edge times of the a6 queries
  if (!s->ring || !s->cur || !src || !dst || !tq || s->V1 <= 0 || s->T <= 0 || s->d != mlp_nbr->d || s->d % 4 != 0)
    return LSTEP_ERR_INVALID_ARG;
  if (head < 0 || head >= s->T || len < 0 || len > s->T || append_slot < 0 || append_slot >= s->T) return LSTEP_ERR_INVALID_ARG;
  if (n_queries > 0 && (!query_ids_host || !nbr_out)) return LSTEP_ERR_INVALID_ARG;
  const int d = s->d, t = mlp_nbr->t, T = s->T;
  const StepWs need = carve_step(nullptr, n_ids, n_edges, n_queries, K, d, t, pe_ws_rows(s));
  if (!workspace || workspace_bytes < need.bytes) return LSTEP_ERR_WORKSPACE;
  StepWs w = carve_step(workspace, n_ids, n_edges, n_queries, K, d, t, pe_ws_rows(s));
  cudaStream_t st = as_stream(stream);
  int rc;
  if (!opt.peer) prof_mark(st, kProfStart);
  // a3: filtered history of the batch nodes straight into the current table
  if (n_ids > 0 && !opt.skip_dft) {
    rc = launch_dft_filter(s->ring, (int64_t)T * d, d, head, T, len, d, ids, n_ids, G, s->cur, d, ids, stream, true);
    if (rc != LSTEP_OK) return rc;
    prof_mark(st, kProfDft);
  }
  // a6 gather + a7 edge aggregate: one heterogeneous launch when both exist and the 128-bit paths apply
  // identical query sets (the same device pointer: the eval loop's negative sources ARE the batch's sources under
  // random negative sampling, evaluate_model_utils.py:51-52) are looked up, gathered and pushed through the MLP ONCE;
  // the MLP's epilogue stores the row to every output set that asked for it (OutFan). Only on the paired-MLP path.
  RowIds q{};
  OutFan fan{};
  int n_uniq = 0;
  for (int c = 0; c < n_queries; ++c) {
    if (!query_ids_host[c]) return LSTEP_ERR_INVALID_ARG;
    int u = 0;
    while (u < n_uniq && q.p[u] != query_ids_host[c]) ++u;
    if (u == n_uniq) q.p[n_uniq++] = query_ids_host[c];
    fan.src_of[c] = (signed char)u;
  }
  const bool can_pair = mlp_nbr->ws && mlp_upd->ws && update_push_available(mlp_upd) && pe_mlp_cluster_supports(mlp_nbr) &&
                        (opt.peer ? opt.peer->n_mine : n_ids) > 0 && n_edges > 0;
  const bool dedup = can_pair && n_uniq < n_queries && q_rows > 0;
  if (!dedup) {
    for (int c = 0; c < n_queries; ++c) q.p[c] = query_ids_host[c];
    n_uniq = n_queries;
  } else {
    fan.period = q_rows;
    fan.n_out = n_queries;
  }
  const int64_t rows = (int64_t)n_uniq * q_rows;
  q.period = q_rows;
  // peer group (csrc/peer.cu): phase A covers the batch nodes this rank owns; the step may be issued in two halves
  const PeerPlan* peer = opt.peer;
  if (peer && (!peer->grp || peer->n_mine < 0 || (peer->n_mine > 0 && (!peer->ids_mine || !peer->pos_mine)) || !update_push_available(mlp_upd) ||
               !opt.skip_dft || !opt.skip_append))
    return LSTEP_ERR_INVALID_ARG;
  const int64_t* ids_a = peer ? peer->ids_mine : ids;
  const int64_t n_a = peer ? peer->n_mine : n_ids;
  const bool first_half = !peer || (peer->phases & 2) != 0, second_half = !peer || (peer->phases & 4) != 0;
  bool edges_done = false, phase_a_done = false;
  float* A = nullptr;      // phase A's aggregate rows / result rows inside the update workspace
  float* new_rows = nullptr;
  int64_t ldA = 0;
  int32_t* counters = nullptr;
  // CTA shape of the fused gather: the stand-alone kernels' 192 threads (t time-frequency threads + d/4 table threads).
  // Narrower CTAs (all resident beside the DFT filter at once) gave no gain: the gather is not bound by residency, its
  // cosines are ~9 us of issue-bound work either way.
  const int t_pad = (int)align_up((size_t)t, 32);
  const int threads = (int)align_up((size_t)t_pad + d / 4, 32);
  const bool vec_ok = d % 4 == 0 && w.lda % 4 == 0 && reinterpret_cast<uintptr_t>(s->cur) % 16 == 0 && threads <= 512;
  if (first_half && rows > 0 && n_a > 0 && n_edges > 0 && vec_ok && t == mlp_upd->t && d == mlp_upd->d) {
    update_ws_phase_a(w.update, n_ids, n_edges, K, d, t, pe_ws_rows(s), &A, &ldA, &counters, &new_rows);
    const int64_t cap = (int64_t)num_sms() * 16;
    // more query rows than one launch has CTAs for (B = 2000): one wave of CTAs with a look-ahead lookup warp each (gather_pipe)
    const bool piped = tuning().gather_pipe != 0 && rows > cap && threads + 32 <= 512;
    const int threads_l = piped ? threads + 32 : threads;
    const int64_t cap_q = piped ? (int64_t)num_sms() * (2048 / threads_l) : cap;
    const int grid_q = (int)(rows < cap_q ? rows : cap_q), grid_e = (int)(n_a < cap ? n_a : cap);
    const size_t smem = std::max((size_t)K * 8 * (piped ? 2 : 1), (size_t)threads_l * kSegPerThread * 8 + 32 * 4);
    if (smem <= 48 * 1024) {
      LookupArgs lk{csr->indptr, csr->nbr, csr->t, csr->num_rows, q, err_flag};
      launch_k(gather_ab_kernel, dim3((unsigned)(grid_q + grid_e)), dim3(threads_l), smem, st, s->cur, tq_q, rows, K, mlp_nbr->tw, d, t, t_pad,
               w.S, w.lda, q_rows, lk, grid_q, ids_a, n_a, src, dst, tq, n_edges, (float)current_time, mlp_upd->tw, A, ldA, counters,
               piped ? threads : 0);
      if ((rc = check_launch("gather_ab")) != LSTEP_OK) return rc;
      prof_mark(st, kProfGather);
      edges_done = true;
    }
  }
  if (first_half && rows > 0) {
    if (!edges_done) {
      rc = launch_nbr_lookup_aggregate(csr, q, s->cur, tq_q, rows, K, mlp_nbr->tw, d, t, w.S, w.lda, err_flag, st);
      if (rc != LSTEP_OK) return rc;
    }
    // the neighbourhood MLP and phase A's MLP in ONE launch when they fit one round of clusters: neither writes the
    // table then (phase A's rows go to new_rows and are applied by the push kernel), so they need no order
    if (edges_done && mlp_nbr->ws && mlp_upd->ws && update_push_available(mlp_upd)) {
      RowIds ida{};
      ida.p[0] = ids_a;
      ida.period = 0;
      rc = launch_pe_mlp_cluster_pair(s->cur, w.S, w.lda, q, rows, mlp_nbr, nbr_out, d, A, ldA, ida, n_a, mlp_upd, new_rows, d, st,
                                      /*late_trigger=*/true, s->V1, dedup ? &fan : nullptr);
      if (rc == LSTEP_OK) {
        phase_a_done = true;
        prof_mark(st, kProfMlpPair);
      } else if (rc != LSTEP_ERR_UNSUPPORTED)
        return rc;
    }
    if (!phase_a_done) {
      if (dedup)  // the pair did not fit one round of clusters: the cluster kernel alone walks the tiles, same fan-out
        rc = launch_pe_mlp_cluster(w.S, w.lda, s->cur, q, rows, rows, nullptr, mlp_nbr, nbr_out, d, nullptr, nullptr, nullptr, st, false, nullptr, 0,
                                   &fan, s->V1);
      else
        rc = launch_pe_mlp(w.S, w.lda, s->cur, q, rows, rows, nullptr, mlp_nbr, nbr_out, d, nullptr, st);
      if (rc != LSTEP_OK) return rc;
    }
  }
  PushOwner own{};
  if (peer) {
    if (first_half) {
      // phase A's rows of the owned batch nodes (stand-alone launches when the paired launch did not apply), then into every
      // rank's new_rows buffer at the node's position in the batch's id list, then barrier 2 is announced
      if (!phase_a_done) {
        rc = launch_phase_a_to_new_rows(s->cur, w.update, n_ids, n_edges, K, pe_ws_rows(s), ids_a, n_a, src, dst, tq, n_edges, (float)current_time,
                                        mlp_upd, edges_done, st);
        if (rc != LSTEP_OK) return rc;
      }
      update_ws_phase_a(w.update, n_ids, n_edges, K, d, t, pe_ws_rows(s), &A, &ldA, &counters, &new_rows);
      if (n_a > 0 && (rc = peer_rows_bcast(new_rows, n_a, d, peer->pos_mine, peer->grp, 1, st)) != LSTEP_OK) return rc;
      if (!second_half && (rc = peer_signal(peer->grp, peer->epoch2, st)) != LSTEP_OK) return rc;  // (else the wait launch announces)
      prof_mark(st, kProfBcast);
    }
    if (!second_half) return LSTEP_OK;
    if ((rc = peer_wait(peer->grp, peer->epoch2, peer->timeout_ms, err_flag, st, first_half)) != LSTEP_OK) return rc;
    prof_mark(st, kProfWait2);
    edges_done = phase_a_done = true;
    own.mul = peer->grp->world;
    own.add = peer->grp->rank;
    own.new_rows = peer->grp->new_rows[peer->grp->rank];
  }
  // a7 + a8
  static std::atomic<int> g_stamp{0};
  int stamp = ++g_stamp;
  if (stamp <= 0) {  // wrapped: restart (a stale equal value only costs a redundant row copy)
    g_stamp = 1;
    stamp = 1;
  }
  if (opt.stamp_out) *opt.stamp_out = stamp;
  int32_t* dirty = nullptr;
  rc = update_pe_impl(s->cur, pe_ws_rows(s), csr, ids, n_ids, src, dst, tq, n_edges, current_time, K, mlp_upd, w.update, w.update_bytes,
                      err_flag, stream, edges_done, opt.skip_append ? nullptr : &dirty, stamp, phase_a_done,
                      s->ring + (int64_t)append_slot * d, (int64_t)T * d, peer ? &own : nullptr);
  if (rc != LSTEP_OK) return rc;
  // 2 CTAs per SM: the append is resident (copying, then waiting for the phase-B MLP) while the NEXT step's DFT filter
  // wants to become resident and prefetch — it must leave thread slots and shared memory for it
  if (opt.skip_append) return LSTEP_OK;
  launch_k(ring_append_kernel, dim3(num_sms() * 2), dim3(256), 0, st, s->cur, s->ring, s->V1, T, d, append_slot, 1, 0, dirty, stamp);
  prof_mark(st, kProfAppend);
  return check_launch("ring_append");
}
}  // namespace lstep

extern "C" int lstep_pe_step(const lstep_pe_stream* s, const lstep_csr* csr, int64_t lo, int64_t n_edges,
                             const int64_t* ids, int64_t n_ids, double current_time, int head, int len, int append_slot,
                             const float* G, const int64_t* const* query_ids_host, int n_queries, float* nbr_out, int K,
                             const lstep_pe_mlp* mlp_nbr, const lstep_pe_mlp* mlp_upd, void* workspace,
                             size_t workspace_bytes, uint32_t* err_flag, void* stream) {
  if (!s || !s->src || !s->dst || !s->t || lo < 0) return LSTEP_ERR_INVALID_ARG;
  return pe_step_core(s, csr, s->src + lo, s->dst + lo, s->t + lo, n_edges, ids, n_ids, current_time, head, len, append_slot, G,
                      query_ids_host, n_queries, nbr_out, K, mlp_nbr, mlp_upd, workspace, workspace_bytes, err_flag, stream);
}

/* A run of consecutive batches of the RESIDENT stream in one call (steady state: full history, one filter G): step i covers
 * edges [lo[i], lo[i] + n_edges[i]), batch nodes ids + ids_off[i] .. ids_off[i+1], update time tmax[i]; query set c of step i
 * is query_ids_host[c] + q_off[i] (n_edges[i] ids each); its outputs go to nbr_out + i * out_step_stride floats (0: every step
 * overwrites the same buffer). The ring position advances by one slot per step; *head_io is updated. The host only pays the
 * launches (6 per step), so the device is never waiting for the interpreter. */
extern "C" int lstep_pe_steps(const lstep_pe_stream* s, const lstep_csr* csr, int64_t n_steps, const int64_t* lo_host,
                              const int64_t* n_edges_host, const int64_t* ids, const int64_t* ids_off_host, const double* tmax_host,
                              int* head_io, int* len_io, const float* G, const int64_t* const* query_ids_host,
                              const int64_t* q_off_host, int n_queries, float* nbr_out, int64_t out_step_stride, int K,
                              const lstep_pe_mlp* mlp_nbr, const lstep_pe_mlp* mlp_upd, void* workspace, size_t workspace_bytes,
                              uint32_t* err_flag, void* stream) {
  if (!s || !s->src || !s->dst || !s->t || n_steps < 0 || !lo_host || !n_edges_host || !ids || !ids_off_host || !tmax_host || !head_io ||
      !len_io || n_queries < 0 || n_queries > 8 || (n_queries > 0 && (!query_ids_host || !q_off_host)))
    return LSTEP_ERR_INVALID_ARG;
  const int T = s->T;
  if (*len_io != T) return LSTEP_ERR_INVALID_ARG;  // steady state only: while the ring fills the filter changes every step
  int head = *head_io;
  for (int64_t i = 0; i < n_steps; ++i) {
    const int64_t* q[8] = {};
    for (int c = 0; c < n_queries; ++c) q[c] = query_ids_host[c] + q_off_host[i];
    const int64_t lo = lo_host[i];
    if (lo < 0) return LSTEP_ERR_INVALID_ARG;
    const int rc = pe_step_core(s, csr, s->src + lo, s->dst + lo, s->t + lo, n_edges_host[i], ids + ids_off_host[i],
                                ids_off_host[i + 1] - ids_off_host[i], tmax_host[i], head, T, head, G, q, n_queries,
                                nbr_out ? nbr_out + i * out_step_stride : nullptr, K, mlp_nbr, mlp_upd, workspace, workspace_bytes, err_flag,
                                stream);
    if (rc != LSTEP_OK) {
      *head_io = head;
      return rc;
    }
    head = (head + 1) % T;
  }
  *head_io = head;
  return LSTEP_OK;
}

/* One rank's share of a step on a node-id sharded group with a replicated table and CSR (l-step_b200/shard.py::ReplicatedTableRank):
 * everything of lstep_pe_step EXCEPT the DFT filter (the caller filters the batch nodes whose history it owns, all-gathers the
 * filtered rows and scatters them into s->cur before this call) and the ring append (the caller appends the rows it owns with
 * lstep_ring_copy_rows). The a6 query sets cover the edges [q_off, q_off + q_rows) of the batch only — this rank's share —
 * query_ids_host[c] pointing at the first of those ids; outputs [n_queries, q_rows, d]. update_pe runs in full on every rank
 * (identical inputs, deterministic kernels: the replicas of the table stay bit-identical without any exchange). */
extern "C" int lstep_pe_step_sharded(const lstep_pe_stream* s, const lstep_csr* csr, int64_t lo, int64_t n_edges, const int64_t* ids,
                                     int64_t n_ids, double current_time, const int64_t* const* query_ids_host, int n_queries,
                                     int64_t q_off, int64_t q_rows, float* nbr_out, int K, const lstep_pe_mlp* mlp_nbr,
                                     const lstep_pe_mlp* mlp_upd, void* workspace, size_t workspace_bytes, uint32_t* err_flag,
                                     void* stream) {
  if (!s || !s->src || !s->dst || !s->t || lo < 0 || q_rows < 0) return LSTEP_ERR_INVALID_ARG;
  StepOpts opt;
  opt.skip_dft = opt.skip_append = true;
  opt.q_off = q_off;
  opt.q_rows = q_rows;
  return pe_step_core_ex(s, csr, s->src + lo, s->dst + lo, s->t + lo, n_edges, ids, n_ids, current_time, 0, 0, 0, nullptr, query_ids_host,
                         q_rows > 0 ? n_queries : 0, nbr_out, K, mlp_nbr, mlp_upd, workspace, workspace_bytes, err_flag, stream, opt);
}

LSTEP_TIMELINE_DEFINE(step)
