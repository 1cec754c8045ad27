// K2 (scatter side) + K4 — LSTEP.update_pe (/root/reference/models/LSTEP.py:268-341) on the
// caller's PE table, in place, with the event order of the reference:
//
//   phase A   agg[v] = sum over batch edges of [pe[other endpoint] || tf]   (old table)
//             pe[ids] <- pe[ids] + tanh(self(pe[ids]) + mlp(agg[ids]))
//   pe[0] = 0
//   phase B   sample most-recent-K neighbours of (ids[i], times[i]);
//             agg2[u] = sum over slots (i,k) with nbr[i,k]==u of [pe[ids[i]] || tf]  (phase-A table)
//             pe[U] <- pe[U] + tanh(mlp(agg2[U])),  U = distinct sampled ids (0 included if padded)
//
// The reference scatters into two zeroed [V1, d+t] buffers (10.9 GB at 10 M nodes). Here no V1-sized float
// buffer exists and every destination row is reduced without float atomics:
//   * phase A (pull): one CTA per batch node scans the 2B endpoint ids (L2 resident), compacts its matches in
//     edge order (source side first, as the two scatter calls do) and adds the rows in exactly the reference's
//     order (body: csrc/gather_bodies.cuh);
//   * phase B, push form (default, csrc/update_push.cu): lookup + claim of a compact accumulator row per distinct
//     destination + exact 32.32 fixed-point integer atomics where a contribution lands, in one kernel; the MLP
//     (csrc/mlp_cluster.cu) reads the accumulator rows;
//   * phase B, pull form (this file; used by the node-id sharded path, which ships float partial rows between
//     ranks, and when the cluster MLP does not cover the shape; LSTEP_PHASEB_PULL=1): an inverse index
//     (destination -> slots) is built with integer atomics on a per-node counter map (count / scan / fill), one
//     warp per destination sorts its slot list (ascending flat index = the reference's add order) and reduces it;
//     longer lists (hubs) are summed in 32.32 fixed point (range: fixed_point_bound, csrc/common.cuh). The padding row 0 collects every empty slot —
//     thousands of contributions at B=200 — and is reduced by a two-level tree.
// All gathers of a phase finish (kernel boundary) before its rows are written, which is what
// makes the in-place write-back safe for nodes that are both source and destination (Q6).
#include <cstdlib>

#include "common.cuh"
#include "mlp_job.cuh"
#include "gather_bodies.cuh"

namespace lstep {

int launch_pe_mlp(const float* A, int64_t lda, const float* pe, RowIds base_ids, int64_t n_rows, int64_t expected_rows,
                  const int32_t* n_rows_dev, const lstep_pe_mlp* m, float* out, int64_t out_stride, float* pe_inplace,
                  cudaStream_t st, bool late_trigger = false);
int launch_sample_count(const lstep_csr* csr, const int64_t* q_node, const double* q_time, int64_t n_rows, int64_t n_valid,
                        int K, int32_t* out_nbr, float* out_t, uint32_t* err_flag, PhaseBHook hook, void* stream);
int launch_phaseB_push(const lstep_csr* csr, const int64_t* ids, const double* q_time, int64_t n_ids, int64_t n_valid, int K,
                       float* pe, int d, int t, const float* tw, float tc, int32_t* claim_of, int64_t* U, int32_t* counters,
                       unsigned long long* acc, int32_t* dirty, int stamp, const float* new_rows, uint32_t* err_flag, cudaStream_t st,
                       unsigned long long* row0_part, int own_mul = 1, int own_add = 0);

constexpr int kRow0Parts = 64;
constexpr int kHubLen = 4;     // a warp reduces a destination's slot list serially (~430 dependent instructions per
                              // slot), so lists longer than this are split into chunk tasks spread over the GPU
constexpr int kChunkLog2 = 2;  // slots per chunk task = 4

struct UpdateWs {
  int32_t* cnt_of;   // [pe_rows]  zero between calls
  int32_t* slot_of;  // [pe_rows]  pull form: slot index of a destination; push form: stamp of the last step whose phase B changed the row
  int32_t* claim_of; // [pe_rows]  zero between calls (push form of phase B: 0 free, -1 being set up, j+1 = accumulator row j)
  unsigned long long* push_row0;  // [kPushRow0Parts][kPushRow0Cols] zero between calls: partial sums of the padding row (push form)
  unsigned long long* hub_acc;  // [#long lists][d+t] 32.32 fixed-point accumulators (zeroed per call by the scan kernel)
  int32_t* counters; // [8]: 0=M, 1=has_zero, 2=n_dest, 3=n_hubs, 4=n_hub_tasks
  int32_t* src32;    // [E]
  int32_t* dst32;    // [E]
  float* dtA;        // [E]
  int32_t* nbrB;     // [N*K]
  float* ntB;        // [N*K]
  int32_t* rank;     // [N*K]
  int32_t* list;     // [N*K]
  int64_t* U;        // [N*K+1]
  int32_t* off;      // [N*K+2]
  int32_t* hubs;     // [N*K/32+1] destinations with more than 32 slots
  int32_t* hub_remaining;  // chunk tasks of the hub still running
  int32_t* task_hub;       // [2*N*K/32+2] hub index of a chunk task
  int32_t* task_chunk;     // [2*N*K/32+2] chunk index of a chunk task
  float* row0_part;  // [kRow0Parts*d]
  float* A;          // [max(N, N*K+1)][lda], lda = d+t rounded up to 4 floats
  unsigned long long* push_acc;  // [N*K+1][d+t] 32.32 fixed-point accumulator rows of the push form
  float* new_rows;   // [N][d] phase A's result rows when its MLP does not write the table itself (streaming step)
  int64_t lda;
  size_t bytes;
};

static UpdateWs carve(void* base, int64_t n_ids, int64_t n_edges, int K, int d, int t, int64_t pe_rows) {
  UpdateWs w;
  size_t o = 0;
  auto take = [&](size_t bytes) {
    void* p = base ? static_cast<char*>(base) + o : nullptr;
    o = align_up(o + bytes, 256);
    return p;
  };
  const size_t nk = (size_t)n_ids * K;
  w.cnt_of = (int32_t*)take(sizeof(int32_t) * pe_rows);
  w.slot_of = (int32_t*)take(sizeof(int32_t) * pe_rows);
  w.claim_of = (int32_t*)take(sizeof(int32_t) * pe_rows);
  w.push_row0 = (unsigned long long*)take(kPushRow0Bytes);
  w.counters = (int32_t*)take(sizeof(int32_t) * 8);
  w.src32 = (int32_t*)take(sizeof(int32_t) * (n_edges + 4));
  w.dst32 = (int32_t*)take(sizeof(int32_t) * (n_edges + 4));
  w.dtA = (float*)take(sizeof(float) * (n_edges + 4));
  w.nbrB = (int32_t*)take(sizeof(int32_t) * nk);
  w.ntB = (float*)take(sizeof(float) * nk);
  w.rank = (int32_t*)take(sizeof(int32_t) * nk);
  w.list = (int32_t*)take(sizeof(int32_t) * nk);
  w.U = (int64_t*)take(sizeof(int64_t) * (nk + 1));
  w.off = (int32_t*)take(sizeof(int32_t) * (nk + 2));
  w.hubs = (int32_t*)take(sizeof(int32_t) * (nk / (kHubLen + 1) + 2));
  w.hub_remaining = (int32_t*)take(sizeof(int32_t) * (nk / (kHubLen + 1) + 2));
  w.task_hub = (int32_t*)take(sizeof(int32_t) * ((nk >> kChunkLog2) + nk / (kHubLen + 1) + 4));
  w.task_chunk = (int32_t*)take(sizeof(int32_t) * ((nk >> kChunkLog2) + nk / (kHubLen + 1) + 4));
  w.hub_acc = (unsigned long long*)take(sizeof(unsigned long long) * (nk / (kHubLen + 1) + 1) * (size_t)(d + t));
  w.row0_part = (float*)take(sizeof(float) * kRow0Parts * d);
  const size_t rowsA = nk + 1 > (size_t)n_ids ? nk + 1 : (size_t)n_ids;
  w.lda = (int64_t)align_up((size_t)(d + t), 4);
  w.A = (float*)take(sizeof(float) * rowsA * w.lda);
  // own storage: the push kernel sets accumulator rows up while the phase-A MLP is still reading A
  w.push_acc = (unsigned long long*)take(sizeof(unsigned long long) * (nk + 1) * (size_t)(d + t));
  w.new_rows = (float*)take(sizeof(float) * (size_t)n_ids * d);
  w.bytes = o;
  return w;
}

// ---------------------------------------------------------------------------------------------
// phase A edge aggregate (body: edge_aggregate_rows, csrc/gather_bodies.cuh)
__global__ void __launch_bounds__(512) edge_aggregate_kernel(const float* __restrict__ pe, const int64_t* __restrict__ ids, int64_t n_ids,
                                                             const int64_t* __restrict__ src, const int64_t* __restrict__ dst,
                                                             const double* __restrict__ times, int64_t n_edges, float tc,
                                                             const float* __restrict__ tw, int d, int t, int t_pad,
                                                             float* __restrict__ A, int64_t lda, int32_t* __restrict__ counters) {
  pdl_launch_dependents();
  pdl_wait();
  edge_aggregate_rows(blockIdx.x, gridDim.x, blockIdx.x == 0, false, pe, ids, n_ids, src, dst, times, n_edges, tc, tw, d, t, t_pad, A, lda, counters);
}

// ---------------------------------------------------------------------------------------------
// step 2 (one CTA): offsets by exclusive scan over U order; slot map; counter map reset; hub list

// Block 0 scans (and, for small batches, also fills the slot lists); blocks 1.. compute the per-part
// partial sums of the padding row.
__global__ void __launch_bounds__(1024) phaseB_scan_kernel(int32_t* __restrict__ cnt_of, int32_t* __restrict__ slot_of,
                                                           int64_t* __restrict__ U, int32_t* __restrict__ off,
                                                           int32_t* __restrict__ hubs, int32_t* __restrict__ hub_remaining,
                                                           int32_t* __restrict__ task_hub, int32_t* __restrict__ task_chunk,
                                                           unsigned long long* __restrict__ hub_acc, int in1,
                                                           int32_t* __restrict__ counters,
                                                           const int32_t* __restrict__ nbrB, int64_t total, int K,
                                                           const int32_t* __restrict__ rank, int32_t* __restrict__ list,
                                                           int fill_here, const float* __restrict__ pe,
                                                           const int64_t* __restrict__ ids, int64_t n_ids, int d,
                                                           float* __restrict__ row0_part) {
  pdl_launch_dependents();
  pdl_wait();
  if (blockIdx.x > 0) {
    {  // accumulator rows of this call's long lists start from zero: at most min(M, N*K/(kHubLen+1)) lists are long
      const int64_t cap = min((int64_t)ld_dep(counters + 0), total / (kHubLen + 1) + 1) * in1;
      ulonglong2* z = reinterpret_cast<ulonglong2*>(hub_acc);
      for (int64_t i = (int64_t)(blockIdx.x - 1) * blockDim.x + threadIdx.x; i < (cap + 1) / 2; i += (int64_t)(gridDim.x - 1) * blockDim.x)
        z[i] = make_ulonglong2(0ull, 0ull);
    }
    if (ld_dep(counters + 1) == 0) return;
    const int part = blockIdx.x - 1;
    for (int c = threadIdx.x; c < d; c += blockDim.x) {
      float acc = 0.f;
      for (int64_t n = part; n < n_ids; n += kRow0Parts) {
        int z = 0;
        for (int k = 0; k < K; ++k) z += (ld_dep(nbrB + n * K + k) == 0);
        if (z) acc = fmaf((float)z, ld_dep(pe + ids[n] * (int64_t)d + c), acc);
      }
      row0_part[part * d + c] = acc;
    }
    return;
  }
  __shared__ int s_warp[32];
  const int M = ld_dep(counters + 0);
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int chunk = (M + blockDim.x - 1) / blockDim.x;
  const int lo = min(M, tid * chunk), hi = min(M, lo + chunk);
  int sum = 0;
  for (int s = lo; s < hi; ++s) sum += ld_dep(cnt_of + ld_dep(U + s));
  int incl = sum;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int v = __shfl_up_sync(kFull, incl, o);
    if (lane >= o) incl += v;
  }
  if (lane == 31) s_warp[wid] = incl;
  __syncthreads();
  if (wid == 0) {
    int v = s_warp[lane], iv = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int x = __shfl_up_sync(kFull, iv, o);
      if (lane >= o) iv += x;
    }
    s_warp[lane] = iv - v;
    if (lane == 31) off[M] = iv;  // total number of non-padding slots
  }
  __syncthreads();
  int run = s_warp[wid] + incl - sum;
  for (int s = lo; s < hi; ++s) {
    const int64_t u = ld_dep(U + s);
    const int deg = ld_dep(cnt_of + u);
    off[s] = run;
    run += deg;
    cnt_of[u] = 0;  // restore the all-zero invariant
    slot_of[u] = s;
    if (deg > kHubLen) {  // long list: reduced by ceil(deg/8) chunk tasks spread over the grid
      const int h = atomicAdd(counters + 3, 1);
      const int nch = (deg + (1 << kChunkLog2) - 1) >> kChunkLog2;
      const int t0 = atomicAdd(counters + 4, nch);
      hubs[h] = s;
      hub_remaining[h] = nch;
      for (int c = 0; c < nch; ++c) {
        task_hub[t0 + c] = h;
        task_chunk[t0 + c] = c;
      }
    }
  }
  if (tid == 0) {
    const int hz = ld_dep(counters + 1);
    counters[2] = M + hz;
    if (hz) U[M] = 0;
  }
  __syncthreads();  // off[] / slot_of[] / the hub list written above are visible to the whole CTA
  if (fill_here) {
    for (int64_t i = tid; i < total; i += blockDim.x) {
      const int32_t u = ld_dep(nbrB + i);
      if (u > 0) list[off[slot_of[u]] + ld_dep(rank + i)] = (int32_t)i;  // off / slot_of: written by this CTA above
    }
  }
}

// step 3 (large batches only): fill slot lists
__global__ void __launch_bounds__(256) phaseB_fill_kernel(const int32_t* __restrict__ nbrB, int64_t total,
                                                          const int32_t* __restrict__ slot_of,
                                                          const int32_t* __restrict__ off,
                                                          const int32_t* __restrict__ rank, int32_t* __restrict__ list) {
  pdl_launch_dependents();
  pdl_wait();
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < total) {
    const int32_t u = ld_dep(nbrB + i);
    if (u > 0) list[ld_dep(off + ld_dep(slot_of + u)) + ld_dep(rank + i)] = (int32_t)i;
  }
}

// One list entry = slot i = (row n, column k): contributes [pe[ids[n]] || cos((tc - nt[i]) * w)].
// The per-entry metadata (source row pointer, dt) is resolved for 32 entries at once (one lane each),
// so the dependent index loads are paid once per chunk, not once per entry; the rows of 4 consecutive
// entries are then loaded together before they are added, in list order.
template <int DVPL, int TFPL>
__device__ __forceinline__ void accumulate_chunk(const float* my_row, float my_dt, int m, int lane, int dvec, int t,
                                                 const float (&w)[TFPL], float4 (&acc)[DVPL], float (&acc_tf)[TFPL]) {
  for (int j0 = 0; j0 < m; j0 += 4) {
    const float4* row[4];
    float dt[4];
    float4 v[4][DVPL];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int j = min(j0 + u, m - 1);
      row[u] = reinterpret_cast<const float4*>(reinterpret_cast<const float*>(__shfl_sync(kFull, (unsigned long long)my_row, j)));
      dt[u] = __shfl_sync(kFull, my_dt, j);
    }
#pragma unroll
    for (int u = 0; u < 4; ++u)
#pragma unroll
      for (int q = 0; q < DVPL; ++q)
        if (lane + 32 * q < dvec) v[u][q] = ld_dep(row[u] + lane + 32 * q);
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      if (j0 + u < m) {
#pragma unroll
        for (int q = 0; q < DVPL; ++q)
          if (lane + 32 * q < dvec) {
            acc[q].x += v[u][q].x;
            acc[q].y += v[u][q].y;
            acc[q].z += v[u][q].z;
            acc[q].w += v[u][q].w;
          }
#pragma unroll
        for (int q = 0; q < TFPL; ++q)
          if (lane + 32 * q < t) acc_tf[q] += time_feature(dt[u], w[q]);
      }
    }
  }
}

// step 4: blocks [0, warp_blocks): one warp per destination with a short list (sorted: fp32 adds in the
// reference's flat order). Blocks [warp_blocks, warp_blocks + hub_blocks): hub chunk tasks — every 32-slot
// chunk of a hub's list is an independent task taken by one warp anywhere on the GPU, accumulated in 32.32
// fixed point and added to the hub's accumulator row with 64-bit integer atomics (exact, so neither the
// arrival order of the list nor the order of the tasks matters: reproducible run to run); the warp that
// finishes a hub's last task converts the row to fp32 and re-zeroes the accumulator. One CTA per hub would
// serialise ~430 dependent instructions per slot on one SM (measured: 29 us for a 225-slot hub). Last block:
// finishes the padding row.
template <int DVPL, int TFPL>
__global__ void __launch_bounds__(256, DVPL <= 2 ? 2 : 1) phaseB_gather_kernel(
    const float* __restrict__ pe, const int64_t* __restrict__ ids, int K, const float* __restrict__ ntB,
    const int32_t* __restrict__ off, const int32_t* __restrict__ list, const int32_t* __restrict__ hubs,
    int32_t* __restrict__ hub_remaining, const int32_t* __restrict__ task_hub, const int32_t* __restrict__ task_chunk,
    unsigned long long* __restrict__ hub_acc, const int32_t* __restrict__ counters, float tc, const float* __restrict__ tw, int d,
    int t, const float* __restrict__ row0_part, float* __restrict__ A, int64_t lda, int warp_blocks, int hub_blocks, float fx_bound,
    uint32_t* err_flag) {
  pdl_launch_dependents();
  pdl_wait();
  const int in1 = d + t;
  const int M = ld_dep(counters + 0);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int nw = blockDim.x >> 5;
  // the grid is sized for the worst case (every slot a distinct destination); surplus CTAs leave at once
  if ((int)blockIdx.x < warp_blocks && (int)blockIdx.x * nw >= M) return;
  const int n_tasks = ld_dep(counters + 4);
  if ((int)blockIdx.x >= warp_blocks && (int)blockIdx.x < warp_blocks + hub_blocks && ((int)blockIdx.x - warp_blocks) * nw >= n_tasks) return;
  const int dvec = d >> 2;
  float w[TFPL];
#pragma unroll
  for (int q = 0; q < TFPL; ++q) w[q] = (lane + 32 * q < t) ? tw[lane + 32 * q] : 0.f;

  if ((int)blockIdx.x == warp_blocks + hub_blocks) {  // ---- padding row
    if (ld_dep(counters + 1)) {
      for (int c = threadIdx.x; c < in1; c += blockDim.x) {
        float acc = 0.f;
        if (c < d)
          for (int p = 0; p < kRow0Parts; ++p) acc += ld_dep(row0_part + p * d + c);
        A[(int64_t)M * lda + c] = acc;  // time features of padded slots are zeroed (LSTEP.py:316)
      }
    }
    return;
  }

  float4 acc[DVPL];
  float acc_tf[TFPL];
#pragma unroll
  for (int q = 0; q < DVPL; ++q) acc[q] = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
  for (int q = 0; q < TFPL; ++q) acc_tf[q] = 0.f;

  if ((int)blockIdx.x < warp_blocks) {  // ---- short lists
    const int s = blockIdx.x * nw + wid;
    if (s >= M) return;
    const int o0 = ld_dep(off + s), len = ld_dep(off + s + 1) - o0;
    if (len > kHubLen) return;  // reduced by hub chunk tasks
    int e = (lane < len) ? ld_dep(list + o0 + lane) : 0x7fffffff;
    // bitonic sort ascending across the warp: restores flat-index (= reference add) order
#pragma unroll
    for (int k = 2; k <= 32; k <<= 1) {
#pragma unroll
      for (int j = k >> 1; j > 0; j >>= 1) {
        const int o = __shfl_xor_sync(kFull, e, j);
        const bool up = ((lane & k) == 0);
        const bool lower = ((lane & j) == 0);
        e = (lower == up) ? min(e, o) : max(e, o);
      }
    }
    const float* my_row = pe;
    float my_dt = 0.f;
    if (lane < len) {
      my_row = pe + ids[e / K] * (int64_t)d;
      my_dt = tc - ld_dep(ntB + e);  // fp32 - fp32 (LSTEP.py:314)
    }
    accumulate_chunk<DVPL, TFPL>(my_row, my_dt, len, lane, dvec, t, w, acc, acc_tf);
    float* arow = A + (int64_t)s * lda;
#pragma unroll
    for (int q = 0; q < DVPL; ++q)
      if (lane + 32 * q < dvec) reinterpret_cast<float4*>(arow)[lane + 32 * q] = acc[q];
#pragma unroll
    for (int q = 0; q < TFPL; ++q)
      if (lane + 32 * q < t) arow[d + lane + 32 * q] = acc_tf[q];
    return;
  }

  // ---- hub chunk tasks (fixed point: a contribution outside fixed_point_bound, csrc/common.cuh, raises the range flag)
  constexpr float kScale = 4294967296.f;           // 2^32
  constexpr float kInv = 2.3283064365386963e-10f;  // 2^-32
  bool bad = false;
  for (int task = ((int)blockIdx.x - warp_blocks) * nw + wid; task < n_tasks; task += hub_blocks * nw) {
    const int h = ld_dep(task_hub + task), c0 = ld_dep(task_chunk + task) << kChunkLog2;
    const int s = ld_dep(hubs + h);
    const int o0 = ld_dep(off + s), len = ld_dep(off + s + 1) - o0;
    const int m = min(1 << kChunkLog2, len - c0);
    const float* my_row = pe;
    float my_dt = 0.f;
    if (lane < m) {
      const int e = ld_dep(list + o0 + c0 + lane);
      my_row = pe + ids[e / K] * (int64_t)d;
      my_dt = tc - ld_dep(ntB + e);
    }
    long long facc[DVPL][4], ftf[TFPL];
#pragma unroll
    for (int q = 0; q < DVPL; ++q) facc[q][0] = facc[q][1] = facc[q][2] = facc[q][3] = 0;
#pragma unroll
    for (int q = 0; q < TFPL; ++q) ftf[q] = 0;
    for (int j0 = 0; j0 < m; j0 += 4) {
      const float4* row[4];
      float dt[4];
      float4 v[4][DVPL];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int j = min(j0 + u, m - 1);
        row[u] = reinterpret_cast<const float4*>(reinterpret_cast<const float*>(__shfl_sync(kFull, (unsigned long long)my_row, j)));
        dt[u] = __shfl_sync(kFull, my_dt, j);
      }
#pragma unroll
      for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int q = 0; q < DVPL; ++q)
          if (lane + 32 * q < dvec) v[u][q] = ld_dep(row[u] + lane + 32 * q);
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        if (j0 + u < m) {
#pragma unroll
          for (int q = 0; q < DVPL; ++q)
            if (lane + 32 * q < dvec) {
              bad |= !(fabsf(v[u][q].x) < fx_bound) || !(fabsf(v[u][q].y) < fx_bound) || !(fabsf(v[u][q].z) < fx_bound) ||
                     !(fabsf(v[u][q].w) < fx_bound);
              facc[q][0] += __float2ll_rn(v[u][q].x * kScale);
              facc[q][1] += __float2ll_rn(v[u][q].y * kScale);
              facc[q][2] += __float2ll_rn(v[u][q].z * kScale);
              facc[q][3] += __float2ll_rn(v[u][q].w * kScale);
            }
#pragma unroll
          for (int q = 0; q < TFPL; ++q)
            if (lane + 32 * q < t) {
              const float f = time_feature(dt[u], w[q]);
              bad |= !(fabsf(f) <= 1.f);
              ftf[q] += __float2ll_rn(f * kScale);
            }
        }
      }
    }
    unsigned long long* hrow = hub_acc + (size_t)h * in1;
#pragma unroll
    for (int q = 0; q < DVPL; ++q) {
      const int cv = lane + 32 * q;
      if (cv < dvec) {
#pragma unroll
        for (int x = 0; x < 4; ++x) atomicAdd(hrow + 4 * cv + x, (unsigned long long)facc[q][x]);
      }
    }
#pragma unroll
    for (int q = 0; q < TFPL; ++q)
      if (lane + 32 * q < t) atomicAdd(hrow + d + lane + 32 * q, (unsigned long long)ftf[q]);
    __threadfence();
    int last = 0;
    if (lane == 0) last = (atomicSub(hub_remaining + h, 1) == 1);
    last = __shfl_sync(kFull, last, 0);
    if (last) {  // every task of this list has added its part: convert the row
      __threadfence();
      float* arow = A + (int64_t)s * lda;
      for (int c = lane; c < in1; c += 32) arow[c] = (float)(long long)__ldcg(hrow + c) * kInv;
    }
  }
  if (__any_sync(kFull, bad) && lane == 0 && err_flag) atomicOr(err_flag, LSTEP_FLAG_FIXED_POINT_RANGE);
}

}  // namespace lstep

using namespace lstep;

extern "C" size_t lstep_update_pe_workspace_bytes(int64_t n_ids, int64_t n_edges, int K, int d, int t,
                                                  int64_t pe_rows) {
  if (n_ids < 0 || n_edges < 0 || K <= 0 || d <= 0 || t < 0 || pe_rows <= 0) return 0;
  return carve(nullptr, n_ids, n_edges, K, d, t, pe_rows).bytes;
}

extern "C" int lstep_update_pe_workspace_init(void* workspace, size_t workspace_bytes, int64_t pe_rows, void* stream) {
  // the per-node maps at the head of the workspace (counter, slot, claim) must be zero on entry; every call
  // leaves them zero
  const size_t head = 3 * align_up(sizeof(int32_t) * (size_t)pe_rows, 256) + kPushRow0Bytes;
  if (!workspace || pe_rows <= 0 || workspace_bytes < head) return LSTEP_ERR_INVALID_ARG;
  cudaError_t e = cudaMemsetAsync(workspace, 0, head, as_stream(stream));
  if (e != cudaSuccess) {
    set_cuda_error(e, "workspace_init");
    return LSTEP_ERR_CUDA;
  }
  return LSTEP_OK;
}

namespace lstep {

static int check_update_args(const float* pe, int64_t pe_rows, const lstep_pe_mlp* mlp, int64_t n_ids, int64_t n_edges, int K,
                             void* workspace, size_t workspace_bytes) {
  if (!pe || !mlp || pe_rows <= 0 || n_ids < 0 || n_edges < 0 || K <= 0) return LSTEP_ERR_INVALID_ARG;
  const int d = mlp->d, t = mlp->t;
  if (d % 4 != 0 || reinterpret_cast<uintptr_t>(pe) % 16 != 0) return LSTEP_ERR_UNSUPPORTED;
  if (pe_rows > 0x7fffffffLL || (int64_t)n_ids * K > 0x7fffffffLL) return LSTEP_ERR_ID_RANGE;
  const int dvec = d / 4;
  const int threads = (int)align_up(align_up((size_t)t, 32) + dvec, 32);
  if (threads > 512 || dvec > 8 * 32 || t > 8 * 32) return LSTEP_ERR_UNSUPPORTED;
  const size_t need = carve(nullptr, n_ids, n_edges, K, d, t, pe_rows).bytes;
  if (!workspace || workspace_bytes < need) return LSTEP_ERR_WORKSPACE;
  return LSTEP_OK;
}

// phase A: aggregate over the batch edges for the rows `ids`, MLP with self term, in place. Also resets
// the phase-B counters.
static int phase_a(float* pe, const UpdateWs& w, const int64_t* ids, int64_t n_ids, const int64_t* src, const int64_t* dst,
                   const double* times, int64_t n_edges, float tc, const lstep_pe_mlp* mlp, cudaStream_t st,
                   bool edges_done = false) {
  const int d = mlp->d, t = mlp->t;
  const int dvec = d / 4;
  const int t_pad = (int)align_up((size_t)t, 32);
  const int threads = (int)align_up((size_t)t_pad + dvec, 32);
  const size_t smem = (size_t)threads * kSegPerThread * 8 + 32 * 4;
  const int64_t grid = n_ids < (int64_t)num_sms() * 16 ? n_ids : (int64_t)num_sms() * 16;
  if (!edges_done) {  // (the streaming step forms the aggregate rows in its fused gather launch, csrc/step.cu)
    launch_k(edge_aggregate_kernel, dim3((unsigned)grid), dim3(threads), smem, st, pe, ids, n_ids, src, dst, times, n_edges, tc, mlp->tw, d,
             t, t_pad, w.A, w.lda, w.counters);
    const int rc = check_launch("edge_aggregate");
    if (rc != LSTEP_OK) return rc;
  }
  // late trigger: the kernel behind this one (phase B's push) may run its pre-wait part next to it, not earlier
  return launch_pe_mlp(w.A, w.lda, pe, single_ids(ids), n_ids, n_ids, nullptr, mlp, nullptr, 0, pe, st, true);
}

}  // namespace lstep
namespace lstep {
// phase A's aggregate rows of `ids` into the update workspace (resets the phase-B counters), then its MLP into the
// workspace's new_rows buffer (row i = ids[i]) instead of the table: the stand-alone form of what the streaming step does
// inside its fused gather / paired MLP launches. n_ids == 0 only resets the counters.
int launch_phase_a_to_new_rows(const float* pe, void* workspace, int64_t ws_ids, int64_t ws_edges, int K, int64_t pe_rows, const int64_t* ids,
                               int64_t n_ids, const int64_t* src, const int64_t* dst, const double* times, int64_t n_edges, float tc,
                               const lstep_pe_mlp* mlp, bool aggregate_done, cudaStream_t st) {
  const int d = mlp->d, t = mlp->t;
  UpdateWs w = carve(workspace, ws_ids, ws_edges, K, d, t, pe_rows);
  if (n_ids == 0) {
    cudaError_t e = cudaMemsetAsync(w.counters, 0, sizeof(int32_t) * 8, st);
    if (e != cudaSuccess) {
      set_cuda_error(e, "phase_a counters");
      return LSTEP_ERR_CUDA;
    }
    return LSTEP_OK;
  }
  if (!aggregate_done) {
    const int dvec = d / 4;
    const int t_pad = (int)align_up((size_t)t, 32);
    const int threads = (int)align_up((size_t)t_pad + dvec, 32);
    const size_t smem = (size_t)threads * kSegPerThread * 8 + 32 * 4;
    const int64_t grid = n_ids < (int64_t)num_sms() * 16 ? n_ids : (int64_t)num_sms() * 16;
    launch_k(edge_aggregate_kernel, dim3((unsigned)grid), dim3(threads), smem, st, pe, ids, n_ids, src, dst, times, n_edges, tc, mlp->tw, d, t,
             t_pad, w.A, w.lda, w.counters);
    const int rc = check_launch("edge_aggregate");
    if (rc != LSTEP_OK) return rc;
  }
  return launch_pe_mlp(w.A, w.lda, pe, single_ids(ids), n_ids, n_ids, nullptr, mlp, w.new_rows, d, nullptr, st, true);
}
}  // namespace lstep
namespace lstep {

// phase B, aggregation half: lookup of (csr_ids[i], q_times[i]) for i < n_valid, inverse index, per
// destination reduction of [pe[row_ids[i]] || tf]. Leaves U (distinct destinations, + 0 when any slot
// was padding), the aggregate rows A and the device counters in the workspace.
static int phase_b_partial(float* pe, int64_t pe_rows, const UpdateWs& w, const lstep_csr* csr, const int64_t* csr_ids,
                           const int64_t* row_ids, int64_t n_ids, const double* q_times, int64_t n_valid, float tc, int K,
                           const lstep_pe_mlp* mlp, uint32_t* err_flag, void* stream) {
  const int d = mlp->d, t = mlp->t;
  const int dvec = d / 4;
  cudaStream_t st = as_stream(stream);
  const int64_t total = n_ids * (int64_t)K;
  int rc;
  {
    PhaseBHook hook{w.cnt_of, w.rank, w.U, w.counters, pe, d};
    rc = launch_sample_count(csr, csr_ids, q_times, n_ids, n_valid, K, w.nbrB, w.ntB, err_flag, hook, stream);
    if (rc != LSTEP_OK) return rc;
  }
  {
    const int fill_here = total <= 16384 ? 1 : 0;
    launch_k(phaseB_scan_kernel, dim3(1 + kRow0Parts), dim3(1024), 0, st, w.cnt_of, w.slot_of, w.U, w.off, w.hubs, w.hub_remaining, w.task_hub,
                                                        w.task_chunk, w.hub_acc, d + t, w.counters, w.nbrB, total, K,
                                                        w.rank, w.list, fill_here, pe, row_ids, n_ids, d, w.row0_part);
    if ((rc = check_launch("phaseB_scan")) != LSTEP_OK) return rc;
    if (!fill_here) {
      launch_k(phaseB_fill_kernel, dim3((unsigned)ceil_div(total, 256)), dim3(256), 0, st, w.nbrB, total, w.slot_of, w.off, w.rank, w.list);
      if ((rc = check_launch("phaseB_fill")) != LSTEP_OK) return rc;
    }
  }
  const int64_t max_dest = total < pe_rows - 1 ? total : pe_rows - 1;  // distinct non-zero destinations
  const int warp_blocks = (int)ceil_div(max_dest > 0 ? max_dest : 1, 8);
  int hub_blocks = (int)(((total >> kChunkLog2) + total / (kHubLen + 1)) / 8) + 1;  // enough warps for every possible chunk task
  if (hub_blocks > 4 * num_sms()) hub_blocks = 4 * num_sms();
  const unsigned blocks = (unsigned)(warp_blocks + hub_blocks + 1);
  const float bound = fixed_point_bound(n_ids, K);
  if (dvec <= 64 && t <= 128)
    launch_k(phaseB_gather_kernel<2, 4>, dim3(blocks), dim3(256), 0, st, pe, row_ids, K, w.ntB, w.off, w.list, w.hubs, w.hub_remaining, w.task_hub,
                                                       w.task_chunk, w.hub_acc, w.counters, tc, mlp->tw, d, t, w.row0_part, w.A, w.lda,
                                                       warp_blocks, hub_blocks, bound, err_flag);
  else
    launch_k(phaseB_gather_kernel<8, 8>, dim3(blocks), dim3(256), 0, st, pe, row_ids, K, w.ntB, w.off, w.list, w.hubs, w.hub_remaining, w.task_hub,
                                                       w.task_chunk, w.hub_acc, w.counters, tc, mlp->tw, d, t, w.row0_part, w.A, w.lda,
                                                       warp_blocks, hub_blocks, bound, err_flag);
  return check_launch("phaseB_gather");
}

// phase B, write-back half: pe[U] += tanh(mlp(A)), no self term (Q3)
static int phase_b_apply(float* pe, int64_t pe_rows, const UpdateWs& w, int64_t n_ids, int K, const lstep_pe_mlp* mlp,
                         cudaStream_t st) {
  const int64_t total = n_ids * (int64_t)K;
  const int64_t max_dest = total < pe_rows - 1 ? total : pe_rows - 1;
  lstep_pe_mlp noself = *mlp;
  noself.ws = nullptr;  // the self term is computed and discarded by the reference (LSTEP.py:334-335, Q3)
  noself.bs = nullptr;
  noself.ws_tc = nullptr;
  return launch_pe_mlp(w.A, w.lda, pe, single_ids(w.U), max_dest + 1, n_ids * 6, w.counters + 2, &noself, nullptr, 0, pe, st);
}

}  // namespace lstep

namespace lstep {
// where phase A's aggregate rows and the phase-B counters live inside an update workspace
void update_ws_phase_a(void* workspace, int64_t n_ids, int64_t n_edges, int K, int d, int t, int64_t pe_rows, float** A, int64_t* lda,
                       int32_t** counters, float** new_rows) {
  UpdateWs w = carve(workspace, n_ids, n_edges, K, d, t, pe_rows);
  *A = w.A;
  *lda = w.lda;
  *counters = w.counters;
  *new_rows = w.new_rows;
}

void update_ws_phase_b_lists(void* workspace, int64_t n_ids, int64_t n_edges, int K, int d, int t, int64_t pe_rows, const int64_t** U,
                             const int32_t** n_dest_dev, const int32_t** stamp_map) {
  UpdateWs w = carve(workspace, n_ids, n_edges, K, d, t, pe_rows);
  *U = w.U;
  *n_dest_dev = w.counters + 2;
  *stamp_map = w.slot_of;
}

// the push form of phase B (and with it the side-buffer form of phase A) is available for this shape
bool update_push_available(const lstep_pe_mlp* mlp) {
  const bool pull = tuning().phaseb_push == 0;
  return !pull && mlp && (mlp->d + mlp->t) % 2 == 0 && mlp->d <= 256 && mlp->t <= 256 && pe_mlp_cluster_supports(mlp);
}

int update_pe_impl(float* pe, int64_t pe_rows, const lstep_csr* csr, const int64_t* ids, int64_t n_ids, const int64_t* src,
                   const int64_t* dst, const double* times, int64_t n_edges, double current_time, int K, const lstep_pe_mlp* mlp,
                   void* workspace, size_t workspace_bytes, uint32_t* err_flag, void* stream, bool edges_done, int32_t** dirty_out, int stamp, bool phase_a_in_new_rows,
                   float* ring_slot, int64_t ring_stride, const PushOwner* owner = nullptr);
}  // namespace lstep

extern "C" int lstep_update_pe(float* pe, int64_t pe_rows, const lstep_csr* csr, const int64_t* ids, int64_t n_ids,
                               const int64_t* src, const int64_t* dst, const double* times, int64_t n_edges,
                               double current_time, int K, const lstep_pe_mlp* mlp, void* workspace,
                               size_t workspace_bytes, uint32_t* err_flag, void* stream) {
  return update_pe_impl(pe, pe_rows, csr, ids, n_ids, src, dst, times, n_edges, current_time, K, mlp, workspace, workspace_bytes,
                        err_flag, stream, false, nullptr, 0, false, nullptr, 0);
}

// edges_done: phase A's aggregate rows (and the zeroed counters) are already in the workspace
int lstep::update_pe_impl(float* pe, int64_t pe_rows, const lstep_csr* csr, const int64_t* ids, int64_t n_ids, const int64_t* src,
                          const int64_t* dst, const double* times, int64_t n_edges, double current_time, int K,
                          const lstep_pe_mlp* mlp, void* workspace, size_t workspace_bytes, uint32_t* err_flag, void* stream,
                          bool edges_done, int32_t** dirty_out, int stamp, bool phase_a_in_new_rows, float* ring_slot,
                          int64_t ring_stride, const PushOwner* owner) {
  // owner (peer group, csrc/peer.cu): phase B of the destinations this rank owns only; phase A's rows of ALL batch nodes
  // are read from owner->new_rows (row i = ids[i], gathered from the owners), the owned ones are applied to `pe`.
  // ring_slot / ring_stride (streaming step, with dirty_out): the phase-B MLP also writes its rows into the history
  // ring's new slot, so the caller's ring append only has to copy the rows NOT carrying `stamp`.
  // phase_a_in_new_rows (streaming step): phase A's MLP has already run (in the caller's paired launch) and left its
  // rows in the workspace's new_rows buffer; the push kernel applies them. Requires update_push_available().
  // dirty_out (streaming step): when the push form runs, *dirty_out = per-node map in which the rows phase B changes
  // carry `stamp` (unique per step; no clearing, stale values never match), which the caller's ring append reads;
  // the phase-B MLP is then launched with a late trigger so that the append may copy the unchanged rows next to it.
  if (dirty_out) *dirty_out = nullptr;
  int rc = check_update_args(pe, pe_rows, mlp, n_ids, n_edges, K, workspace, workspace_bytes);
  if (rc != LSTEP_OK) return rc;
  if (!csr || (n_ids > 0 && !ids) || (n_edges > 0 && (!src || !dst || !times))) return LSTEP_ERR_INVALID_ARG;
  if (csr->num_rows > pe_rows) return LSTEP_ERR_INVALID_ARG;
  const int d = mlp->d, t = mlp->t;
  UpdateWs w = carve(workspace, n_ids, n_edges, K, d, t, pe_rows);
  cudaStream_t st = as_stream(stream);
  const float tc = (float)current_time;
  if (n_ids == 0) {  // nothing to update; the reference still zeroes the padding row (LSTEP.py:317)
    cudaError_t e = cudaMemsetAsync(pe, 0, sizeof(float) * d, st);
    if (e != cudaSuccess) {
      set_cuda_error(e, "update_pe memset");
      return LSTEP_ERR_CUDA;
    }
    return LSTEP_OK;
  }
  if (phase_a_in_new_rows && !update_push_available(mlp)) return LSTEP_ERR_INVALID_ARG;
  if (owner && (!phase_a_in_new_rows || !owner->new_rows || owner->mul < 1 || owner->add < 0 || owner->add >= owner->mul)) return LSTEP_ERR_INVALID_ARG;
  if (!phase_a_in_new_rows && (rc = phase_a(pe, w, ids, n_ids, src, dst, times, n_edges, tc, mlp, st, edges_done)) != LSTEP_OK) return rc;
  const int64_t n_valid = n_ids < n_edges ? n_ids : n_edges;  // zip(node_ids, times) truncation (Q1)
  {
    // phase B, push form (csrc/update_push.cu): lookup + exact fixed-point accumulation where the contribution
    // lands, then the MLP straight off the accumulator rows. LSTEP_PHASEB_PULL=1 selects the pull form below.
    if (update_push_available(mlp)) {
      rc = launch_phaseB_push(csr, ids, times, n_ids, n_valid, K, pe, d, t, mlp->tw, tc, w.claim_of, w.U, w.counters, w.push_acc,
                              w.slot_of, stamp, owner ? owner->new_rows : (phase_a_in_new_rows ? w.new_rows : nullptr), err_flag, st,
                              w.push_row0, owner ? owner->mul : 1, owner ? owner->add : 0);
      if (rc != LSTEP_OK) return rc;
      prof_mark(st, kProfPush);
      const int64_t total = n_ids * (int64_t)K;
      const int64_t max_dest = total < pe_rows - 1 ? total : pe_rows - 1;
      lstep_pe_mlp noself = *mlp;
      noself.ws = nullptr;  // the self term is computed and discarded by the reference (LSTEP.py:334-335, Q3)
      noself.bs = nullptr;
      noself.ws_tc = nullptr;
      if (dirty_out) *dirty_out = w.slot_of;
      // expected rows: ~4 distinct sampled neighbours per batch node on the benchmark graphs (measured 3.9); a launch
      // with more rows than the chosen tile covers in one round of clusters just walks a second round
      rc = launch_pe_mlp_cluster(nullptr, 0, pe, single_ids(w.U), max_dest + 1, n_ids * 4 / (owner ? owner->mul : 1) + 1, w.counters + 2, &noself, nullptr, 0, pe,
                                 w.push_acc, w.claim_of, st, dirty_out != nullptr, dirty_out ? ring_slot : nullptr, ring_stride);
      prof_mark(st, kProfMlpB);
      return rc;
    }
  }
  if ((rc = phase_b_partial(pe, pe_rows, w, csr, ids, ids, n_ids, times, n_valid, tc, K, mlp, err_flag, stream)) != LSTEP_OK) return rc;
  return phase_b_apply(pe, pe_rows, w, n_ids, K, mlp, st);
}

// ---- the same phases as separate entry points (node-id sharded tables: the phases are separated by
// ---- row exchanges between ranks, see l-step_b200/shard.py)
extern "C" int lstep_update_pe_phase_a(float* pe, int64_t pe_rows, const int64_t* ids, int64_t n_ids, const int64_t* src,
                                       const int64_t* dst, const double* times, int64_t n_edges, double current_time, int K,
                                       const lstep_pe_mlp* mlp, void* workspace, size_t workspace_bytes, void* stream) {
  int rc = check_update_args(pe, pe_rows, mlp, n_ids, n_edges, K, workspace, workspace_bytes);
  if (rc != LSTEP_OK) return rc;
  if (n_ids == 0) return LSTEP_OK;
  if (!ids || (n_edges > 0 && (!src || !dst || !times))) return LSTEP_ERR_INVALID_ARG;
  UpdateWs w = carve(workspace, n_ids, n_edges, K, mlp->d, mlp->t, pe_rows);
  return phase_a(pe, w, ids, n_ids, src, dst, times, n_edges, (float)current_time, mlp, as_stream(stream));
}

extern "C" int lstep_update_pe_phase_b_partial(float* pe, int64_t pe_rows, const lstep_csr* csr, const int64_t* csr_ids,
                                               const int64_t* row_ids, int64_t n_ids, const double* q_times, int64_t n_valid,
                                               int64_t n_edges_layout, double current_time, int K, const lstep_pe_mlp* mlp,
                                               void* workspace, size_t workspace_bytes, uint32_t* err_flag, void* stream) {
  int rc = check_update_args(pe, pe_rows, mlp, n_ids, n_edges_layout, K, workspace, workspace_bytes);
  if (rc != LSTEP_OK) return rc;
  if (!csr || n_ids <= 0 || !csr_ids || !row_ids || !q_times || n_valid < 0) return LSTEP_ERR_INVALID_ARG;
  UpdateWs w = carve(workspace, n_ids, n_edges_layout, K, mlp->d, mlp->t, pe_rows);
  cudaError_t e = cudaMemsetAsync(w.counters, 0, sizeof(int32_t) * 8, as_stream(stream));
  if (e != cudaSuccess) {
    set_cuda_error(e, "phase_b counters");
    return LSTEP_ERR_CUDA;
  }
  return phase_b_partial(pe, pe_rows, w, csr, csr_ids, row_ids, n_ids, q_times, n_valid, (float)current_time, K, mlp, err_flag,
                         stream);
}

extern "C" int lstep_update_pe_workspace_layout(int64_t n_ids, int64_t n_edges, int K, int d, int t, int64_t pe_rows,
                                                int64_t* offsets /* [4]: counters, U, A (bytes), lda (floats) */) {
  if (!offsets || n_ids < 0 || n_edges < 0 || K <= 0 || d <= 0 || t < 0 || pe_rows <= 0) return LSTEP_ERR_INVALID_ARG;
  char base[1];
  UpdateWs w = carve(base, n_ids, n_edges, K, d, t, pe_rows);
  offsets[0] = reinterpret_cast<char*>(w.counters) - base;
  offsets[1] = reinterpret_cast<char*>(w.U) - base;
  offsets[2] = reinterpret_cast<char*>(w.A) - base;
  offsets[3] = w.lda;
  return LSTEP_OK;
}

// out[s][:] = sum of rows[seg_off[s] .. seg_off[s+1]) in order (fixed order => reproducible): combines
// the per-rank partial aggregates of a destination.
namespace lstep {
__global__ void __launch_bounds__(256) segment_sum_rows_kernel(const float* __restrict__ rows, int64_t ld,
                                                               const int64_t* __restrict__ seg_off, int64_t n_seg, int width,
                                                               float* __restrict__ out, int64_t ldo) {
  for (int64_t s = blockIdx.x; s < n_seg; s += gridDim.x) {
    const int64_t lo = seg_off[s], hi = seg_off[s + 1];
    for (int c = threadIdx.x; c < width; c += blockDim.x) {
      float acc = 0.f;
      for (int64_t r = lo; r < hi; ++r) acc += rows[r * ld + c];
      out[s * ldo + c] = acc;
    }
  }
}
}  // namespace lstep

extern "C" int lstep_segment_sum_rows(const float* rows, int64_t ld, const int64_t* seg_off, int64_t n_seg, int width,
                                      float* out, int64_t ldo, void* stream) {
  if (n_seg < 0 || width <= 0) return LSTEP_ERR_INVALID_ARG;
  if (n_seg == 0) return LSTEP_OK;
  if (!rows || !seg_off || !out) return LSTEP_ERR_INVALID_ARG;
  const int64_t grid = n_seg < (int64_t)num_sms() * 8 ? n_seg : (int64_t)num_sms() * 8;
  segment_sum_rows_kernel<<<(unsigned)grid, 256, 0, as_stream(stream)>>>(rows, ld, seg_off, n_seg, width, out, ldo);
  return check_launch("segment_sum_rows");
}
