// Peer group: the scale-out PE step over NVLink peer memory (BASELINE config 5: 10 M nodes, 8 x B200; SURVEY §8(e)).
//
// Layout. Every rank holds a REPLICA of the current PE table [V1, d] (6.9 GB at 10 M nodes) and of the temporal CSR, and
// OWNS the nodes v with v % world == rank: their PE history (change log, csrc/changelog.cu) and every piece of work whose
// result is a row of an owned node. Replicas are kept equal through PEER MEMORY (CUDA IPC mappings over NVLink / NVSwitch):
// an owner copies the rows it changes, as contiguous blocks, into small fixed regions of every other rank (inbox, filt and
// new_rows buffers), each rank scatters what it received into its own replica, and two flag barriers per step, also in
// peer memory, order everything. No NCCL call, no host involvement, no data-dependent message size:
//
//     filter     owned batch nodes: history -> filtered row -> local table AND every other rank's filt buffer (at the
//                node's position in the batch's id list)                                           (1/world of the rows)
//     ---------- barrier 1 + refresh (one launch): scatter into the local replica (a) the rows the previous step changed on
//                the other ranks (this rank's inbox blocks), (b) the other owners' filtered rows of this step (filt buffer)
//     gather     a6 lookup + aggregate of this rank's 1/world share of the query rows  ||  a7 edge aggregate of the owned
//                batch nodes                                                                     (reads the local replica)
//     MLP pair   neighbourhood MLP of the share -> outputs  ||  phase-A MLP of the owned batch nodes -> local new_rows
//     bcast      new_rows[i] -> every rank's new_rows buffer at row pos_mine[i] (2.7 MB per step in total)
//     ---------- barrier 2: phase A's rows of ALL batch nodes are in every rank's new_rows buffer --------------------------
//     push       lookup of ALL batch nodes (replicated: 4 k warp searches), accumulation for the OWNED destinations only
//                (exact fixed point, csrc/update_push.cu); the owned batch nodes' phase-A rows go into the local table
//     MLP (B)    owned destinations: table row <- row + tanh(mlp(aggregate))                      (local table)
//     append     owned changed rows (owned batch nodes, owned destinations, row 0 on rank 0) become events of the change log
//     publish    the slot's events (count, node ids, rows) -> this rank's block in every other rank's inbox; in the native
//                multi-step call on a side stream, next to the next step's filter
//
// Why two barriers are enough:
//   * what a rank writes into another rank, and when it is read: its inbox block (written by publish(s), complete before this
//     rank announces barrier 1 of s+1, read by the receiver's refresh of s+1, rewritten by publish(s+1), which follows barrier
//     2 of s+1 — announced by every rank only after its refresh of s+1); the filt buffer (written by filter(s+1) before barrier
//     1 of s+1, read by the refresh of s+1, rewritten by filter(s+2), which follows barrier 2 of s+1 likewise); the new_rows
//     buffer (written by bcast(s) before barrier 2 of s, read by push(s), rewritten by bcast(s+1), which follows barrier 1 of
//     s+1 — announced by every rank only after its push(s)).
//   * between barrier 2 of a step and the next barrier 1 a rank touches only rows it owns (push applies owned phase-A rows,
//     the phase-B MLP reads and writes owned destinations, the append reads owned rows); its replica is stale for the rows
//     OTHER owners change in that interval, which it does not read before the next refresh.
//   * the refresh writes disjoint rows in its two passes: rows changed by the previous step are skipped when they belong to
//     the current batch (sorted id list, warp search) — their filtered row is newer.
// Everything that crosses NVLink is a contiguous store into a small fixed region. Measured and dropped (profiles/
// r02_peer_bw.txt, r02_scaleout_history.md): owners storing changed rows straight into the other 6.9 GB replicas (scattered
// peer stores thrash the peer TLB: 43 GB/s against 500 GB/s contiguous; 200 us per step), and ranks PULLING the events out of
// the owners' change logs instead of a publication (peer reads of a different, TLB-cold slot every step: 126 GB/s at 8 ranks).
//
// Results equal the single-GPU step's bit for bit: every row is computed by one rank from the same inputs with the same
// kernels, and phase B's sums are exact 32.32 fixed point (independent of who adds what in which order).
//
// Barrier = flag exchange in peer memory: rank r announces epoch e by storing e into flags[g][r] of every rank g
// (st.release.sys after a system-scope fence; the kernels that store into peers fence their own stores too); a rank waits
// by polling its OWN flag block (ld.acquire.sys) until all `world` entries are >= e. The wait is bounded (timeout_ms on the
// global timer): a missing peer raises LSTEP_FLAG_PEER_TIMEOUT instead of hanging the device. The inserted kernels are
// programmatic dependent launches that wait first and trigger second, so the successor's pre-wait work (the gather's
// lookups and cosines, the push kernel's lookups and claims) runs while this rank waits for the others.
#include <algorithm>
#include <cstring>

#include "common.cuh"
#include "step_core.cuh"

namespace lstep {

int changelog_filter_peer(const lstep_changelog* cl, int head, int len, const int64_t* ids, int64_t n_ids, const float* G, float* out,
                          int64_t out_stride, const int64_t* out_ids, float* const* out2, int n_out2, const int64_t* out2_ids, void* stream);

namespace {

struct PeerPtrs {
  float* p[LSTEP_MAX_PEERS];
  int n;
};
struct FlagPtrs {
  uint32_t* p[LSTEP_MAX_PEERS];
  int n, rank;
};

bool valid_group(const lstep_peer_group* g) {
  if (!g || g->world < 1 || g->world > LSTEP_MAX_PEERS || g->rank < 0 || g->rank >= g->world) return false;
  for (int i = 0; i < g->world; ++i)
    if (!g->new_rows[i] || !g->flags[i]) return false;
  return g->table[g->rank] != nullptr;
}

// dst[g][dst_rows[i]][:] = src[i][:] for every rank g (the local one included): one warp per row
__global__ void __launch_bounds__(256) peer_rows_bcast_kernel(const float* __restrict__ src, int64_t n_rows, int d,
                                                              const int64_t* __restrict__ dst_rows, PeerPtrs dst) {
  pdl_wait();  // every inserted kernel of the peer step: wait first, then let the successor become resident (late trigger)
  pdl_launch_dependents();
  const int lane = threadIdx.x & 31;
  const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5, n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  const int dvec = d >> 2;
  for (int64_t i = warp; i < n_rows; i += n_warps) {
    const int64_t r = dst_rows ? dst_rows[i] : i;
    const float4* s = reinterpret_cast<const float4*>(src + i * (int64_t)d);
    for (int c = lane; c < dvec; c += 32) {
      const float4 x = __ldcg(s + c);
      for (int g = 0; g < dst.n; ++g) reinterpret_cast<float4*>(dst.p[g] + r * (int64_t)d)[c] = x;
    }
  }
  __threadfence_system();
}

// ---- inbox: what the other ranks WRITE into this rank between two barriers 1, as contiguous blocks in a small, fixed region
// (scattered accesses to a multi-GB peer mapping, and reads of peer memory in general, are slow: 43 GB/s scattered against
// 500 GB/s contiguous stores, and 126 GB/s for contiguous READS of the owners' change logs at 8 ranks, profiles/r02_peer_bw.txt
// and r02_scaleout_history.md). One block per source rank: { int32 count, pad[3]; int32 node[cap]; float row[cap][d] } = the rows
// the source changed in the previous step.
__host__ __device__ inline size_t inbox_rows_off(int64_t cap) { return align_up(16 + 4 * (size_t)cap, 256); }
__host__ __device__ inline size_t inbox_stride(int64_t cap, int d) { return align_up(inbox_rows_off(cap) + (size_t)cap * d * 4, 256); }

struct InboxPtrs {
  unsigned char* p[LSTEP_MAX_PEERS];  // the OTHER ranks' blocks for this source (publish) / this rank's blocks of the other sources (refresh)
  int n;
};

// events [0, cnt) of the change log's slot -> every other rank's inbox block for this rank: count, node ids, rows
__global__ void __launch_bounds__(256) peer_publish_kernel(lstep_changelog cl, int slot, InboxPtrs dst, int64_t cap) {
  pdl_wait();
  pdl_launch_dependents();
  const int cnt = min(min((int)((unsigned)__ldcg(cl.ev_cnt + slot) & ((1u << 20) - 1)), cl.cap), (int)cap);
  const int dvec = cl.d >> 2;
  const int64_t gtid = blockIdx.x * (int64_t)blockDim.x + threadIdx.x, nthr = (int64_t)gridDim.x * blockDim.x;
  const int32_t* node = cl.ev_node + (size_t)slot * cl.cap;
  const float4* rows = reinterpret_cast<const float4*>(cl.ev_row + (size_t)slot * cl.cap * cl.d);
  const size_t roff = inbox_rows_off(cap);
  if (gtid == 0)
    for (int g = 0; g < dst.n; ++g) *reinterpret_cast<int32_t*>(dst.p[g]) = cnt;
  for (int64_t i = gtid; i < cnt; i += nthr) {
    const int32_t v = __ldcg(node + i);
    for (int g = 0; g < dst.n; ++g) reinterpret_cast<int32_t*>(dst.p[g] + 16)[i] = v;
  }
  const int64_t total = (int64_t)cnt * dvec;
  constexpr int kPer = 4;
  for (int64_t base = 0; base < total; base += nthr * kPer) {
    float4 x[kPer];
#pragma unroll
    for (int e = 0; e < kPer; ++e) {
      const int64_t i = base + gtid + e * nthr;
      if (i < total) x[e] = __ldcg(rows + i);
    }
#pragma unroll
    for (int e = 0; e < kPer; ++e) {
      const int64_t i = base + gtid + e * nthr;
      if (i < total)
        for (int g = 0; g < dst.n; ++g) reinterpret_cast<float4*>(dst.p[g] + roff)[i] = x[e];
    }
  }
  __threadfence_system();
}

// is v in the ascending list a[0 .. n)? 32-ary search by a full warp (all lanes pass the same arguments)
__device__ __forceinline__ bool warp_contains_sorted(const int64_t* __restrict__ a, int64_t n, int64_t v, int lane) {
  int64_t lo = 0, hi = n;
  while (hi - lo > 32) {
    const int64_t len = hi - lo;
    const int64_t p = lo + (len * (lane + 1)) / 33;
    const int j = __popc(__ballot_sync(kFull, a[p] < v));  // pivots 0 .. j-1 are < v, pivot j (if any) is >= v
    const int64_t pa = lo + (len * j) / 33, pb = lo + (len * (j + 1)) / 33;
    if (j < 32) hi = pb + 1;
    if (j > 0) lo = pa + 1;
  }
  const bool hit = lo + lane < hi && a[lo + lane] == v;
  return __any_sync(kFull, hit);
}

// Barrier wait + refresh of this rank's replica (one launch): every CTA waits (thread 0 polls this rank's own flag block), then
//   pass 1  the rows the PREVIOUS step changed on the other ranks, from this rank's inbox blocks — except the nodes of the
//           current batch (ids, ascending), whose owners' filtered row of THIS step is newer;
//   pass 2  the filtered rows of the current batch nodes this rank does not own, from this rank's filt buffer (row p = the node
//           at position p of the batch's id list, stored there by its owner's filter kernel).
// The two passes write disjoint rows; everything is read from LOCAL memory.
__global__ void __launch_bounds__(256) peer_wait_apply_kernel(const uint32_t* flags, uint32_t epoch, unsigned long long timeout_ns,
                                                              uint32_t* err_flag, InboxPtrs src, const float* __restrict__ filt, int world,
                                                              int rank, int64_t cap, float* table, int d, int64_t V1,
                                                              const int64_t* __restrict__ ids, int64_t n_ids, FlagPtrs announce) {
  __shared__ int s_ok;
  pdl_wait();
  pdl_launch_dependents();
  // announce.n > 0: this launch also ANNOUNCES the epoch (block 0; every earlier kernel of the stream has completed) — the
  // barrier is then one launch instead of two
  if (blockIdx.x == 0 && announce.n > 0) {
    __threadfence_system();
    if ((int)threadIdx.x < announce.n)
      asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(announce.p[threadIdx.x] + announce.rank), "r"(epoch) : "memory");
  }
  if (threadIdx.x == 0) {
    bool ok = true;
    unsigned long long t0;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
    for (int g = 0; g < world && ok; ++g) {
      for (;;) {
        uint32_t v;
        asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(flags + g) : "memory");
        if ((int32_t)(v - epoch) >= 0) break;
        unsigned long long t1;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
        if (t1 - t0 > timeout_ns) {
          ok = false;
          break;
        }
        __nanosleep(100);
      }
    }
    if (!ok && err_flag && blockIdx.x == 0) atomicOr(err_flag, LSTEP_FLAG_PEER_TIMEOUT);
    s_ok = ok;
    __threadfence_system();
  }
  __syncthreads();
  if (!s_ok) return;
  const int dvec = d >> 2;
  const int lane = threadIdx.x & 31;
  const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5, n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  const size_t roff = inbox_rows_off(cap);
  for (int g = 0; g < src.n; ++g) {
    const unsigned char* blk = src.p[g];
    const int cnt = min(__ldcg(reinterpret_cast<const int32_t*>(blk)), (int)cap);
    const int32_t* node = reinterpret_cast<const int32_t*>(blk + 16);
    const float4* rows = reinterpret_cast<const float4*>(blk + roff);
    for (int64_t i0 = warp * 2; i0 < cnt; i0 += n_warps * 2) {  // two rows per warp and round: more loads in flight
      int64_t v[2];
      float4 x[2][2];
      bool take[2];
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const int64_t i = i0 + u;
        take[u] = i < cnt;
        v[u] = take[u] ? (int64_t)__ldcg(node + i) : -1;
        take[u] = take[u] && v[u] >= 0 && v[u] < V1;
        if (take[u]) {
          x[u][0] = __ldcg(rows + i * dvec + lane);
          if (lane + 32 < dvec) x[u][1] = __ldcg(rows + i * dvec + lane + 32);
        }
      }
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        if (!take[u]) continue;
        if (n_ids > 0 && warp_contains_sorted(ids, n_ids, v[u], lane)) continue;
        float4* dst = reinterpret_cast<float4*>(table + v[u] * (int64_t)d);
        dst[lane] = x[u][0];
        if (lane + 32 < dvec) dst[lane + 32] = x[u][1];
      }
    }
  }
  for (int64_t p = warp; p < n_ids; p += n_warps) {
    const int64_t v = ids[p];
    if ((int)(v % world) == rank || v < 0 || v >= V1) continue;
    const float4* row = reinterpret_cast<const float4*>(filt + p * (int64_t)d);
    for (int c = lane; c < dvec; c += 32) reinterpret_cast<float4*>(table + v * (int64_t)d)[c] = __ldcg(row + c);
  }
}

__global__ void peer_signal_kernel(FlagPtrs f, uint32_t epoch) {
  pdl_wait();
  pdl_launch_dependents();
  // every earlier kernel of the stream has completed (plain launch) and fenced its peer stores; fence again, then announce
  __threadfence_system();
  const int g = threadIdx.x;
  if (g < f.n) asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(f.p[g] + f.rank), "r"(epoch) : "memory");
}

__global__ void peer_wait_kernel(const uint32_t* flags, int world, uint32_t epoch, unsigned long long timeout_ns, uint32_t* err_flag,
                                 FlagPtrs announce) {
  pdl_wait();
  pdl_launch_dependents();
  const int g = threadIdx.x;
  if (announce.n > 0) {  // (see peer_wait_apply_kernel)
    __threadfence_system();
    if (g < announce.n) asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(announce.p[g] + announce.rank), "r"(epoch) : "memory");
  }
  bool ok = true;
  if (g < world) {
    unsigned long long t0;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
    for (;;) {
      uint32_t v;
      asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(flags + g) : "memory");
      if ((int32_t)(v - epoch) >= 0) break;
      unsigned long long t1;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
      if (t1 - t0 > timeout_ns) {
        ok = false;
        break;
      }
      __nanosleep(100);
    }
  }
  if (!ok && err_flag) atomicOr(err_flag, LSTEP_FLAG_PEER_TIMEOUT);
  __threadfence_system();
}

}  // namespace

int peer_rows_bcast(const float* src, int64_t n_rows, int d, const int64_t* dst_rows, const lstep_peer_group* grp, int which, cudaStream_t st) {
  if (!valid_group(grp) || !src || n_rows < 0 || d <= 0 || d % 4 != 0) return LSTEP_ERR_INVALID_ARG;
  if (n_rows == 0) return LSTEP_OK;
  PeerPtrs dst{};
  for (int g = 0; g < grp->world; ++g) {
    float* p = which == 0 ? grp->table[g] : grp->new_rows[g];
    if (!p) return LSTEP_ERR_INVALID_ARG;
    dst.p[dst.n++] = p;
  }
  const int64_t grid = std::min<int64_t>(ceil_div(n_rows * 32, 256), (int64_t)num_sms() * 8);
  launch_k(peer_rows_bcast_kernel, dim3((unsigned)grid), dim3(256), 0, st, src, n_rows, d, dst_rows, dst);
  return check_launch("peer_rows_bcast");
}

int peer_signal(const lstep_peer_group* g, uint32_t epoch, cudaStream_t st) {
  if (!valid_group(g)) return LSTEP_ERR_INVALID_ARG;
  FlagPtrs f{};
  for (int i = 0; i < g->world; ++i) f.p[i] = g->flags[i];
  f.n = g->world;
  f.rank = g->rank;
  launch_k(peer_signal_kernel, dim3(1), dim3(32), 0, st, f, epoch);
  return check_launch("peer_signal");
}

static FlagPtrs flag_ptrs(const lstep_peer_group* g, bool announce) {
  FlagPtrs f{};
  if (announce) {
    for (int i = 0; i < g->world; ++i) f.p[i] = g->flags[i];
    f.n = g->world;
    f.rank = g->rank;
  }
  return f;
}

int peer_wait(const lstep_peer_group* g, uint32_t epoch, int timeout_ms, uint32_t* err_flag, cudaStream_t st, bool announce) {
  if (!valid_group(g)) return LSTEP_ERR_INVALID_ARG;
  const unsigned long long ns = (unsigned long long)(timeout_ms > 0 ? timeout_ms : 2000) * 1000000ull;
  launch_k(peer_wait_kernel, dim3(1), dim3(32), 0, st, (const uint32_t*)g->flags[g->rank], g->world, epoch, ns, err_flag, flag_ptrs(g, announce));
  return check_launch("peer_wait");
}

static bool valid_inbox(const lstep_peer_group* g) {
  if (g->world == 1) return true;
  if (g->cap <= 0) return false;
  for (int i = 0; i < g->world; ++i)
    if (!g->inbox[i] || !g->filt[i]) return false;
  return true;
}

// the events of the change log's `slot` into every other rank's inbox
static int peer_publish(const lstep_changelog* cl, int slot, const lstep_peer_group* g, int64_t expect_rows, cudaStream_t st) {
  if (g->world == 1) return LSTEP_OK;
  if (!valid_inbox(g) || g->cap < cl->cap) return LSTEP_ERR_INVALID_ARG;
  InboxPtrs dst{};
  const size_t stride = inbox_stride(g->cap, cl->d);
  for (int i = 0; i < g->world; ++i)
    if (i != g->rank) dst.p[dst.n++] = static_cast<unsigned char*>(g->inbox[i]) + (size_t)g->rank * stride;
  const int64_t work = std::max<int64_t>(expect_rows, 1) * (cl->d / 4);
  const int64_t grid = std::max<int64_t>(1, std::min<int64_t>(ceil_div(work, 256 * 4), (int64_t)num_sms() * 4));
  launch_k(peer_publish_kernel, dim3((unsigned)grid), dim3(256), 0, st, *cl, slot, dst, g->cap);
  return check_launch("peer_publish");
}

// wait for barrier `epoch`, then refresh this rank's table replica from its inbox and filt buffer (see peer_wait_apply_kernel)
static int peer_wait_apply(const lstep_peer_group* g, uint32_t epoch, int timeout_ms, uint32_t* err_flag, int d, int64_t V1, int64_t expect_rows,
                           const int64_t* ids, int64_t n_ids, cudaStream_t st, bool announce) {
  if (g->world == 1) return peer_wait(g, epoch, timeout_ms, err_flag, st, announce);
  if (!valid_inbox(g) || d > 256) return LSTEP_ERR_INVALID_ARG;
  InboxPtrs src{};
  const size_t stride = inbox_stride(g->cap, d);
  for (int i = 0; i < g->world; ++i)
    if (i != g->rank) src.p[src.n++] = static_cast<unsigned char*>(g->inbox[g->rank]) + (size_t)i * stride;
  const unsigned long long ns = (unsigned long long)(timeout_ms > 0 ? timeout_ms : 2000) * 1000000ull;
  const int64_t grid = std::max<int64_t>(1, std::min<int64_t>(ceil_div(std::max<int64_t>(expect_rows, 1) * 16, 256), (int64_t)num_sms() * 4));
  launch_k(peer_wait_apply_kernel, dim3((unsigned)grid), dim3(256), 0, st, (const uint32_t*)g->flags[g->rank], epoch, ns, err_flag, src,
           (const float*)g->filt[g->rank], g->world, g->rank, g->cap, g->table[g->rank], d, V1, ids, n_ids, flag_ptrs(g, announce));
  return check_launch("peer_wait_apply");
}

}  // namespace lstep

using namespace lstep;

extern "C" size_t lstep_peer_inbox_bytes(int world, int64_t cap, int d) {
  if (world < 1 || world > LSTEP_MAX_PEERS || cap <= 0 || d <= 0 || d % 4 != 0) return 0;
  return (size_t)world * inbox_stride(cap, d);
}

extern "C" int lstep_ipc_alloc(size_t bytes, void** ptr) {
  if (!ptr || bytes == 0) return LSTEP_ERR_INVALID_ARG;
  cudaError_t e = cudaMalloc(ptr, bytes);
  if (e == cudaSuccess) e = cudaMemset(*ptr, 0, bytes);
  if (e != cudaSuccess) {
    set_cuda_error(e, "ipc_alloc");
    return LSTEP_ERR_CUDA;
  }
  return LSTEP_OK;
}
extern "C" int lstep_ipc_free(void* ptr) {
  if (!ptr) return LSTEP_OK;
  cudaError_t e = cudaFree(ptr);
  if (e != cudaSuccess) {
    set_cuda_error(e, "ipc_free");
    return LSTEP_ERR_CUDA;
  }
  return LSTEP_OK;
}
extern "C" int lstep_ipc_export(void* ptr, unsigned char handle_out[64]) {
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
  if (!ptr || !handle_out) return LSTEP_ERR_INVALID_ARG;
  cudaIpcMemHandle_t h;
  cudaError_t e = cudaIpcGetMemHandle(&h, ptr);
  if (e != cudaSuccess) {
    set_cuda_error(e, "ipc_export");
    return LSTEP_ERR_CUDA;
  }
  memcpy(handle_out, &h, 64);
  return LSTEP_OK;
}
extern "C" int lstep_ipc_open(const unsigned char handle[64], void** ptr) {
  if (!handle || !ptr) return LSTEP_ERR_INVALID_ARG;
  cudaIpcMemHandle_t h;
  memcpy(&h, handle, 64);
  cudaError_t e = cudaIpcOpenMemHandle(ptr, h, cudaIpcMemLazyEnablePeerAccess);
  if (e != cudaSuccess) {
    set_cuda_error(e, "ipc_open");
    return LSTEP_ERR_CUDA;
  }
  return LSTEP_OK;
}
extern "C" int lstep_ipc_close(void* ptr) {
  if (!ptr) return LSTEP_OK;
  cudaError_t e = cudaIpcCloseMemHandle(ptr);
  if (e != cudaSuccess) {
    set_cuda_error(e, "ipc_close");
    return LSTEP_ERR_CUDA;
  }
  return LSTEP_OK;
}

/* dst[g][dst_rows[i]] = src[i] for every rank g whose bit is set in rank_mask (which: 0 = table replicas, 1 = new_rows buffers) */
extern "C" int lstep_peer_rows_bcast(const float* src, int64_t n_rows, int d, const int64_t* dst_rows, const lstep_peer_group* grp, int which,
                                     uint32_t rank_mask, void* stream) {
  if (!grp) return LSTEP_ERR_INVALID_ARG;
  lstep_peer_group g2 = *grp;
  int n = 0;
  for (int g = 0; g < grp->world && g < LSTEP_MAX_PEERS; ++g)
    if (rank_mask & (1u << g)) {
      g2.table[n] = grp->table[g];
      g2.new_rows[n] = grp->new_rows[g];
      g2.flags[n] = grp->flags[g];
      ++n;
    }
  if (n == 0) return LSTEP_OK;
  g2.world = n;
  g2.rank = 0;
  return peer_rows_bcast(src, n_rows, d, dst_rows, &g2, which, as_stream(stream));
}

extern "C" int lstep_peer_signal(const lstep_peer_group* g, uint32_t epoch, void* stream) { return peer_signal(g, epoch, as_stream(stream)); }
/* announce `epoch`, wait for every rank, then apply the inbox (the rows the last step changed on the other ranks): afterwards, in
 * stream order, this rank's replica equals every other one */
extern "C" int lstep_peer_sync_tables(const lstep_peer_group* g, uint32_t epoch, int timeout_ms, uint32_t* err_flag, int d, int64_t V1,
                                      void* stream) {
  if (!valid_group(g) || d <= 0 || d % 4 != 0 || V1 <= 0) return LSTEP_ERR_INVALID_ARG;
  int rc = peer_signal(g, epoch, as_stream(stream));
  if (rc != LSTEP_OK) return rc;
  return peer_wait_apply(g, epoch, timeout_ms, err_flag, d, V1, 1 << 16, nullptr, 0, as_stream(stream), false);
}
extern "C" int lstep_peer_wait(const lstep_peer_group* g, uint32_t epoch, int timeout_ms, uint32_t* err_flag, void* stream) {
  return peer_wait(g, epoch, timeout_ms, err_flag, as_stream(stream), false);
}

int lstep::side_lane_open(SideLane* lane) {
  if (cudaStreamCreateWithFlags(&lane->stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreateWithFlags(&lane->appended, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&lane->published, cudaEventDisableTiming) != cudaSuccess) {
    set_cuda_error(cudaGetLastError(), "peer side lane");
    return LSTEP_ERR_CUDA;
  }
  return LSTEP_OK;
}

void lstep::side_lane_close(SideLane* lane, cudaStream_t st) {
  // the caller's stream order must cover the last publication; the lane's objects are released once it has run
  if (lane->pending) cudaStreamWaitEvent(st, lane->published, 0);
  cudaEventDestroy(lane->appended);
  cudaEventDestroy(lane->published);
  cudaStreamDestroy(lane->stream);  // (asynchronous: the stream is released when its work has completed)
}

namespace lstep {
namespace {
// ids_mine / pos_mine of one batch (see peer_plan_mine): blocks of blockDim ids in order; in each, a warp ballot ranks a thread's
// owned id within its warp and a scan of the warp counts ranks the warp within the block
__global__ void __launch_bounds__(1024) peer_plan_kernel(const int64_t* __restrict__ ids, int64_t n_ids, int world, int rank,
                                                         int64_t* __restrict__ ids_mine, int64_t* __restrict__ pos_mine) {
  __shared__ int s_off[32];
  __shared__ int s_total;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, n_warps = blockDim.x >> 5;
  int64_t base = 0;
  for (int64_t i0 = 0; i0 < n_ids; i0 += blockDim.x) {
    const int64_t i = i0 + threadIdx.x;
    const int64_t v = i < n_ids ? ids[i] : -1;
    const bool mine = v >= 0 && v % world == rank;
    const unsigned bal = __ballot_sync(kFull, mine);
    if (lane == 0) s_off[warp] = __popc(bal);
    __syncthreads();
    if (warp == 0) {
      const int c = lane < n_warps ? s_off[lane] : 0;
      int x = c;
      for (int o = 1; o < 32; o <<= 1) {
        const int y = __shfl_up_sync(kFull, x, o);
        if (lane >= o) x += y;
      }
      s_off[lane] = x - c;  // exclusive
      if (lane == 31) s_total = x;
    }
    __syncthreads();
    if (mine) {
      const int64_t p = base + s_off[warp] + __popc(bal & ((1u << lane) - 1u));
      ids_mine[p] = v;
      pos_mine[p] = i;
    }
    base += s_total;
    __syncthreads();  // (s_off / s_total are rewritten by the next block of ids)
  }
}
}  // namespace
}  // namespace lstep

int lstep::peer_plan_mine(const int64_t* ids, int64_t n_ids, int world, int rank, int64_t* ids_mine, int64_t* pos_mine, cudaStream_t st) {
  if (n_ids < 0 || world < 1 || rank < 0 || rank >= world || (n_ids > 0 && (!ids || !ids_mine || !pos_mine))) return LSTEP_ERR_INVALID_ARG;
  if (n_ids == 0) return LSTEP_OK;
  const int threads = (int)std::min<int64_t>(1024, ceil_div(n_ids, 32) * 32);
  peer_plan_kernel<<<1, threads, 0, st>>>(ids, n_ids, world, rank, ids_mine, pos_mine);
  return check_launch("peer_plan");
}

int lstep::peer_step_check(const lstep_pe_stream* s, const lstep_changelog* cl, const lstep_csr* csr, const lstep_peer_group* grp, int64_t n_edges,
                           int head, int len, const lstep_pe_mlp* mlp_nbr, const lstep_pe_mlp* mlp_upd, int phases, int64_t q_rows) {
  if (!s || !s->cur || !cl || !csr || !valid_group(grp) || n_edges < 0 || !mlp_nbr || !mlp_upd || (phases & ~7) || q_rows < 0)
    return LSTEP_ERR_INVALID_ARG;
  if (grp->table[grp->rank] != s->cur || cl->row_mul != grp->world || cl->row_add != grp->rank || cl->d != s->d) return LSTEP_ERR_INVALID_ARG;
  if (grp->world > 1 && grp->cap < cl->cap) return LSTEP_ERR_INVALID_ARG;
  if (head < 0 || head >= cl->T || len < 0 || len > cl->T) return LSTEP_ERR_INVALID_ARG;
  if (!update_push_available(mlp_upd)) return LSTEP_ERR_UNSUPPORTED;
  return LSTEP_OK;
}

// the resident form: the batch is edges [lo, lo + n_edges) of the descriptor's stream
static int step_peer_impl(const lstep_pe_stream* s, const lstep_changelog* cl, const lstep_csr* csr, const lstep_peer_group* grp, int64_t lo,
                          int64_t n_edges, const int64_t* ids, int64_t n_ids, const int64_t* ids_mine, const int64_t* pos_mine, int64_t n_mine,
                          double current_time, int head, int len, const float* G, const int64_t* const* query_ids_host, int n_queries,
                          int64_t q_off, int64_t q_rows, float* nbr_out, int K, const lstep_pe_mlp* mlp_nbr, const lstep_pe_mlp* mlp_upd,
                          void* workspace, size_t workspace_bytes, uint32_t* err_flag, uint32_t epoch_base, int timeout_ms, int phases,
                          void* stream, SideLane* side) {
  if (!s || !s->src || !s->dst || !s->t || lo < 0 || n_ids < 0 || n_mine < 0 || n_mine > n_ids) return LSTEP_ERR_INVALID_ARG;
  const int rc = peer_step_check(s, cl, csr, grp, n_edges, head, len, mlp_nbr, mlp_upd, phases, q_rows);
  if (rc != LSTEP_OK) return rc;
  return peer_step_core(s, cl, csr, grp, s->src + lo, s->dst + lo, s->t + lo, n_edges, ids, n_ids, ids_mine, pos_mine, n_mine, current_time, head,
                        len, G, query_ids_host, n_queries, q_off, q_rows, nbr_out, K, mlp_nbr, mlp_upd, workspace, workspace_bytes, err_flag,
                        epoch_base, timeout_ms, phases, stream, side);
}

extern "C" int lstep_pe_step_peer(const lstep_pe_stream* s, const lstep_changelog* cl, const lstep_csr* csr, const lstep_peer_group* grp,
                                  int64_t lo, int64_t n_edges, const int64_t* ids, int64_t n_ids, const int64_t* ids_mine,
                                  const int64_t* pos_mine, int64_t n_mine, double current_time, int head, int len, const float* G,
                                  const int64_t* const* query_ids_host, int n_queries, int64_t q_off, int64_t q_rows, float* nbr_out,
                                  int K, const lstep_pe_mlp* mlp_nbr, const lstep_pe_mlp* mlp_upd, void* workspace,
                                  size_t workspace_bytes, uint32_t* err_flag, uint32_t epoch_base, int timeout_ms, int phases,
                                  void* stream) {
  return step_peer_impl(s, cl, csr, grp, lo, n_edges, ids, n_ids, ids_mine, pos_mine, n_mine, current_time, head, len, G, query_ids_host, n_queries,
                        q_off, q_rows, nbr_out, K, mlp_nbr, mlp_upd, workspace, workspace_bytes, err_flag, epoch_base, timeout_ms, phases, stream,
                        nullptr);
}

// The step body on explicit batch pointers; the callers have made peer_step_check's checks.
int lstep::peer_step_core(const lstep_pe_stream* s, const lstep_changelog* cl, const lstep_csr* csr, const lstep_peer_group* grp, const int64_t* src,
                          const int64_t* dst, const double* tq, int64_t n_edges, const int64_t* ids, int64_t n_ids, const int64_t* ids_mine,
                          const int64_t* pos_mine, int64_t n_mine, double current_time, int head, int len, const float* G,
                          const int64_t* const* query_ids_host, int n_queries, int64_t q_off, int64_t q_rows, float* nbr_out, int K,
                          const lstep_pe_mlp* mlp_nbr, const lstep_pe_mlp* mlp_upd, void* workspace, size_t workspace_bytes, uint32_t* err_flag,
                          uint32_t epoch_base, int timeout_ms, int phases, void* stream, SideLane* side) {
  cudaStream_t st = as_stream(stream);
  int rc;
  if (phases & 1) {
    prof_mark(st, kProfStart);
    // the filtered rows go into the local table and, at the node's position in the batch's id list, into EVERY other rank's filt
    // buffer (a 2.7 MB region: stores into it do not thrash the peer TLB the way stores into the 6.9 GB replicas did)
    float* filt_dst[LSTEP_MAX_PEERS];
    int n_filt = 0;
    for (int g = 0; g < grp->world; ++g)
      if (g != grp->rank) filt_dst[n_filt++] = grp->filt[g];
    if (n_mine > 0 && (rc = changelog_filter_peer(cl, head, len, ids_mine, n_mine, G, s->cur, s->d, ids_mine, filt_dst, n_filt, pos_mine, stream)) !=
                          LSTEP_OK)
      return rc;
    // (a whole step in one call: the wait launch below announces the barrier itself)
    if ((phases & 2) == 0 && (rc = peer_signal(grp, epoch_base + 1, st)) != LSTEP_OK) return rc;
    prof_mark(st, kProfDft);
  }
  if (!(phases & 6)) return LSTEP_OK;
  if (phases & 2) {
    if (side && side->pending) {  // the previous step's publication (side stream) must be complete before this rank announces barrier 1
      if (cudaStreamWaitEvent(st, side->published, 0) != cudaSuccess) return LSTEP_ERR_CUDA;
      side->pending = false;
    }
    // (rows a step changes: ~ (K + 1) per batch node at most; the grid is sized for a typical 8 per batch node)
    if ((rc = peer_wait_apply(grp, epoch_base + 1, timeout_ms, err_flag, s->d, s->V1, n_ids * 8, ids, n_ids, st, (phases & 1) != 0)) != LSTEP_OK)
      return rc;
    prof_mark(st, kProfWait1);
  }
  PeerPlan plan;
  plan.grp = grp;
  plan.ids_mine = ids_mine;
  plan.pos_mine = pos_mine;
  plan.n_mine = n_mine;
  plan.epoch2 = epoch_base + 2;
  plan.timeout_ms = timeout_ms;
  plan.phases = phases & 6;
  int slot;
  rc = changelog_step_close(s, cl, csr, src, dst, tq, n_edges, ids, n_ids, current_time, head, len, query_ids_host, n_queries, q_off, q_rows,
                            nbr_out, K, mlp_nbr, mlp_upd, workspace, workspace_bytes, err_flag, stream, &plan, &slot);
  if (rc != LSTEP_OK || !(phases & 4)) return rc;
  if (side && grp->world > 1) {
    if (cudaEventRecord(side->appended, st) != cudaSuccess || cudaStreamWaitEvent(side->stream, side->appended, 0) != cudaSuccess)
      return LSTEP_ERR_CUDA;
    rc = peer_publish(cl, slot, grp, n_ids * 8 / grp->world + 1, side->stream);
    if (rc == LSTEP_OK && cudaEventRecord(side->published, side->stream) != cudaSuccess) return LSTEP_ERR_CUDA;
    side->pending = true;
  } else {
    rc = peer_publish(cl, slot, grp, n_ids * 8 / grp->world + 1, st);
  }
  prof_mark(st, kProfAppend);
  return rc;
}

extern "C" int lstep_pe_steps_peer(const lstep_pe_stream* s, const lstep_changelog* cl, const lstep_csr* csr, const lstep_peer_group* grp,
                                   int64_t n_steps, const int64_t* lo_host, const int64_t* n_edges_host, const double* tmax_host,
                                   const int64_t* ids, const int64_t* ids_off_host, const int64_t* ids_mine, const int64_t* pos_mine,
                                   const int64_t* mine_off_host, int* head_io, const float* G, const int64_t* const* query_ids_host,
                                   const int64_t* q_base_host, int n_queries, float* nbr_out, int64_t out_step_stride, int K,
                                   const lstep_pe_mlp* mlp_nbr, const lstep_pe_mlp* mlp_upd, void* workspace, size_t workspace_bytes,
                                   uint32_t* err_flag, uint32_t* epoch_io, int timeout_ms, void* stream) {
  if (!cl || !valid_group(grp) || n_steps < 0 || !lo_host || !n_edges_host || !tmax_host || !ids || !ids_off_host || !mine_off_host || !head_io ||
      !epoch_io || n_queries < 0 || n_queries > 8 || (n_queries > 0 && (!query_ids_host || !q_base_host)))
    return LSTEP_ERR_INVALID_ARG;
  const int T = cl->T;
  int head = *head_io;
  uint32_t epoch = *epoch_io;
  int rc = LSTEP_OK;
  SideLane lane;
  const bool overlap = grp->world > 1 && n_steps > 1;
  if (overlap && (rc = side_lane_open(&lane)) != LSTEP_OK) return rc;
  for (int64_t i = 0; i < n_steps; ++i) {
    const int64_t n = n_edges_host[i];
    const int64_t q_off = grp->rank * n / grp->world, q_rows = (grp->rank + 1) * n / grp->world - q_off;
    const int64_t* q[8] = {};
    for (int c = 0; c < n_queries; ++c) q[c] = query_ids_host[c] + q_base_host[i] + q_off;
    const int64_t m0 = mine_off_host[i], m1 = mine_off_host[i + 1];
    rc = step_peer_impl(s, cl, csr, grp, lo_host[i], n, ids + ids_off_host[i], ids_off_host[i + 1] - ids_off_host[i],
                        ids_mine ? ids_mine + m0 : nullptr, pos_mine ? pos_mine + m0 : nullptr, m1 - m0, tmax_host[i], head, T, G, q, n_queries, q_off,
                        q_rows, nbr_out ? nbr_out + i * out_step_stride : nullptr, K, mlp_nbr, mlp_upd, workspace, workspace_bytes, err_flag, epoch,
                        timeout_ms, 7, stream, overlap ? &lane : nullptr);
    if (rc != LSTEP_OK) break;
    epoch += 2;
    head = (head + 1) % T;
  }
  if (overlap) side_lane_close(&lane, as_stream(stream));
  *head_io = head;
  *epoch_io = epoch;
  return rc;
}
