// Change-log PE history (SURVEY §7 / §8(e) capacity caveat: "a versioned (change-log) history — piecewise-constant rows
// make the collapsed filter a [span sum] per version").
//
// The reference keeps the last T snapshots of the WHOLE table ([V1, T, d]: 688 GB at 10 M nodes, T = 100) although a step
// changes only the batch nodes and their sampled neighbours (~13 k of 10 M rows at B = 2000). The dense ring of the
// streaming API inherits that: every step writes one row per node (the H term, 2 * V1 * d * 4 B = 13.8 GB per step at
// 10 M nodes — 4.6 ms of pure copy against 0.3 ms of kernels). Here the same history is stored as
//
//     base[v]                 value of node v at the OLDEST step of the window (window index 0)
//     events[slot][e]         (node, row) for every row a step changed, one list per window step (ring over T slots),
//                             with a per-slot hash table node -> e and a per-node bit mask of the slots holding an event
//
// i.e. V1 + T * (rows changed per step) rows instead of V1 * T: 6.9 GB + 0.9 GB for the 10 M-node graph. It is exactly the
// same function of time: x[v, f] = row of the latest event of v at a window index <= f, else base[v].
//
//   filter   out[n, c] = sum_f G[f, c] x[n, f, c] = w_0[c] base[n, c] + sum_j w_j[c] row_j[c],  w_j[c] = sum of G[f, c] over the
//            window indices the version j covers (plain fp32 sums of G over the span: no prefix-sum differences, no
//            cancellation). A node costs (events in window + 1) row reads instead of T.
//   append   the rows a step changed are {sorted batch nodes} u {distinct phase-B destinations U}; U comes from the push
//            kernel's list, batch nodes already in U are recognised by the push kernel's stamp map. Each gets a slot in
//            the step's event list (atomic counter; order inside a step is irrelevant: lookups go through the hash).
//   retire   when the window slides, the events of the step that leaves become the nodes' new base rows.
//
// Node-id sharded groups: a rank keeps base rows / masks / events of the nodes it owns only (local row = (v - row_add) /
// row_mul for v % row_mul == row_add).
#include <algorithm>
#include <cstring>

#include "common.cuh"
#include "step_core.cuh"

namespace lstep {
namespace {

constexpr unsigned long long kEmpty = ~0ull;

__device__ __forceinline__ uint32_t hash_node(uint32_t v) {
  v ^= v >> 16;
  v *= 0x7feb352du;
  v ^= v >> 15;
  v *= 0x846ca68bu;
  v ^= v >> 16;
  return v;
}

__device__ __forceinline__ int hash_find(const unsigned long long* __restrict__ tab, int H, uint32_t node) {
  uint32_t h = hash_node(node) & (uint32_t)(H - 1);
  for (int probes = 0; probes < H; ++probes) {
    const unsigned long long e = __ldcg(tab + h);
    if (e == kEmpty) return -1;
    if ((uint32_t)(e >> 32) == node) return (int)(uint32_t)e;
    h = (h + 1) & (uint32_t)(H - 1);
  }
  return -1;
}

// Optional extra destinations of a filtered row (peer group, csrc/peer.cu): row n also goes to p[g] + ids[n] * out_stride — the
// other ranks' filt buffers, indexed by the node's position in the batch's id list (small, fixed regions of peer memory).
struct Out2 {
  float* p[LSTEP_MAX_PEERS];
  int n;
  const int64_t* ids;
};

// A node's value is piecewise constant over the window: version 0 = the base row, version j = the row of its j-th event;
// out = sum_j (sum of G over the window positions version j covers) * row_j.
// A node is a chain of dependent, random HBM reads (id -> event mask -> hash slots -> event rows) and almost no arithmetic:
// the kernel is as fast as the number of nodes it keeps in flight and as its longest chain. Measured at B = 2000
// (profiles/r02_ncu_scaleout_kernels.txt): a CTA per node = 592 nodes in flight, 6.4 waves, 64.7 us; a warp per node =
// one wave, but a hub with an event in every window step is 26 dependent rounds of row loads for ONE warp: 93 us.
// Hence both: every warp of a CTA looks its node up and, when the node has at most kFilterSmall events, finishes it alone
// (four versions = eight 16-byte loads per lane in flight); nodes with more events are then done by the whole CTA, the warps
// taking the versions round-robin and adding their partial sums in warp order (fixed: bit-reproducible).
// Lane l owns the column groups l and l + 32 (d/4 <= 64).
constexpr int kFilterWarps = 8;
constexpr int kFilterSmall = 11;  // versions incl. the base row: 12 = three rounds of four
struct FilterAcc {
  float4 a0, a1;
};
// adds versions jj = first, first + stride, ... <= ne of one node to (a0, a1): the lane's two column groups
__device__ __forceinline__ void filter_versions(const lstep_changelog& cl, int head, int64_t lrow, const int* s_evf, const int* s_evi, int ne,
                                                int first, int stride, const float4* __restrict__ Gv, int lane, bool has2, FilterAcc& acc) {
  const int d = cl.d, dvec = d >> 2, T = cl.T;
  for (int j0 = first; j0 <= ne; j0 += 4 * stride) {
    float4 r0[4], r1[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int jj = j0 + u * stride;
      if (jj <= ne) {
        const float4* row;
        if (jj == 0)
          row = reinterpret_cast<const float4*>(cl.base + lrow * (int64_t)d);
        else {
          const int slot = (head + s_evf[jj - 1]) % T;
          row = reinterpret_cast<const float4*>(cl.ev_row + ((size_t)slot * cl.cap + s_evi[jj - 1]) * d);
        }
        r0[u] = __ldcg(row + lane);
        if (has2) r1[u] = __ldcg(row + lane + 32);
      }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int jj = j0 + u * stride;
      if (jj <= ne) {
        const int f0 = jj == 0 ? 0 : s_evf[jj - 1], f1 = s_evf[jj];
        float4 w0 = make_float4(0.f, 0.f, 0.f, 0.f), w1 = w0;  // sums of G over [f0, f1): plain fp32 sums, no prefix differences
#pragma unroll 4
        for (int f = f0; f < f1; ++f) {
          const float4 g0 = __ldg(Gv + (size_t)f * dvec + lane);
          w0.x += g0.x;
          w0.y += g0.y;
          w0.z += g0.z;
          w0.w += g0.w;
          if (has2) {
            const float4 g1 = __ldg(Gv + (size_t)f * dvec + lane + 32);
            w1.x += g1.x;
            w1.y += g1.y;
            w1.z += g1.z;
            w1.w += g1.w;
          }
        }
        acc.a0.x = fmaf(w0.x, r0[u].x, acc.a0.x);
        acc.a0.y = fmaf(w0.y, r0[u].y, acc.a0.y);
        acc.a0.z = fmaf(w0.z, r0[u].z, acc.a0.z);
        acc.a0.w = fmaf(w0.w, r0[u].w, acc.a0.w);
        if (has2) {
          acc.a1.x = fmaf(w1.x, r1[u].x, acc.a1.x);
          acc.a1.y = fmaf(w1.y, r1[u].y, acc.a1.y);
          acc.a1.z = fmaf(w1.z, r1[u].z, acc.a1.z);
          acc.a1.w = fmaf(w1.w, r1[u].w, acc.a1.w);
        }
      }
    }
  }
}
__device__ __forceinline__ void filter_store(float* __restrict__ out, int64_t orow, int64_t out_stride, int lane, bool has2, const FilterAcc& acc,
                                             const Out2& o2, int64_t n) {
  *reinterpret_cast<float4*>(out + orow * out_stride + 4 * lane) = acc.a0;
  if (has2) *reinterpret_cast<float4*>(out + orow * out_stride + 4 * (lane + 32)) = acc.a1;
  if (o2.n) {
    const int64_t off = o2.ids[n] * out_stride;
    for (int g = 0; g < o2.n; ++g) {
      *reinterpret_cast<float4*>(o2.p[g] + off + 4 * lane) = acc.a0;
      if (has2) *reinterpret_cast<float4*>(o2.p[g] + off + 4 * (lane + 32)) = acc.a1;
    }
  }
}

__global__ void __launch_bounds__(kFilterWarps * 32, 2) changelog_filter_kernel(lstep_changelog cl, int head, int len, const int64_t* __restrict__ ids,
                                                                                int64_t n_ids, const float* __restrict__ G, float* __restrict__ out,
                                                                                int64_t out_stride, const int64_t* __restrict__ out_ids,
                                                                                Out2 o2) {
  __shared__ int s_evf_all[kFilterWarps][130];  // window positions that carry an event (ascending), then `len`
  __shared__ int s_evi_all[kFilterWarps][129];  // their event indices
  __shared__ int s_ne[kFilterWarps];            // events of the warp's node, -1: no node / done by the warp itself
  __shared__ float4 s_part[kFilterWarps][64];   // partial sums of a node the whole CTA works on
  pdl_wait();
  pdl_launch_dependents();
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  int* s_evf = s_evf_all[wid];
  int* s_evi = s_evi_all[wid];
  const int dvec = cl.d >> 2, T = cl.T;
  const bool has2 = lane + 32 < dvec;
  const float4* Gv = reinterpret_cast<const float4*>(G);
  for (int64_t nb = (int64_t)blockIdx.x * kFilterWarps; nb < n_ids; nb += (int64_t)gridDim.x * kFilterWarps) {
    const int64_t n = nb + wid;
    int ne = -1;
    int64_t lrow = 0;
    if (n < n_ids) {
      const int64_t v = ids[n];
      lrow = (v - cl.row_add) / cl.row_mul;
      // ---- which window positions carry an event of v: lane l looks at positions l, l+32, l+64, l+96 (independent probes)
      const uint4 mask = __ldcg(reinterpret_cast<const uint4*>(cl.ev_mask + lrow * 4));
      int idx[4];
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        const int f = lane + 32 * r;
        idx[r] = -1;
        if (f < len) {
          const int slot = (head + f) % T;
          const uint32_t mw = (slot >> 5) == 0 ? mask.x : (slot >> 5) == 1 ? mask.y : (slot >> 5) == 2 ? mask.z : mask.w;
          if (mw & (1u << (slot & 31))) idx[r] = hash_find(cl.ev_hash + (size_t)slot * cl.H, cl.H, (uint32_t)v);
        }
      }
      ne = 0;
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        const unsigned m = __ballot_sync(kFull, idx[r] >= 0);
        if (idx[r] >= 0) {
          const int pos = ne + __popc(m & ((1u << lane) - 1));
          s_evf[pos] = lane + 32 * r;
          s_evi[pos] = idx[r];
        }
        ne += __popc(m);
      }
      if (lane == 0) s_evf[ne] = len;
      __syncwarp();
      if (ne <= kFilterSmall) {  // the warp finishes its node alone
        if (lane < dvec) {
          FilterAcc acc{make_float4(0.f, 0.f, 0.f, 0.f), make_float4(0.f, 0.f, 0.f, 0.f)};
          filter_versions(cl, head, lrow, s_evf, s_evi, ne, 0, 1, Gv, lane, has2, acc);
          filter_store(out, out_ids ? out_ids[n] : n, out_stride, lane, has2, acc, o2, n);
        }
        ne = -1;
      }
    }
    if (lane == 0) s_ne[wid] = ne;
    __syncthreads();
    // ---- nodes with many events: the whole CTA, versions round-robin over the warps
    for (int w = 0; w < kFilterWarps; ++w) {
      const int ne_w = s_ne[w];
      if (ne_w < 0) continue;  // (uniform over the CTA)
      const int64_t n_w = nb + w;
      const int64_t lrow_w = (ids[n_w] - cl.row_add) / cl.row_mul;
      FilterAcc acc{make_float4(0.f, 0.f, 0.f, 0.f), make_float4(0.f, 0.f, 0.f, 0.f)};
      if (lane < dvec) {
        filter_versions(cl, head, lrow_w, s_evf_all[w], s_evi_all[w], ne_w, wid, kFilterWarps, Gv, lane, has2, acc);
        if (wid > 0) {
          s_part[wid][lane] = acc.a0;
          if (has2) s_part[wid][lane + 32] = acc.a1;
        }
      }
      __syncthreads();
      if (wid == 0 && lane < dvec) {
        for (int x = 1; x < kFilterWarps; ++x) {
          const float4 p0 = s_part[x][lane];
          acc.a0.x += p0.x;
          acc.a0.y += p0.y;
          acc.a0.z += p0.z;
          acc.a0.w += p0.w;
          if (has2) {
            const float4 p1 = s_part[x][lane + 32];
            acc.a1.x += p1.x;
            acc.a1.y += p1.y;
            acc.a1.z += p1.z;
            acc.a1.w += p1.w;
          }
        }
        filter_store(out, out_ids ? out_ids[n_w] : n_w, out_stride, lane, has2, acc, o2, n_w);
      }
      __syncthreads();
    }
  }
  if (o2.n) __threadfence_system();
}

// The events of `slot` (the step leaving the window) become base rows; their mask bits are cleared; the slot is made ready
// for the step's new events: hash table emptied, event count reset by the block that finishes last (the blocks count
// themselves in the bits above kCntBits of the same word, so no separate launch or memset sits between retire and append).
constexpr int kCntBits = 20;  // cap < 2^20 events per step
__global__ void __launch_bounds__(256) changelog_retire_kernel(lstep_changelog cl, int slot) {
  pdl_wait();  // (everything before this kernel is complete; the successor may become resident now)
  pdl_launch_dependents();
  const int cnt = min((int)((unsigned)__ldcg(cl.ev_cnt + slot) & ((1u << kCntBits) - 1)), cl.cap);
  const int dvec = cl.d >> 2;
  const int64_t total = (int64_t)cnt * dvec;
  const int64_t gtid = blockIdx.x * (int64_t)blockDim.x + threadIdx.x, nthr = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = gtid; i < total; i += nthr) {
    const int e = (int)(i / dvec), c = (int)(i % dvec);
    const int64_t v = cl.ev_node[(size_t)slot * cl.cap + e];
    const int64_t lrow = (v - cl.row_add) / cl.row_mul;
    reinterpret_cast<float4*>(cl.base + lrow * (int64_t)cl.d)[c] =
        reinterpret_cast<const float4*>(cl.ev_row + ((size_t)slot * cl.cap + e) * cl.d)[c];
    if (c == 0) atomicAnd(cl.ev_mask + lrow * 4 + (slot >> 5), ~(1u << (slot & 31)));
  }
  ulonglong2* tab = reinterpret_cast<ulonglong2*>(cl.ev_hash + (size_t)slot * cl.H);  // H is a power of two >= 2
  for (int64_t i = gtid; i < cl.H / 2; i += nthr) tab[i] = make_ulonglong2(kEmpty, kEmpty);
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned old = atomicAdd(reinterpret_cast<unsigned*>(cl.ev_cnt + slot), 1u << kCntBits);
    if ((old >> kCntBits) == gridDim.x - 1) cl.ev_cnt[slot] = 0;  // every block has read the count
  }
}

// Items [0, nU) = the distinct phase-B destinations U (nU read from the device when n_u_dev != NULL), items [nU, nU + n_ids)
// = the batch nodes, skipped when the stamp map says U already holds them, then (with_row0) the padding row.
// One THREAD decides one item (owned? already covered?), a block of 256 items draws its event indices with ONE atomic on the
// slot's counter (one atomic per item serialised 48 k same-address atomics at B = 2000: 60 us, all of it waiting for the
// counter), every thread records its own event (node, hash entry, mask bit), and the warps then copy the rows of their 32
// items, four rows in flight.
__global__ void __launch_bounds__(256) changelog_append_kernel(lstep_changelog cl, int slot, const float* __restrict__ table,
                                                               const int64_t* __restrict__ U, const int32_t* __restrict__ n_u_dev, int64_t n_u,
                                                               const int64_t* __restrict__ ids, int64_t n_ids,
                                                               const int32_t* __restrict__ stamp_map, int stamp, int with_row0,
                                                               uint32_t* err_flag) {
  __shared__ int s_cnt[8];
  __shared__ int s_base;
  pdl_wait();
  pdl_launch_dependents();
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  if (n_u_dev) {
    const int64_t nd = __ldcg(n_u_dev);
    n_u = nd < n_u ? nd : n_u;
  }
  const int dvec = cl.d >> 2;
  const int64_t n_items = n_u + n_ids + (with_row0 ? 1 : 0);
  for (int64_t base = (int64_t)blockIdx.x * 256; base < n_items; base += (int64_t)gridDim.x * 256) {
    const int64_t it = base + tid;
    int64_t v = -1;
    if (it < n_items) {
      if (it < n_u) {
        v = __ldcg(reinterpret_cast<const long long*>(U) + it);
      } else {
        // a batch node, or (last item) the padding row 0, which update_pe zeroes in every call (LSTEP.py:317)
        v = it < n_u + n_ids ? ids[it - n_u] : 0;
        if (it == n_u + n_ids && n_ids > 0 && ids[0] == 0) v = -1;
        if (v >= 0 && U && stamp_map && __ldcg(stamp_map + v) == stamp) v = -1;  // phase B changed this row too: U holds it
      }
      if (v >= 0 && v % cl.row_mul != cl.row_add) v = -1;  // not owned by this rank
    }
    const unsigned m = __ballot_sync(kFull, v >= 0);
    if (lane == 0) s_cnt[wid] = __popc(m);
    __syncthreads();
    if (tid == 0) {
      int tot = 0;
      for (int w = 0; w < 8; ++w) tot += s_cnt[w];
      s_base = tot ? atomicAdd(cl.ev_cnt + slot, tot) : 0;
    }
    __syncthreads();
    int idx = s_base + __popc(m & ((1u << lane) - 1));
    for (int w = 0; w < wid; ++w) idx += s_cnt[w];
    if (v >= 0) {
      if (idx >= cl.cap) {
        if (err_flag) atomicOr(err_flag, LSTEP_FLAG_CHANGELOG_FULL);
      } else {
        const int64_t lrow = (v - cl.row_add) / cl.row_mul;
        cl.ev_node[(size_t)slot * cl.cap + idx] = (int32_t)v;
        unsigned long long* tab = cl.ev_hash + (size_t)slot * cl.H;
        const unsigned long long entry = ((unsigned long long)(uint32_t)v << 32) | (uint32_t)idx;
        uint32_t h = hash_node((uint32_t)v) & (uint32_t)(cl.H - 1);
        while (atomicCAS(tab + h, kEmpty, entry) != kEmpty) h = (h + 1) & (uint32_t)(cl.H - 1);
        atomicOr(cl.ev_mask + lrow * 4 + (slot >> 5), 1u << (slot & 31));
      }
    }
    // ---- rows: the warp copies table[v] -> event row for its valid items, four at a time
    unsigned mm = __ballot_sync(kFull, v >= 0 && idx < cl.cap);
    while (mm) {
      const float4* srow[4];
      float4* drow[4];
      int nq = 0;
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        if (mm) {
          const int src = __ffs(mm) - 1;
          mm &= mm - 1;
          const int64_t vv = __shfl_sync(kFull, v, src);
          const int ii = __shfl_sync(kFull, idx, src);
          srow[q] = reinterpret_cast<const float4*>(table + vv * (int64_t)cl.d);
          drow[q] = reinterpret_cast<float4*>(cl.ev_row + ((size_t)slot * cl.cap + ii) * cl.d);
          nq = q + 1;
        }
      }
      for (int c = lane; c < dvec; c += 32) {
        float4 x[4];
#pragma unroll
        for (int q = 0; q < 4; ++q)
          if (q < nq) x[q] = __ldcg(srow[q] + c);
#pragma unroll
        for (int q = 0; q < 4; ++q)
          if (q < nq) drow[q][c] = x[q];
      }
    }
    __syncthreads();
  }
}

bool valid(const lstep_changelog* cl) {
  return cl && cl->base && cl->ev_node && cl->ev_row && cl->ev_cnt && cl->ev_hash && cl->ev_mask && cl->rows > 0 && cl->T > 0 && cl->T <= 128 &&
         cl->cap > 0 && cl->cap < (1 << kCntBits) && cl->H >= 2 * cl->cap && (cl->H & (cl->H - 1)) == 0 && cl->d > 0 && cl->d % 4 == 0 && cl->d <= 512 && cl->row_mul > 0 &&
         cl->row_add >= 0 && cl->row_add < cl->row_mul;
}

}  // namespace

}  // namespace lstep

using namespace lstep;

namespace lstep {
int changelog_filter_peer(const lstep_changelog* cl, int head, int len, const int64_t* ids, int64_t n_ids, const float* G, float* out,
                          int64_t out_stride, const int64_t* out_ids, float* const* out2, int n_out2, const int64_t* out2_ids, void* stream);
}  // namespace lstep

extern "C" int lstep_changelog_filter(const lstep_changelog* cl, int head, int len, const int64_t* ids, int64_t n_ids, const float* G,
                                      float* out, int64_t out_stride, const int64_t* out_ids, void* stream) {
  return changelog_filter_peer(cl, head, len, ids, n_ids, G, out, out_stride, out_ids, nullptr, 0, nullptr, stream);
}
int lstep::changelog_filter_peer(const lstep_changelog* cl, int head, int len, const int64_t* ids, int64_t n_ids, const float* G, float* out,
                                 int64_t out_stride, const int64_t* out_ids, float* const* out2, int n_out2, const int64_t* out2_ids, void* stream) {
  if (n_out2 < 0 || n_out2 > LSTEP_MAX_PEERS || (n_out2 > 0 && (!out2 || !out2_ids))) return LSTEP_ERR_INVALID_ARG;
  Out2 o2{};
  for (int g = 0; g < n_out2; ++g) o2.p[g] = out2[g];
  o2.n = n_out2;
  o2.ids = out2_ids;
  if (!valid(cl) || head < 0 || head >= cl->T || len < 0 || len > cl->T || n_ids < 0) return LSTEP_ERR_INVALID_ARG;
  if (n_ids == 0) return LSTEP_OK;
  if (!ids || !G || !out || out_stride % 4 != 0 || (reinterpret_cast<uintptr_t>(out) & 15)) return LSTEP_ERR_INVALID_ARG;
  if (cl->d > 256) return LSTEP_ERR_UNSUPPORTED;  // (a lane owns two 16-byte column groups)
  const int64_t grid = std::min<int64_t>(ceil_div(n_ids, kFilterWarps), (int64_t)num_sms() * 8);
  launch_k(changelog_filter_kernel, dim3((unsigned)grid), dim3(kFilterWarps * 32), 0, as_stream(stream), *cl, head, len, ids, n_ids, G, out, out_stride,
           out_ids, o2);
  return check_launch("changelog_filter");
}

/* Close a step: when `retire` is set the events of `slot` (the oldest step, leaving the window) are folded into the base rows
 * first; then the rows of `table` for U[0 .. n_u) (n_u = min(n_u, *n_u_dev) when n_u_dev != NULL) and for the ids whose
 * stamp_map entry differs from `stamp` become the slot's new events. */
extern "C" int lstep_changelog_append(const lstep_changelog* cl, int slot, int retire, const float* table, const int64_t* U,
                                      const int32_t* n_u_dev, int64_t n_u, const int64_t* ids, int64_t n_ids, const int32_t* stamp_map,
                                      int stamp, int with_row0, uint32_t* err_flag, void* stream) {
  if (!valid(cl) || slot < 0 || slot >= cl->T || n_u < 0 || n_ids < 0 || !table) return LSTEP_ERR_INVALID_ARG;
  if ((n_u > 0 && !U) || (n_ids > 0 && !ids)) return LSTEP_ERR_INVALID_ARG;
  cudaStream_t st = as_stream(stream);
  cudaError_t e;
  if (retire) {  // (also empties the slot's hash table and resets its event count)
    launch_k(changelog_retire_kernel, dim3((unsigned)num_sms() * 2), dim3(256), 0, st, *cl, slot);
    int rc = check_launch("changelog_retire");
    if (rc != LSTEP_OK) return rc;
  } else if ((e = cudaMemsetAsync(cl->ev_hash + (size_t)slot * cl->H, 0xff, sizeof(unsigned long long) * cl->H, st)) != cudaSuccess ||
             (e = cudaMemsetAsync(cl->ev_cnt + slot, 0, sizeof(int32_t), st)) != cudaSuccess) {  // (history still filling)
    set_cuda_error(e, "changelog memset");
    return LSTEP_ERR_CUDA;
  }
  if (n_u + n_ids == 0 && !with_row0) return LSTEP_OK;
  const int64_t grid = std::min<int64_t>(ceil_div(n_u + n_ids + 1, 256), (int64_t)num_sms() * 8);
  launch_k(changelog_append_kernel, dim3((unsigned)grid), dim3(256), 0, st, *cl, slot, table, U, n_u_dev, n_u, ids, n_ids, stamp_map, stamp, with_row0,
           err_flag);
  return check_launch("changelog_append");
}

namespace lstep {
// The argument checks of the change-log step that do not concern the batch pointers (every caller makes them before it
// enqueues anything, so a host-fed call rejects bad arguments before its copy-in and append).
int changelog_step_check(const lstep_pe_stream* s, const lstep_changelog* cl, int head, int len, const lstep_pe_mlp* mlp_upd) {
  if (!s || !s->cur || !valid(cl) || !mlp_upd) return LSTEP_ERR_INVALID_ARG;
  if (cl->d != s->d || head < 0 || head >= cl->T || len < 0 || len > cl->T) return LSTEP_ERR_INVALID_ARG;
  if (!update_push_available(mlp_upd)) return LSTEP_ERR_UNSUPPORTED;  // the append needs the push kernel's U list and stamp map
  return LSTEP_OK;
}

// The change-log step on explicit batch pointers (src/dst/tq = the batch's n_edges endpoints and times on the device): the
// resident lstep_pe_step_changelog passes the stream's edges, the host-fed calls (csrc/host_step.cu) their staged slot.
// Never reads s->src / s->dst / s->t.
int changelog_step_core(const lstep_pe_stream* s, const lstep_changelog* cl, const lstep_csr* csr, const int64_t* src, const int64_t* dst,
                        const double* tq, int64_t n_edges, const int64_t* ids, int64_t n_ids, double current_time, int head, int len,
                        const float* G, const int64_t* const* query_ids_host, int n_queries, int64_t q_off, int64_t q_rows, float* nbr_out,
                        int K, const lstep_pe_mlp* mlp_nbr, const lstep_pe_mlp* mlp_upd, void* workspace, size_t workspace_bytes,
                        uint32_t* err_flag, void* stream, int phase) {
  if (n_edges < 0 || n_ids < 0) return LSTEP_ERR_INVALID_ARG;
  int rc = changelog_step_check(s, cl, head, len, mlp_upd);
  if (rc != LSTEP_OK) return rc;
  if (phase != 2 && n_ids > 0) {
    if (cl->row_mul != 1) return LSTEP_ERR_INVALID_ARG;  // sharded groups filter through lstep_changelog_filter themselves
    if ((rc = lstep_changelog_filter(cl, head, len, ids, n_ids, G, s->cur, s->d, ids, stream)) != LSTEP_OK) return rc;
  }
  if (phase == 1) return LSTEP_OK;
  int slot;
  return changelog_step_close(s, cl, csr, src, dst, tq, n_edges, ids, n_ids, current_time, head, len, query_ids_host, n_queries, q_off, q_rows,
                              nbr_out, K, mlp_nbr, mlp_upd, workspace, workspace_bytes, err_flag, stream, nullptr, &slot);
}

int changelog_step_close(const lstep_pe_stream* s, const lstep_changelog* cl, const lstep_csr* csr, const int64_t* src, const int64_t* dst,
                         const double* tq, int64_t n_edges, const int64_t* ids, int64_t n_ids, double current_time, int head, int len,
                         const int64_t* const* query_ids_host, int n_queries, int64_t q_off, int64_t q_rows, float* nbr_out, int K,
                         const lstep_pe_mlp* mlp_nbr, const lstep_pe_mlp* mlp_upd, void* workspace, size_t workspace_bytes,
                         uint32_t* err_flag, void* stream, const PeerPlan* peer, int* slot) {
  StepOpts opt;
  opt.skip_dft = opt.skip_append = true;
  opt.q_off = q_off;
  opt.q_rows = q_rows;
  opt.peer = peer;
  int stamp = 0;
  opt.stamp_out = &stamp;
  lstep_pe_stream s2 = *s;
  if (!s2.ring) s2.ring = s2.cur;  // (never touched: the core neither filters nor appends)
  const int64_t qr = q_rows < 0 ? n_edges : q_rows;
  int rc = pe_step_core_ex(&s2, csr, src, dst, tq, n_edges, ids, n_ids, current_time, 0, 0, 0, nullptr, query_ids_host, qr > 0 ? n_queries : 0,
                           nbr_out, K, mlp_nbr, mlp_upd, workspace, workspace_bytes, err_flag, stream, opt);
  if (rc != LSTEP_OK || (peer && !(peer->phases & 4))) return rc;
  const int64_t* U = nullptr;
  const int32_t *n_dest = nullptr, *stamp_map = nullptr;
  int64_t n_u_max = 0;
  if (n_ids > 0) {
    update_ws_phase_b_lists(workspace, n_ids, n_edges, K, s->d, mlp_upd->t, pe_ws_rows(s), &U, &n_dest, &stamp_map);
    const int64_t total = n_ids * (int64_t)K;
    n_u_max = (total < s->V1 - 1 ? total : s->V1 - 1) + 1;
  }
  const bool full = len == cl->T;
  *slot = full ? head : (head + len) % cl->T;
  return lstep_changelog_append(cl, *slot, full ? 1 : 0, s->cur, U, n_dest, n_u_max, ids, n_ids, stamp_map, stamp, n_ids > 0 ? 1 : 0, err_flag,
                                stream);
}
}  // namespace lstep

/* lstep_pe_step on a change-log history: filter of the batch nodes into the table, the step's kernels, retire + append.
 * head / len: the window (slot of its oldest step, number of valid steps <= T); the step's events go to slot
 * (head + len) % T while the history is filling, to `head` (after retiring it) once len == T. q_off / q_rows as in
 * lstep_pe_step_sharded (q_rows < 0: all edges). filter_ids / n_filter: the batch nodes whose history THIS rank holds
 * (= ids for a single GPU); their filtered rows are written to filter_out (row i, pitch d) when filter_out != NULL — the
 * caller all-gathers and scatters them — and straight into the table otherwise. */
extern "C" int lstep_pe_step_changelog(const lstep_pe_stream* s, const lstep_changelog* cl, const lstep_csr* csr, int64_t lo, int64_t n_edges,
                                       const int64_t* ids, int64_t n_ids, double current_time, int head, int len, const float* G,
                                       const int64_t* const* query_ids_host, int n_queries, int64_t q_off, int64_t q_rows, float* nbr_out,
                                       int K, const lstep_pe_mlp* mlp_nbr, const lstep_pe_mlp* mlp_upd, void* workspace,
                                       size_t workspace_bytes, uint32_t* err_flag, void* stream, int phase) {
  // phase 0: everything; 1: filter only (into filter destination = table); 2: everything after the filter
  if (!s || !s->src || !s->dst || !s->t || !s->cur || !valid(cl) || lo < 0 || n_edges < 0 || n_ids < 0 || !mlp_upd) return LSTEP_ERR_INVALID_ARG;
  return changelog_step_core(s, cl, csr, s->src + lo, s->dst + lo, s->t + lo, n_edges, ids, n_ids, current_time, head, len, G, query_ids_host,
                             n_queries, q_off, q_rows, nbr_out, K, mlp_nbr, mlp_upd, workspace, workspace_bytes, err_flag, stream, phase);
}
