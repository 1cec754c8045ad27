// Bodies of the two read-only gather kernels of a step, shared by their stand-alone kernels
// (csrc/aggregate.cu, csrc/update.cu) and by the fused launch of the streaming step (csrc/step.cu): the
// neighbourhood aggregate of the C query sets (a6) and phase A's edge aggregate (a7) both only READ the
// current table, so one heterogeneous grid runs them side by side.
#pragma once
#include "common.cuh"

namespace lstep {

// kLookup: the kernel does the most-recent-K lookup itself (warp 0, warp_recent_range) instead of reading the
// sampler's output — the streaming step's form: one launch and no [rows, K] round trip through global memory.
struct LookupArgs {
  const int64_t* indptr;
  const int32_t* c_nbr;
  const double* c_t;
  int64_t num_rows;
  RowIds q_node;
  uint32_t* err_flag;
};

template <int VEC, bool kLookup>
__device__ __forceinline__ void nbr_aggregate_rows(int64_t first_row, int64_t row_stride, bool late_wait, const float* __restrict__ pe,
                                                            const double* __restrict__ q_time,
                                                            const int32_t* __restrict__ nbr,
                                                            const float* __restrict__ nbr_t, int64_t n_rows, int K,
                                                            const float* __restrict__ tw, int d, int t, int t_pad,
                                                            float* __restrict__ S, int64_t ldS, int64_t period, LookupArgs lk) {
  // thread f < t owns time frequency f and adds its K cosines in order k = 0 .. K-1
  extern __shared__ __align__(16) unsigned char smem_raw[];
  int32_t* s_nbr = reinterpret_cast<int32_t*>(smem_raw);
  float* s_dt = reinterpret_cast<float*>(s_nbr + K);
  const int tid = threadIdx.x;
  const int dvec = d / VEC;
  for (int64_t row = first_row; row < n_rows; row += row_stride) {
    const double tq = q_time[period ? row % period : row];
    if (kLookup) {
      if (tid < 32) {
        const int64_t node = lk.q_node.at(row);
        int64_t first = 0;
        int take = 0;
        if (node < 0 || node >= lk.num_rows) {
          if (tid == 0 && lk.err_flag) atomicOr(lk.err_flag, LSTEP_FLAG_NODE_OUT_OF_RANGE);
        } else {
          warp_recent_range(lk.indptr, lk.c_t, node, tq, K, tid, first, take);
        }
        const int pad = K - take;
        for (int k = tid; k < K; k += 32) {
          int32_t n = 0;
          float tt = 0.f;
          if (k >= pad) {
            const int64_t e = first + (k - pad);
            n = lk.c_nbr[e];
            tt = (float)lk.c_t[e];  // the sampler returns fp32 times (utils.py:166,208)
          }
          s_nbr[k] = n;
          s_dt[k] = (float)(tq - (double)tt);  // f64 - f32 promotes to f64, then .float() (LSTEP.py:228-230)
        }
      }
    } else {
      for (int k = tid; k < K; k += blockDim.x) {
        s_nbr[k] = ld_dep(nbr + row * K + k);
        // f64 - f32 promotes to f64, then .float() (LSTEP.py:228-230)
        s_dt[k] = (float)(tq - (double)ld_dep(nbr_t + row * K + k));
      }
    }
    __syncthreads();
#ifdef LSTEP_TIMELINE
    if (late_wait && tid == 0) atomicMax(&g_timeline[6 * 4 + 2], gtimer());  // last lookup done
#endif
    if (tid < t) {
      float acc = 0.f;
      const float w = tw[tid];
      for (int k = 0; k < K; ++k)
        if (s_nbr[k] != 0) acc += time_feature(s_dt[k], w);
      S[row * ldS + d + tid] = acc;
#ifdef LSTEP_TIMELINE
      if (late_wait && tid == 0) atomicMax(&g_timeline[7 * 4 + 2], gtimer());  // last cosine block done
#endif
    }
    if (tid >= t_pad && tid - t_pad < dvec) {
      // late_wait (fused launch of the streaming step): lookups and cosines depend on nothing the kernel in front
      // writes, so only the threads that read the table wait for it
      if (late_wait) {
        pdl_wait();
#ifdef LSTEP_TIMELINE
        if (tid == t_pad) atomicMin(&g_timeline[1 * 4 + 1], gtimer());
        if (tid == t_pad) atomicMax(&g_timeline[8 * 4 + 2], gtimer());  // last wait return (nbr rows)
#endif
      }
      const int cv = tid - t_pad;
      if (VEC == 4) {
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        int k = 0;
        // the K row loads sit on the step's critical path (they wait for the kernel in front): 10 in flight per thread
        // (one L2 round trip per 10 rows), added in order k = 0..K-1
        for (; k + 10 <= K; k += 10) {
          float4 v[10];
#pragma unroll
          for (int u = 0; u < 10; ++u)
            v[u] = ld_dep(reinterpret_cast<const float4*>(pe + (int64_t)s_nbr[k + u] * d) + cv);
#pragma unroll
          for (int u = 0; u < 10; ++u) {
            acc.x += v[u].x;
            acc.y += v[u].y;
            acc.z += v[u].z;
            acc.w += v[u].w;
          }
        }
        for (; k + 4 <= K; k += 4) {
          float4 v[4];
#pragma unroll
          for (int u = 0; u < 4; ++u)
            v[u] = ld_dep(reinterpret_cast<const float4*>(pe + (int64_t)s_nbr[k + u] * d) + cv);
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            acc.x += v[u].x;
            acc.y += v[u].y;
            acc.z += v[u].z;
            acc.w += v[u].w;
          }
        }
        for (; k < K; ++k) {
          const float4 v = ld_dep(reinterpret_cast<const float4*>(pe + (int64_t)s_nbr[k] * d) + cv);
          acc.x += v.x;
          acc.y += v.y;
          acc.z += v.z;
          acc.w += v.w;
        }
        reinterpret_cast<float4*>(S + row * ldS)[cv] = acc;
      } else {
        float acc = 0.f;
        for (int k = 0; k < K; ++k) acc += ld_dep(pe + (int64_t)s_nbr[k] * d + cv);
        S[row * ldS + cv] = acc;
      }
    }
    __syncthreads();
  }
}

// The same rows for launches in which a CTA walks SEVERAL query rows (B = 2000: 6 000 rows over one wave of CTAs): an extra warp
// (threads [lk_base, lk_base + 32)) does nothing but the most-recent-K lookups and runs ONE ROW AHEAD of the cosine / table
// threads through a double-buffered neighbour list — the lookup is a chain of ~5 dependent L2 / HBM round trips (~3 us)
// during which, in the form above, the other 160 threads of the CTA wait. Same arithmetic, same order: results are
// bit-identical to nbr_aggregate_rows. (float4 table path only; late_wait as above.)
__device__ __forceinline__ void nbr_aggregate_rows_piped(int64_t first_row, int64_t row_stride, bool late_wait, const float* __restrict__ pe,
                                                         const double* __restrict__ q_time, int64_t n_rows, int K,
                                                         const float* __restrict__ tw, int d, int t, int t_pad, float* __restrict__ S,
                                                         int64_t ldS, int64_t period, LookupArgs lk, int lk_base) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  int32_t* s_nbr_all = reinterpret_cast<int32_t*>(smem_raw);       // [2][K]
  float* s_dt_all = reinterpret_cast<float*>(s_nbr_all + 2 * K);   // [2][K]
  const int tid = threadIdx.x;
  const int dvec = d / 4;
  const bool is_lk = tid >= lk_base && tid < lk_base + 32;
  const int lane = tid - lk_base;
  auto lookup = [&](int64_t row, int buf) {  // (lookup warp only)
    int32_t* s_nbr = s_nbr_all + buf * K;
    float* s_dt = s_dt_all + buf * K;
    const double tq = q_time[period ? row % period : row];
    const int64_t node = lk.q_node.at(row);
    int64_t first = 0;
    int take = 0;
    if (node < 0 || node >= lk.num_rows) {
      if (lane == 0 && lk.err_flag) atomicOr(lk.err_flag, LSTEP_FLAG_NODE_OUT_OF_RANGE);
    } else {
      warp_recent_range(lk.indptr, lk.c_t, node, tq, K, lane, first, take);
    }
    const int pad = K - take;
    for (int k = lane; k < K; k += 32) {
      int32_t n = 0;
      float tt = 0.f;
      if (k >= pad) {
        const int64_t e = first + (k - pad);
        n = lk.c_nbr[e];
        tt = (float)lk.c_t[e];  // the sampler returns fp32 times (utils.py:166,208)
      }
      s_nbr[k] = n;
      s_dt[k] = (float)(tq - (double)tt);  // f64 - f32 promotes to f64, then .float() (LSTEP.py:228-230)
    }
  };
  if (is_lk && first_row < n_rows) lookup(first_row, 0);
  __syncthreads();
  int buf = 0;
  for (int64_t row = first_row; row < n_rows; row += row_stride, buf ^= 1) {
    const int32_t* s_nbr = s_nbr_all + buf * K;
    const float* s_dt = s_dt_all + buf * K;
    if (is_lk) {
      if (row + row_stride < n_rows) lookup(row + row_stride, buf ^ 1);
    } else {
      if (tid < t) {
        float acc = 0.f;
        const float w = tw[tid];
        for (int k = 0; k < K; ++k)
          if (s_nbr[k] != 0) acc += time_feature(s_dt[k], w);
        S[row * ldS + d + tid] = acc;
      }
      if (tid >= t_pad && tid - t_pad < dvec) {
        if (late_wait) pdl_wait();
        const int cv = tid - t_pad;
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        int k = 0;
        for (; k + 10 <= K; k += 10) {
          float4 v[10];
#pragma unroll
          for (int u = 0; u < 10; ++u) v[u] = ld_dep(reinterpret_cast<const float4*>(pe + (int64_t)s_nbr[k + u] * d) + cv);
#pragma unroll
          for (int u = 0; u < 10; ++u) {
            acc.x += v[u].x;
            acc.y += v[u].y;
            acc.z += v[u].z;
            acc.w += v[u].w;
          }
        }
        for (; k + 4 <= K; k += 4) {
          float4 v[4];
#pragma unroll
          for (int u = 0; u < 4; ++u) v[u] = ld_dep(reinterpret_cast<const float4*>(pe + (int64_t)s_nbr[k + u] * d) + cv);
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            acc.x += v[u].x;
            acc.y += v[u].y;
            acc.z += v[u].z;
            acc.w += v[u].w;
          }
        }
        for (; k < K; ++k) {
          const float4 v = ld_dep(reinterpret_cast<const float4*>(pe + (int64_t)s_nbr[k] * d) + cv);
          acc.x += v.x;
          acc.y += v.y;
          acc.z += v.z;
          acc.w += v.w;
        }
        reinterpret_cast<float4*>(S + row * ldS)[cv] = acc;
      }
    }
    __syncthreads();  // buf is consumed and buf ^ 1 is filled: swap
  }
}

// dpe[nbr[i,k], :] += dS[i, :d]   (training only; fp32 atomics)

// phase A: one CTA per batch node. Threads [0,t): time frequencies; [t_pad, t_pad+d/4): PE columns.
constexpr int kSegPerThread = 4;

__device__ __forceinline__ void edge_aggregate_rows(int64_t first_node, int64_t node_stride, bool zero_counters, bool late_wait,
                                                    const float* __restrict__ pe,
                                                             const int64_t* __restrict__ ids, int64_t n_ids,
                                                             const int64_t* __restrict__ src,
                                                             const int64_t* __restrict__ dst,
                                                             const double* __restrict__ times, int64_t n_edges, float tc,
                                                             const float* __restrict__ tw, int d, int t, int t_pad,
                                                             float* __restrict__ A, int64_t lda,
                                                             int32_t* __restrict__ counters) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int nthr = blockDim.x;
  const int seg = nthr * kSegPerThread;
  int32_t* s_other = reinterpret_cast<int32_t*>(smem_raw);  // [seg]
  float* s_dt = reinterpret_cast<float*>(s_other + seg);    // [seg]
  int32_t* s_warp = reinterpret_cast<int32_t*>(s_dt + seg); // [32] warp totals
  __shared__ int s_total;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int dvec = d / 4;
  const bool is_tf = tid < t;
  const bool is_pe = tid >= t_pad && tid - t_pad < dvec;
  const int cv = tid - t_pad;
  if (zero_counters && tid < 8) counters[tid] = 0;  // phase-B counters, consumed by later launches

  for (int64_t n = first_node; n < n_ids; n += node_stride) {
    const int64_t node = ids[n];
    float acc_tf = 0.f;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    const float w = is_tf ? tw[tid] : 0.f;
    for (int side = 0; side < 2; ++side) {
      const int64_t* match = side == 0 ? src : dst;  // scatter #1 indexes by src (LSTEP.py:283-286), #2 by dst
      const int64_t* other = side == 0 ? dst : src;
      for (int64_t lo = 0; lo < n_edges; lo += seg) {
        // ordered compaction of the matches in [lo, lo+seg)
        const int64_t e0 = lo + (int64_t)tid * kSegPerThread;
        int64_t mv[kSegPerThread];
        int cnt = 0;
#pragma unroll
        for (int u = 0; u < kSegPerThread; ++u) {
          mv[u] = (e0 + u < n_edges) ? match[e0 + u] : -1;
          cnt += (mv[u] == node);
        }
        int incl = cnt;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const int v = __shfl_up_sync(kFull, incl, o);
          if (lane >= o) incl += v;
        }
        if (lane == 31) s_warp[wid] = incl;
        __syncthreads();
        if (wid == 0) {
          const int nw = nthr >> 5;
          int v = lane < nw ? s_warp[lane] : 0;
          int iv = v;
#pragma unroll
          for (int o = 1; o < 32; o <<= 1) {
            const int x = __shfl_up_sync(kFull, iv, o);
            if (lane >= o) iv += x;
          }
          if (lane < nw) s_warp[lane] = iv - v;  // exclusive
          if (lane == 31) s_total = iv;
        }
        __syncthreads();
        int pos = s_warp[wid] + incl - cnt;
#pragma unroll
        for (int u = 0; u < kSegPerThread; ++u) {
          if (mv[u] == node) {
            s_other[pos] = (int32_t)other[e0 + u];
            // torch.Tensor([current_time]) is fp32; fp32 - fp64 promotes to fp64; then .float() (LSTEP.py:277, Q4)
            s_dt[pos] = (float)((double)tc - times[e0 + u]);
            ++pos;
          }
        }
        __syncthreads();
        const int total = s_total;
        if (is_tf) {
          for (int j = 0; j < total; ++j) acc_tf += time_feature(s_dt[j], w);
        }
        if (is_pe) {
          if (late_wait) pdl_wait();
          int j = 0;
          for (; j + 4 <= total; j += 4) {
            float4 v[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) v[u] = ld_dep(reinterpret_cast<const float4*>(pe + (int64_t)s_other[j + u] * d) + cv);
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              acc.x += v[u].x;
              acc.y += v[u].y;
              acc.z += v[u].z;
              acc.w += v[u].w;
            }
          }
          for (; j < total; ++j) {
            const float4 v = ld_dep(reinterpret_cast<const float4*>(pe + (int64_t)s_other[j] * d) + cv);
            acc.x += v.x;
            acc.y += v.y;
            acc.z += v.z;
            acc.w += v.w;
          }
        }
        __syncthreads();
      }
    }
    if (is_tf) A[n * lda + d + tid] = acc_tf;
    if (is_pe) reinterpret_cast<float4*>(A + n * lda)[cv] = acc;
  }
}


}  // namespace lstep
