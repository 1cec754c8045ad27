// update_pe phase B, push form (LSTEP.update_pe, /root/reference/models/LSTEP.py:305-341) — ONE kernel for
//   nbr, _, nt = sampler(ids, times, K)                       (:306-308, zip truncation Q1/Q1b)
//   agg2[nbr[i,k]] += [ pe[ids[i]] || cos((tc - nt[i,k]) * w) ]   (:314-322, padded slots: time features zeroed,
//                                                                  destination 0 collects pe[ids[i]] only)
// followed by the MLP over the distinct destinations (csrc/mlp_cluster.cu reads the accumulators directly).
//
// The pull form in csrc/update.cu builds an inverse index (count -> scan -> fill) and then reduces every
// destination's slot list in the reference's order: four launches and a single-CTA scan, 40 us of a 110 us
// step for ~1 MB of useful traffic. Here every contribution is ADDED WHERE IT LANDS:
//   * up to four small CTAs per batch node i (push_split_for), each owning a share of the K slots (the SM-side issue rate of
//     64-bit reductions, ~1.3 cycles per lane, is what bounds the kernel: many small CTAs spread it evenly over
//     the 148 SMs); warp 0 of each does the most-recent-K lookup (same 32-ary search as csrc/sampler.cu);
//   * each distinct destination u is given a compact accumulator row on first touch: atomicCAS on a per-node
//     claim map (0 = free, -1 = being set up, j+1 = row j); the winner zeroes the row, fences, and publishes
//     j+1; later arrivals (in any CTA) spin until the row is published — the winner never waits on anyone;
//   * contributions are accumulated in 32.32 fixed point with 64-bit integer atomics (RED at L2): integer
//     addition is associative, so the result is EXACT and independent of arrival order — bit-reproducible
//     run to run, and one rounding (at the final conversion) instead of one per addition of the
//     reference's sequential fp32 sum. The padding destination 0 receives z_i * pe[ids[i]] (z_i = number of
//     padded slots of row i) as one contribution per row.
//     Exact only while every column sum fits in int64: the kernel raises LSTEP_FLAG_FIXED_POINT_RANGE when a batch row's
//     value is non-finite or reaches fixed_point_bound(n_ids, K) (csrc/common.cuh), or a time feature is non-finite.
// The claim map is returned to all-zero by the MLP kernel once a row has been consumed; U (row -> node id)
// and the row count (counters[2]) are what the MLP launch reads. Accumulator rows need no invariant: a row
// is zeroed by whoever claims it.
#include "common.cuh"

namespace lstep {

constexpr float kFixScale = 4294967296.f;  // 2^32
constexpr int kPushThreads = 128;          // upper bound (launch bounds); small batches use 64-thread CTAs
// CTAs per batch node: each repeats the node's lookup, so the split only pays while the launch has too few CTAs to fill
// the GPU. Reddit shape (B = 200, ~310 batch nodes): 4 CTAs of 64 threads per node = 1 240 CTAs. B = 2000 (~3 800 batch
// nodes): at 4 per node the launch is 15 208 CTAs = 3.2 waves of a 32-CTA-per-SM GPU, each wave a full lookup + claim latency
// chain (73.6 us, profiles/r02_ncu_scaleout_kernels.txt); one 128-thread CTA per node is a single wave.
inline int push_split_for(int64_t n_ids) { return n_ids <= 1184 ? 4 : (n_ids <= 2368 ? 2 : 1); }

template <int DQ, int TQ>
__global__ void __launch_bounds__(kPushThreads) phaseB_push_kernel(const int64_t* __restrict__ indptr, const int32_t* __restrict__ c_nbr,
                                                          const double* __restrict__ c_t, int64_t num_rows,
                                                          const int64_t* __restrict__ ids, const double* __restrict__ q_time,
                                                          int64_t n_ids, int64_t n_valid, int K, float* pe, int d, int t,
                                                          const float* __restrict__ tw, float tc, int32_t* claim_of,
                                                          int64_t* __restrict__ U, int32_t* counters,
                                                          unsigned long long* acc, int32_t* dirty, int stamp, const float* new_rows, uint32_t* err_flag,
                                                          unsigned long long* row0_part, int own_mul, int own_add, int kPushSplit,
                                                          int use_parts, float fx_bound) {
  // own_mul > 1 (peer group, csrc/peer.cu): this rank accumulates only the destinations u with u % own_mul == own_add and
  // applies only the phase-A rows of the batch nodes it owns; the lookup of every batch node is replicated.
  // Dependency structure (programmatic dependent launch): the kernel in front is the phase-A MLP, launched with
  // a LATE trigger, so this kernel is resident only after everything before that MLP has completed. The lookup
  // and the claim phase touch nothing the phase-A MLP reads or writes (CSR, ids, claim map, counters, U, the
  // accumulator rows), so they run BEFORE the wait, next to the MLP; the wait sits in front of the first access
  // to the table (pe[0] = 0 and the phase-A rows).
  TL_ENTRY(3);
  pdl_launch_dependents();
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int Kcap = (K + kPushSplit - 1) / kPushSplit;
  int32_t* s_nbr = reinterpret_cast<int32_t*>(smem_raw);     // [Kcap] this CTA's slots
  float* s_dt = reinterpret_cast<float*>(s_nbr + Kcap);      // [Kcap]  tc - nt (fp32 - fp32, LSTEP.py:314)
  int32_t* s_slot = reinterpret_cast<int32_t*>(s_dt + Kcap); // [Kcap]  accumulator row of the slot's destination, -1 = padding
  __shared__ int s_z, s_j0;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  const int in1 = d + t;
  const int64_t row = blockIdx.x / kPushSplit;
  const int part = blockIdx.x % kPushSplit;
  const int Kp = (K + kPushSplit - 1) / kPushSplit;
  const int k_lo = min(K, part * Kp), k_hi = min(K, k_lo + Kp);  // this CTA's slots
  // the CTA that finishes last folds the partial sums of the padding row into its accumulator row (counters[5] counts
  // finished CTAs; zeroed with the other counters by the step's edge-aggregate launch)
  auto finish = [&]() {
    __shared__ int s_last;
    if (!use_parts) return;  // (small batches add to the padding row's accumulator directly: the contention is small there)
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_last = atomicAdd(counters + 5, 1) == (int)gridDim.x - 1;
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    const int c0 = atomicAdd(claim_of + 0, 0);
    for (int c = threadIdx.x; c < d; c += blockDim.x) {
      long long sum = 0;
#pragma unroll
      for (int p0 = 0; p0 < kPushRow0Parts; p0 += 8) {  // eight loads in flight
        long long v[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) v[u] = (long long)__ldcg(row0_part + (p0 + u) * kPushRow0Cols + c);
#pragma unroll
        for (int u = 0; u < 8; ++u) sum += v[u];
      }
#pragma unroll
      for (int p = 0; p < kPushRow0Parts; ++p) row0_part[p * kPushRow0Cols + c] = 0ull;
      if (sum != 0 && c0 > 0) atomicAdd(acc + (size_t)(c0 - 1) * in1 + c, (unsigned long long)sum);
    }
  };
  if (k_lo >= k_hi) {
    finish();
    return;
  }

  if (warp == 0) {
    // ---- lookup: strictly-earlier count by warp-cooperative 32-ary search, last min(K, c) entries right-aligned
    int64_t end = 0, cnt = 0;
    if (row < n_valid) {
      const int64_t node = ids[row];
      if (node < 0 || node >= num_rows) {
        if (lane == 0 && err_flag) atomicOr(err_flag, LSTEP_FLAG_NODE_OUT_OF_RANGE);
      } else {
        const int64_t lo = indptr[node];
        int64_t a = lo, b = indptr[node + 1];
        const double tq = q_time[row];
        while (b - a > 32) {
          const int64_t len = b - a;
          const int64_t p = a + (len * (lane + 1)) / 33;
          const int jj = __popc(__ballot_sync(kFull, c_t[p] < tq));
          const int64_t pa = a + (len * jj) / 33, pb = a + (len * (jj + 1)) / 33;
          if (jj < 32) b = pb;
          if (jj > 0) a = pa + 1;
        }
        const int64_t p = a + lane;
        const bool less = (p < b) && (c_t[p] < tq);
        end = a + __popc(__ballot_sync(kFull, less));
        cnt = end - lo;
      }
    }
    const int take = (int)(cnt < K ? cnt : K);
    const int pad = K - take;
    const int64_t first = end - take;
    // ---- claim an accumulator row per distinct destination
    int z = 0;
    for (int k0 = k_lo; k0 < k_hi; k0 += 32) {
      const int k = k0 + lane;
      int32_t u = 0;
      float dt = 0.f;
      if (k < k_hi && k >= pad) {
        const int64_t e = first + (k - pad);
        u = c_nbr[e];
        dt = tc - (float)c_t[e];  // neighbour times are returned as fp32 (utils.py:166,208), then fp32 - fp32
      }
      const bool active = k < k_hi && u > 0 && (own_mul == 1 || u % own_mul == own_add);
      z += __popc(__ballot_sync(kFull, k < k_hi && u <= 0));
      const unsigned grp = __match_any_sync(kFull, active ? u : -(lane + 1));
      const int leader = __ffs(grp) - 1;
      int j = -1;
      bool won = false;
      if (active && lane == leader) {
        const int old = atomicCAS(claim_of + u, 0, -1);
        if (old == 0) {
          j = atomicAdd(counters + 2, 1);
          U[j] = (int64_t)u;
          dirty[u] = stamp;  // this table row changes in phase B of step `stamp` (read by the step's ring append)
          won = true;
        } else if (old > 0) {
          j = old - 1;
        }
      }
      // winners' rows are zeroed by the whole warp before they are published
      unsigned wm = __ballot_sync(kFull, won);
      while (wm) {
        const int src = __ffs(wm) - 1;
        wm &= wm - 1;
        const int jj = __shfl_sync(kFull, j, src);
        ulonglong2* zr = reinterpret_cast<ulonglong2*>(acc + (size_t)jj * in1);  // in1 even: 16-byte rows
        for (int c = lane; c < in1 / 2; c += 32) zr[c] = make_ulonglong2(0ull, 0ull);
      }
      __threadfence();
      __syncwarp();
      if (won) atomicExch(claim_of + u, j + 1);
      if (active && lane == leader && j < 0) {  // someone else is setting the row up: wait for its number
        int v;
        unsigned spins = 0;
        do {
          v = atomicAdd(claim_of + u, 0);
          if (++spins > (1u << 26)) __trap();
        } while (v <= 0);
        j = v - 1;
      }
      j = __shfl_sync(kFull, j, leader);
      if (k < k_hi) {
        s_nbr[k - k_lo] = u;
        s_dt[k - k_lo] = dt;
        s_slot[k - k_lo] = active ? j : -1;
      }
    }
    // ---- the padding destination: node 0 collects z * pe[ids[row]] (on the rank that owns node 0)
    int j0 = -1;
    if (own_add != 0) z = 0;
    if (z > 0) {
      bool won = false;
      if (lane == 0) {
        const int old = atomicCAS(claim_of + 0, 0, -1);
        if (old == 0) {
          j0 = atomicAdd(counters + 2, 1);
          U[j0] = 0;
          dirty[0] = stamp;
          won = true;
        } else if (old > 0) {
          j0 = old - 1;
        }
      }
      won = __shfl_sync(kFull, (int)won, 0) != 0;
      if (won) {
        const int jj = __shfl_sync(kFull, j0, 0);
        ulonglong2* zr = reinterpret_cast<ulonglong2*>(acc + (size_t)jj * in1);
        for (int c = lane; c < in1 / 2; c += 32) zr[c] = make_ulonglong2(0ull, 0ull);
        __threadfence();
        __syncwarp();
        if (lane == 0) atomicExch(claim_of + 0, j0 + 1);
      } else if (lane == 0 && j0 < 0) {
        int v;
        unsigned spins = 0;
        do {
          v = atomicAdd(claim_of + 0, 0);
          if (++spins > (1u << 26)) __trap();
        } while (v <= 0);
        j0 = v - 1;
      }
    }
    if (lane == 0) {
      s_z = z;
      s_j0 = j0;
    }
  }
  __syncthreads();
  // ---- time features of this CTA's slots: they depend on the lookup only, so they are accumulated BEFORE the
  // wait as well (the accumulator rows are private to this kernel)
  float w[TQ];
#pragma unroll
  for (int q = 0; q < TQ; ++q) w[q] = (lane + 32 * q < t) ? tw[lane + 32 * q] : 0.f;
  bool bad = false;  // a contribution outside the fixed-point range (fixed_point_bound, csrc/common.cuh); a cosine fails only when non-finite
  for (int k = warp; k < k_hi - k_lo; k += nwarps) {
    const int j = s_slot[k];
    if (j < 0) continue;
    unsigned long long* rowp = acc + (size_t)j * in1 + d;
    const float dt = s_dt[k];
#pragma unroll
    for (int q = 0; q < TQ; ++q) {
      const int jf = lane + 32 * q;
      if (jf < t) {
        const float f = time_feature(dt, w[q]);
        bad |= !(fabsf(f) <= 1.f);
        atomicAdd(rowp + jf, (unsigned long long)__float2ll_rn(f * kFixScale));
      }
    }
  }

  pdl_wait();  // phase A has written the table
  TL_WAITED(3);
  if (blockIdx.x == 0 && own_add == 0)  // (peer group: the owner of row 0 only — its final row reaches the other replicas from there)
    for (int c = threadIdx.x; c < d; c += blockDim.x) pe[c] = 0.f;  // pe[0] = 0 (LSTEP.py:317); no batch row reads row 0 below

  // ---- this row's PE in fixed point (phase-A table), once per warp. new_rows != NULL (streaming step): phase A
  // wrote its result rows to a side buffer (its MLP ran in the same launch as the neighbourhood MLP, which still
  // read the old table); this kernel both uses them and applies them to the table (one CTA per row).
  const int64_t node = ids[row];
  const float* src_row = new_rows ? new_rows + row * (int64_t)d : pe + node * (int64_t)d;
  long long fx[DQ];
#pragma unroll
  for (int q = 0; q < DQ; ++q) {
    const int c = lane + 32 * q;
    const float x = (c < d && node > 0) ? ld_dep(src_row + c) : 0.f;
    bad |= !(fabsf(x) < fx_bound);
    fx[q] = __float2ll_rn(x * kFixScale);
  }
  // (every slot of a batch row adds the row somewhere: to its destination or, padded, to row 0 — on the rank that owns it)
  if (__any_sync(kFull, bad) && lane == 0 && err_flag) atomicOr(err_flag, LSTEP_FLAG_FIXED_POINT_RANGE);
  if (new_rows && part == 0 && node > 0 && (own_mul == 1 || node % own_mul == own_add))  // row 0 is zeroed above (LSTEP.py:317 follows the phase-A write)
    for (int c = threadIdx.x; c < d; c += blockDim.x) pe[node * (int64_t)d + c] = ld_dep(src_row + c);
  for (int k = warp; k < k_hi - k_lo; k += nwarps) {
    const int j = s_slot[k];
    if (j < 0) continue;
    unsigned long long* rowp = acc + (size_t)j * in1;
#pragma unroll
    for (int q = 0; q < DQ; ++q) {
      const int c = lane + 32 * q;
      if (c < d) atomicAdd(rowp + c, (unsigned long long)fx[q]);
    }
  }
  if (s_z > 0 && warp == nwarps - 1) {
    unsigned long long* rowp = use_parts ? row0_part + (size_t)(row % kPushRow0Parts) * kPushRow0Cols : acc + (size_t)s_j0 * in1;
    const unsigned long long zz = (unsigned long long)s_z;
#pragma unroll
    for (int q = 0; q < DQ; ++q) {
      const int c = lane + 32 * q;
      if (c < d) atomicAdd(rowp + c, zz * (unsigned long long)fx[q]);  // (two's complement: the signed product's bits; no overflow in range)
    }
  }
  finish();
  TL_EXIT(3);
}

// enqueue the push kernel; on return (stream order) acc rows [0, counters[2]) hold the aggregates of the
// destinations U[0 .. counters[2])
int launch_phaseB_push(const lstep_csr* csr, const int64_t* ids, const double* q_time, int64_t n_ids, int64_t n_valid, int K,
                       float* pe, int d, int t, const float* tw, float tc, int32_t* claim_of, int64_t* U, int32_t* counters,
                       unsigned long long* acc, int32_t* dirty, int stamp, const float* new_rows, uint32_t* err_flag, cudaStream_t st,
                       unsigned long long* row0_part, int own_mul, int own_add) {
  if (own_mul < 1 || own_add < 0 || own_add >= own_mul || !row0_part || d > kPushRow0Cols) return LSTEP_ERR_INVALID_ARG;
  if (!csr || !ids || !q_time || !dirty || n_ids <= 0 || K <= 0 || (d + t) % 2 != 0) return LSTEP_ERR_INVALID_ARG;
  const int split = push_split_for(n_ids);
  // (peer group of >= 4 ranks: a CTA accumulates only the ~K / world slots this rank owns — two warps are enough, and twice as many
  // CTAs are resident for the replicated lookups; ONE warp per CTA was measured slower: push 42 -> 51 us at N=4, 37 -> 43 us at N=8)
  const int threads = (split == 4 || own_mul >= 4) ? 64 : kPushThreads;
  const size_t smem = (size_t)((K + split - 1) / split) * 12;
  const int use_parts = split < 4 ? 1 : 0;  // padding-row partial sums + fold: only where thousands of CTAs would hit one row
  const float bound = fixed_point_bound(n_ids, K);
  if (d <= 6 * 32 && t <= 4 * 32)
    launch_k(phaseB_push_kernel<6, 4>, dim3((unsigned)(n_ids * split)), dim3(threads), smem, st, csr->indptr, csr->nbr, csr->t, csr->num_rows, ids,
             q_time, n_ids, n_valid, K, pe, d, t, tw, tc, claim_of, U, counters, acc, dirty, stamp, new_rows, err_flag, row0_part, own_mul, own_add, split, use_parts, bound);
  else if (d <= 8 * 32 && t <= 8 * 32)
    launch_k(phaseB_push_kernel<8, 8>, dim3((unsigned)(n_ids * split)), dim3(threads), smem, st, csr->indptr, csr->nbr, csr->t, csr->num_rows, ids,
             q_time, n_ids, n_valid, K, pe, d, t, tw, tc, claim_of, U, counters, acc, dirty, stamp, new_rows, err_flag, row0_part, own_mul, own_add, split, use_parts, bound);
  else
    return LSTEP_ERR_UNSUPPORTED;
  return check_launch("phaseB_push");
}

}  // namespace lstep

LSTEP_TIMELINE_DEFINE(push)
