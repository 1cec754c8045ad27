// K2 (gather side) — neighbourhood PE aggregate of LSTEP.compute_neighborhood_pe
// (/root/reference/models/LSTEP.py:228-238):
//   S[i] = sum_k [ pe[nbr[i,k]] || (nbr[i,k] != 0) * cos(fp32(q_time[i] - nbr_t[i,k]) * w) ]
// One CTA per query row, two warp-aligned roles working concurrently: `t` threads own one time
// frequency each (K accurate cosines, never materialising the [K, d+t] concatenation), d/4
// threads own one 128-bit column group of the PE row and add the K gathered rows in order
// k = 0..K-1 (the PE table is L2 resident: 7.6 MB at Reddit size). Padded slots (id 0) read
// pe[0] like any other row — it is non-zero after an update (SURVEY Q2).
#include <algorithm>

#include "common.cuh"
#include "gather_bodies.cuh"

namespace lstep {

template <int VEC, bool kLookup>
__global__ void __launch_bounds__(512) nbr_aggregate_kernel(const float* __restrict__ pe, const double* __restrict__ q_time,
                                                            const int32_t* __restrict__ nbr, const float* __restrict__ nbr_t,
                                                            int64_t n_rows, int K, const float* __restrict__ tw, int d, int t, int t_pad,
                                                            float* __restrict__ S, int64_t ldS, int64_t period, LookupArgs lk) {
  pdl_launch_dependents();
  pdl_wait();
  nbr_aggregate_rows<VEC, kLookup>(blockIdx.x, gridDim.x, false, pe, q_time, nbr, nbr_t, n_rows, K, tw, d, t, t_pad, S, ldS, period, lk);
}

__global__ void __launch_bounds__(256) nbr_aggregate_bwd_kernel(const float* __restrict__ dS,
                                                                const int32_t* __restrict__ nbr, int64_t n_rows, int K,
                                                                int d, int t, float* __restrict__ dpe) {
  const int in1 = d + t;
  for (int64_t row = blockIdx.x; row < n_rows; row += gridDim.x) {
    for (int c = threadIdx.x; c < d; c += blockDim.x) {
      const float g = dS[row * in1 + c];
      for (int k = 0; k < K; ++k) atomicAdd(dpe + (int64_t)nbr[row * K + k] * d + c, g);
    }
  }
}

// f2 — the edge / time mixer of LSTEP.aggregated_node_embeddings (models/LSTEP.py:146-167). The reference builds
// [tf_k || edge_feat_k] for the K most recent neighbours, runs edge_mlp_1 (Linear) on each and then edge_agg (a Linear
// over the K axis): both are linear and nothing non-linear sits between them, so
//     edge_agg(edge_mlp_1(C))[i] = W1 (sum_k a_k C[i,k,:]) + (sum_k a_k) b1 + b_agg
// and the [n, K, 272] intermediate (K x the flops and bytes) never needs to exist. This kernel forms
//     X[i] = sum_k a_k [ (nbr_k != 0) cos(fp32(t_i - t_k) w) || edge_feat[eid_k] ]              ([n, t + Fe])
// in one pass: warp 0 does the most-recent-K lookup (with edge ids), `t` threads own a time frequency, Fe/4 threads a
// 128-bit column group of the gathered edge-feature rows. The two small Linear layers that follow run on X.
__global__ void __launch_bounds__(512) feature_aggregate_kernel(const int64_t* __restrict__ indptr, const int32_t* __restrict__ c_nbr,
                                                                const int32_t* __restrict__ c_eid, const double* __restrict__ c_t,
                                                                int64_t num_rows, const int64_t* __restrict__ q_node,
                                                                const double* __restrict__ q_time, int64_t n_rows, int64_t n_valid, int K,
                                                                const float* __restrict__ edge_feats, int64_t n_edge_rows, int Fe,
                                                                const float* __restrict__ tw, int t, int t_pad,
                                                                const float* __restrict__ agg_w, float* __restrict__ X,
                                                                uint32_t* __restrict__ err_flag) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  int32_t* s_nbr = reinterpret_cast<int32_t*>(smem_raw);
  int32_t* s_eid = s_nbr + K;
  float* s_dt = reinterpret_cast<float*>(s_eid + K);
  float* s_a = s_dt + K;
  const int tid = threadIdx.x;
  const bool v4 = (Fe % 4 == 0) && ((reinterpret_cast<uintptr_t>(edge_feats) & 15) == 0);
  const int fvec = v4 ? Fe / 4 : Fe;
  const int ldx = t + Fe;
  for (int k = tid; k < K; k += blockDim.x) s_a[k] = agg_w[k];
  for (int64_t row = blockIdx.x; row < n_rows; row += gridDim.x) {
    if (tid < 32) {
      int64_t first = 0;
      int take = 0;
      double tq = 0.0;
      if (row < n_valid) {  // rows beyond min(len(ids), len(times)) stay all-padding (zip truncation, utils.py:169)
        const int64_t node = q_node[row];
        tq = q_time[row];
        if (node < 0 || node >= num_rows) {
          if (tid == 0 && err_flag) atomicOr(err_flag, LSTEP_FLAG_NODE_OUT_OF_RANGE);
        } else {
          warp_recent_range(indptr, c_t, node, tq, K, tid, first, take);
        }
      }
      const int pad = K - take;
      for (int k = tid; k < K; k += 32) {
        int32_t n = 0, e = 0;
        float tt = 0.f;
        if (k >= pad) {
          const int64_t at = first + (k - pad);
          n = c_nbr[at];
          e = c_eid[at];
          tt = (float)c_t[at];
        }
        if (e < 0 || e >= n_edge_rows) {
          if (err_flag) atomicOr(err_flag, LSTEP_FLAG_NODE_OUT_OF_RANGE);
          e = 0;
        }
        s_nbr[k] = n;
        s_eid[k] = e;
        s_dt[k] = (float)(tq - (double)tt);  // numpy f64 - f32 -> f64, then .float() (LSTEP.py:153)
      }
    }
    __syncthreads();
    if (tid < t) {
      const float w = tw[tid];
      float acc = 0.f;
      for (int k = 0; k < K; ++k)
        if (s_nbr[k] != 0) acc = fmaf(s_a[k], time_feature(s_dt[k], w), acc);
      X[row * ldx + tid] = acc;
    }
    if (tid >= t_pad && tid - t_pad < fvec) {
      const int cv = tid - t_pad;
      if (v4) {
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int k = 0; k < K; ++k) {
          const float4 v = __ldg(reinterpret_cast<const float4*>(edge_feats + (int64_t)s_eid[k] * Fe) + cv);
          const float a = s_a[k];
          acc.x = fmaf(a, v.x, acc.x);
          acc.y = fmaf(a, v.y, acc.y);
          acc.z = fmaf(a, v.z, acc.z);
          acc.w = fmaf(a, v.w, acc.w);
        }
        float* dst = X + row * ldx + t + 4 * cv;  // (row pitch t + Fe need not be 16-byte aligned)
        dst[0] = acc.x;
        dst[1] = acc.y;
        dst[2] = acc.z;
        dst[3] = acc.w;
      } else {
        float acc = 0.f;
        for (int k = 0; k < K; ++k) acc = fmaf(s_a[k], __ldg(edge_feats + (int64_t)s_eid[k] * Fe + cv), acc);
        X[row * ldx + t + cv] = acc;
      }
    }
    __syncthreads();
  }
}

// a5 stand-alone: out[i][j] = time_feature(dt[i], w[j]) (the function every fused kernel calls)
__global__ void __launch_bounds__(256) time_features_kernel(const float* __restrict__ dt, int64_t n, const float* __restrict__ w, int t,
                                                            float* __restrict__ out) {
  const int64_t total = n * t;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x)
    out[i] = time_feature(dt[i / t], w[i % t]);
}

int launch_pe_mlp(const float* A, int64_t lda, const float* pe, RowIds base_ids, int64_t n_rows, int64_t expected_rows,
                  const int32_t* n_rows_dev, const lstep_pe_mlp* m, float* out, int64_t out_stride, float* pe_inplace,
                  cudaStream_t st, bool late_trigger = false);

static bool aligned16(const void* p) { return reinterpret_cast<uintptr_t>(p) % 16 == 0; }

template <bool kLookup>
static int launch_nbr_aggregate_t(const float* pe, const double* q_time, const int32_t* nbr, const float* nbr_t, int64_t n_rows, int K,
                                  const float* tw, int d, int t, float* S, int64_t ldS, int64_t period, LookupArgs lk, cudaStream_t st) {
  const bool v4 = d % 4 == 0 && ldS % 4 == 0 && aligned16(pe) && aligned16(S);
  const int dvec = v4 ? d / 4 : d;
  const int t_pad = (int)align_up((size_t)t, 32);
  const int threads = (int)align_up((size_t)t_pad + dvec, 32);
  if (threads > 512) return LSTEP_ERR_UNSUPPORTED;
  const size_t smem = (size_t)K * 8;
  if (smem > 48 * 1024) return LSTEP_ERR_UNSUPPORTED;
  const int64_t grid = n_rows < (int64_t)num_sms() * 16 ? n_rows : (int64_t)num_sms() * 16;
  if (v4)
    launch_k(nbr_aggregate_kernel<4, kLookup>, dim3((unsigned)grid), dim3(threads), smem, st, pe, q_time, nbr, nbr_t, n_rows, K, tw, d, t,
             t_pad, S, ldS, period, lk);
  else
    launch_k(nbr_aggregate_kernel<1, kLookup>, dim3((unsigned)grid), dim3(threads), smem, st, pe, q_time, nbr, nbr_t, n_rows, K, tw, d, t,
             t_pad, S, ldS, period, lk);
  return check_launch("nbr_aggregate");
}

int launch_nbr_aggregate(const float* pe, const double* q_time, const int32_t* nbr, const float* nbr_t,
                         int64_t n_rows, int K, const float* tw, int d, int t, float* S, int64_t ldS, int64_t period,
                         cudaStream_t st) {
  return launch_nbr_aggregate_t<false>(pe, q_time, nbr, nbr_t, n_rows, K, tw, d, t, S, ldS, period, LookupArgs{}, st);
}

// lookup + aggregate in one launch (row r: node q_node.at(r), time q_time[q_node.time_index(r)])
int launch_nbr_lookup_aggregate(const lstep_csr* csr, RowIds q_node, const float* pe, const double* q_time, int64_t n_rows, int K,
                                const float* tw, int d, int t, float* S, int64_t ldS, uint32_t* err_flag, cudaStream_t st) {
  if (!csr || K <= 0 || !q_node.p[0] || !q_time) return LSTEP_ERR_INVALID_ARG;
  LookupArgs lk{csr->indptr, csr->nbr, csr->t, csr->num_rows, q_node, err_flag};
  return launch_nbr_aggregate_t<true>(pe, q_time, nullptr, nullptr, n_rows, K, tw, d, t, S, ldS, q_node.period, lk, st);
}

}  // namespace lstep

using namespace lstep;

extern "C" int lstep_nbr_aggregate(const float* pe, int64_t pe_rows, const double* q_time, const int32_t* nbr,
                                   const float* nbr_t, int64_t n_rows, int K, const float* tw, int d, int t, float* S,
                                   void* stream) {
  if (n_rows < 0 || K <= 0 || d <= 0 || t < 0 || pe_rows <= 0) return LSTEP_ERR_INVALID_ARG;
  if (n_rows == 0) return LSTEP_OK;
  if (!pe || !q_time || !nbr || !nbr_t || !S || (t > 0 && !tw)) return LSTEP_ERR_INVALID_ARG;
  return launch_nbr_aggregate(pe, q_time, nbr, nbr_t, n_rows, K, tw, d, t, S, d + t, 0, as_stream(stream));
}

extern "C" int lstep_nbr_aggregate_bwd(const float* dS, const int32_t* nbr, int64_t n_rows, int K, int d, int t,
                                       float* dpe, int64_t pe_rows, void* stream) {
  if (n_rows < 0 || K <= 0 || d <= 0 || pe_rows <= 0) return LSTEP_ERR_INVALID_ARG;
  if (n_rows == 0) return LSTEP_OK;
  if (!dS || !nbr || !dpe) return LSTEP_ERR_INVALID_ARG;
  const int64_t grid = n_rows < (int64_t)num_sms() * 8 ? n_rows : (int64_t)num_sms() * 8;
  nbr_aggregate_bwd_kernel<<<(unsigned)grid, 256, 0, as_stream(stream)>>>(dS, nbr, n_rows, K, d, t, dpe);
  return check_launch("nbr_aggregate_bwd");
}

extern "C" int lstep_neighborhood_pe(const float* pe, int64_t pe_rows, const int64_t* q_node, const double* q_time,
                                     const int32_t* nbr, const float* nbr_t, int64_t n_rows, int K,
                                     const lstep_pe_mlp* mlp, float* out, void* workspace, size_t workspace_bytes,
                                     void* stream) {
  if (n_rows < 0 || K <= 0 || !mlp || pe_rows <= 0) return LSTEP_ERR_INVALID_ARG;
  if (n_rows == 0) return LSTEP_OK;
  if (!pe || !q_node || !q_time || !nbr || !nbr_t || !out || !workspace) return LSTEP_ERR_INVALID_ARG;
  const int64_t ldS = (int64_t)align_up((size_t)(mlp->d + mlp->t), 4);  // 16-byte aligned rows
  const size_t need = (size_t)n_rows * ldS * sizeof(float);
  if (workspace_bytes < need) return LSTEP_ERR_WORKSPACE;
  float* S = reinterpret_cast<float*>(workspace);
  int rc = launch_nbr_aggregate(pe, q_time, nbr, nbr_t, n_rows, K, mlp->tw, mlp->d, mlp->t, S, ldS, 0, as_stream(stream));
  if (rc != LSTEP_OK) return rc;
  return launch_pe_mlp(S, ldS, pe, single_ids(q_node), n_rows, n_rows, nullptr, mlp, out, mlp->d, nullptr, as_stream(stream));
}

extern "C" int lstep_nbr_lookup_aggregate(const lstep_csr* csr, const int64_t* q_node, const double* q_time, int64_t n_rows, int K,
                                          const float* pe, int64_t pe_rows, const float* tw, int d, int t, float* S,
                                          uint32_t* err_flag, void* stream) {
  if (n_rows < 0 || K <= 0 || d <= 0 || t < 0 || pe_rows <= 0) return LSTEP_ERR_INVALID_ARG;
  if (n_rows == 0) return LSTEP_OK;
  if (!csr || !pe || !q_node || !q_time || !S || (t > 0 && !tw)) return LSTEP_ERR_INVALID_ARG;
  return launch_nbr_lookup_aggregate(csr, single_ids(q_node), pe, q_time, n_rows, K, tw, d, t, S, d + t, err_flag, as_stream(stream));
}

extern "C" int lstep_time_features(const float* dt, int64_t n, const float* w, int t, float* out, void* stream) {
  if (n < 0 || t <= 0 || (n > 0 && (!dt || !w || !out))) return LSTEP_ERR_INVALID_ARG;
  if (n == 0) return LSTEP_OK;
  const int64_t blocks = std::min<int64_t>(ceil_div(n * t, 256), (int64_t)num_sms() * 8);
  time_features_kernel<<<(unsigned)blocks, 256, 0, as_stream(stream)>>>(dt, n, w, t, out);
  return check_launch("time_features");
}

extern "C" int lstep_feature_aggregate(const lstep_csr* csr, const int64_t* q_node, const double* q_time, int64_t n_rows, int64_t n_valid,
                                       int K, const float* edge_feats, int64_t n_edge_rows, int Fe, const float* tw, int t,
                                       const float* agg_w, float* X, uint32_t* err_flag, void* stream) {
  if (n_rows < 0 || n_valid < 0 || n_valid > n_rows || K <= 0 || Fe <= 0 || t < 0 || n_edge_rows <= 0) return LSTEP_ERR_INVALID_ARG;
  if (n_rows == 0) return LSTEP_OK;
  if (!csr || !csr->eid || !q_node || !q_time || !edge_feats || !agg_w || !X || (t > 0 && !tw)) return LSTEP_ERR_INVALID_ARG;
  const bool v4 = Fe % 4 == 0 && aligned16(edge_feats);
  const int t_pad = (int)align_up((size_t)t, 32);
  const int threads = (int)align_up((size_t)t_pad + (v4 ? Fe / 4 : Fe), 32);
  const size_t smem = (size_t)K * 16;
  if (threads > 512 || smem > 48 * 1024) return LSTEP_ERR_UNSUPPORTED;
  const int64_t grid = std::min<int64_t>(n_rows, (int64_t)num_sms() * 16);
  feature_aggregate_kernel<<<(unsigned)grid, threads, smem, as_stream(stream)>>>(csr->indptr, csr->nbr, csr->eid, csr->t, csr->num_rows, q_node,
                                                                                 q_time, n_rows, n_valid, K, edge_feats, n_edge_rows, Fe, tw, t,
                                                                                 t_pad, agg_w, X, err_flag);
  return check_launch("feature_aggregate");
}
