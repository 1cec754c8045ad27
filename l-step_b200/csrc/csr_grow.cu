// Growable CSR: the a1 adjacency with room at the end of every row, so that edges can be appended batch by batch
// instead of rebuilding the whole CSR (csr_build.cu: a radix sort of all 2E entries) for every batch.
//
// Layout: the ordinary lstep_csr plus int32 fill[num_rows]. Row v holds its real entries at
// [indptr[v], indptr[v] + fill[v]); the rest of [indptr[v], indptr[v+1]) is padding (t = +inf, nbr = 0, eid = 0).
// Every reader (warp_recent_range, sample_recent_kernel, phaseB_push_kernel, feature_aggregate_kernel) counts the entries
// of the row with t < tq (strict, fp64) and reads only entries before that count, and none reads csr->nnz: padding is
// never selected and the row stays sorted, so every existing entry point reads a growable CSR unchanged and returns
// what it returns on an exact CSR of the same edges.
//
// Appending keeps the reference's order (utils/utils.py:292-299, 99: adj[src] gets (dst, eid, t), then adj[dst] gets
// (src, eid, t), in data order; each row is then sorted stably by t): with globally non-decreasing times, appending in
// (edge, side) order IS that stable sort, across batch boundaries and ties included.
#include <math_constants.h>

#include "common.cuh"

namespace lstep {

constexpr int kIngestChunkEdges = 2048;  // edges per chunk (<= 4096 entries = 32 KB of sort keys); chunks go in order
constexpr int kIngestPosBits = 12;       // bits of an entry's position in its chunk: log2(2 * kIngestChunkEdges)

// one warp per row: the row's real entries move to their new place, the rest of the new row becomes padding. Rows
// [src_rows, new_rows) are new (no entries: all padding); rows [new_rows, fill_rows) are allocated but not live: fill 0.
__global__ void __launch_bounds__(256) csr_relayout_kernel(const int64_t* __restrict__ indptr, const int32_t* __restrict__ nbr,
                                                           const int32_t* __restrict__ eid, const double* __restrict__ t,
                                                           const int32_t* __restrict__ fill, int64_t src_rows, int64_t new_rows,
                                                           int64_t fill_rows, const int64_t* __restrict__ new_indptr,
                                                           int32_t* __restrict__ out_nbr, int32_t* __restrict__ out_eid,
                                                           double* __restrict__ out_t, int32_t* __restrict__ out_fill,
                                                           uint32_t* err_flag) {
  const int64_t v = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (v >= fill_rows) return;
  if (v >= new_rows) {
    if (lane == 0) out_fill[v] = 0;
    return;
  }
  const int64_t lo = v < src_rows ? indptr[v] : 0;
  const int64_t f = v >= src_rows ? 0 : fill ? (int64_t)fill[v] : indptr[v + 1] - lo;
  const int64_t nlo = new_indptr[v], cap = new_indptr[v + 1] - nlo;
  const int64_t n = f < cap ? f : cap;
  for (int64_t k = lane; k < cap; k += 32) {
    if (k < n) {
      out_nbr[nlo + k] = nbr[lo + k];
      out_eid[nlo + k] = eid[lo + k];
      out_t[nlo + k] = t[lo + k];
    } else {
      out_nbr[nlo + k] = 0;
      out_eid[nlo + k] = 0;
      out_t[nlo + k] = CUDART_INF;
    }
  }
  if (lane == 0) {
    out_fill[v] = (int32_t)n;
    if (n < f && err_flag) atomicOr(err_flag, LSTEP_FLAG_CSR_FULL);
  }
}

// padding for the tail [new_indptr[new_rows], total) of a relaid CSR, which lstep_csr_add_rows hands out to new rows
__global__ void __launch_bounds__(256) csr_pad_tail_kernel(const int64_t* __restrict__ new_indptr, int64_t new_rows, int64_t total,
                                                           int32_t* __restrict__ out_nbr, int32_t* __restrict__ out_eid,
                                                           double* __restrict__ out_t) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t k = new_indptr[new_rows] + blockIdx.x * (int64_t)blockDim.x + threadIdx.x; k < total; k += stride) {
    out_nbr[k] = 0;
    out_eid[k] = 0;
    out_t[k] = CUDART_INF;
  }
}

// rows [r0, r0 + n) become live: indptr[r0 + 1 + i] = indptr[r0] + cap[0] + ... + cap[i], fill = 0. One CTA, a block scan
// per chunk of 1024 rows; the entries the rows take were padded when the tail was laid out, so nothing else is written.
__global__ void __launch_bounds__(1024) csr_add_rows_kernel(int64_t* indptr, int32_t* fill, int64_t r0, int64_t n,
                                                            const int64_t* __restrict__ cap) {
  __shared__ int64_t s_sum[1024];
  __shared__ int64_t s_base;
  const int tid = threadIdx.x;
  if (tid == 0) s_base = indptr[r0];
  __syncthreads();
  for (int64_t c0 = 0; c0 < n; c0 += 1024) {
    const int64_t i = c0 + tid;
    s_sum[tid] = i < n ? cap[i] : 0;
    __syncthreads();
    for (int o = 1; o < 1024; o <<= 1) {  // Hillis-Steele inclusive scan
      const int64_t x = tid >= o ? s_sum[tid - o] : 0;
      __syncthreads();
      s_sum[tid] += x;
      __syncthreads();
    }
    if (i < n) {
      indptr[r0 + 1 + i] = s_base + s_sum[tid];
      fill[r0 + i] = 0;
    }
    __syncthreads();
    if (tid == 1023) s_base += s_sum[1023];
    __syncthreads();
  }
}

// first index in s[0, m) whose key is >= x (s sorted ascending)
__device__ __forceinline__ int lower_bound_smem(const unsigned long long* s, int m, unsigned long long x) {
  int a = 0, b = m;
  while (a < b) {
    const int mid = (a + b) >> 1;
    if (s[mid] < x)
      a = mid + 1;
    else
      b = mid;
  }
  return a;
}

// One CTA appends the 2n entries of a batch, chunk by chunk in edge order. Each chunk's entries are keyed
// (row << 12 | position in the chunk), the position being 2 * edge + side, and sorted in shared memory (bitonic, over the
// next power of two >= 2 * edges in the chunk): an entry's rank among the chunk's earlier entries of its row is then its
// distance from the start of its row's segment, found by a binary search. It goes to indptr[row] + fill[row] + rank;
// after a barrier, the last entry of each segment advances fill[row]. Deterministic: no atomics decide a position.
// The CTA and its shared memory are sized to the batch (csr_ingest_launch), so that it fits on an SM beside the kernels
// of a step it overlaps.
__global__ void __launch_bounds__(1024) csr_ingest_kernel(const int64_t* __restrict__ indptr, int32_t* c_nbr, int32_t* c_eid,
                                                          double* c_t, int64_t num_rows, int32_t* fill,
                                                          const int64_t* __restrict__ src, const int64_t* __restrict__ dst,
                                                          const int64_t* __restrict__ eid, int64_t eid_base,
                                                          const double* __restrict__ t, int64_t n_edges, uint32_t* err_flag) {
  extern __shared__ unsigned long long s_key[];  // [next power of two >= 2 * edges of the largest chunk]
  constexpr unsigned long long kNone = ~0ull;
  constexpr unsigned kPosMask = (1u << kIngestPosBits) - 1;
  const int tid = threadIdx.x, nt = blockDim.x;
  for (int64_t c0 = 0; c0 < n_edges; c0 += kIngestChunkEdges) {
    const int ne = (int)(n_edges - c0 < kIngestChunkEdges ? n_edges - c0 : kIngestChunkEdges);
    const int m = 2 * ne;
    int m2 = 2;
    while (m2 < m) m2 <<= 1;
    for (int p = tid; p < m2; p += nt) {
      unsigned long long key = kNone;
      if (p < m) {
        const int64_t i = c0 + (p >> 1);
        const int64_t s = src[i], d = dst[i];
        const int64_t id = eid ? eid[i] : eid_base + i;
        if (s < 0 || s >= num_rows || d < 0 || d >= num_rows || id < 0 || id > 0x7fffffffLL) {
          // the whole edge is dropped (the reference raises IndexError at utils.py:298)
          if ((p & 1) == 0 && err_flag) atomicOr(err_flag, LSTEP_FLAG_NODE_OUT_OF_RANGE);
        } else {
          key = ((unsigned long long)((p & 1) ? d : s) << kIngestPosBits) | (unsigned long long)p;
        }
      }
      s_key[p] = key;
    }
    __syncthreads();
    for (int k = 2; k <= m2; k <<= 1) {
      for (int j = k >> 1; j > 0; j >>= 1) {
        for (int p = tid; p < m2; p += nt) {
          const int q = p ^ j;
          if (q > p) {
            const unsigned long long a = s_key[p], b = s_key[q];
            if (((p & k) == 0) == (a > b)) {
              s_key[p] = b;
              s_key[q] = a;
            }
          }
        }
        __syncthreads();
      }
    }
    for (int j = tid; j < m; j += nt) {
      const unsigned long long key = s_key[j];
      if (key == kNone) continue;
      const int64_t row = (int64_t)(key >> kIngestPosBits);
      const int p = (int)(key & kPosMask);
      const int seg0 = lower_bound_smem(s_key, m, (unsigned long long)row << kIngestPosBits);
      const int seg1 = lower_bound_smem(s_key, m, (unsigned long long)(row + 1) << kIngestPosBits);
      const int rank = j - seg0, cnt = seg1 - seg0;
      const int64_t lo = indptr[row], cap = indptr[row + 1] - lo;
      const int32_t f = fill[row];
      if ((int64_t)f + cnt > cap) {  // no room: nothing of this chunk goes to the row
        if (rank == 0 && err_flag) atomicOr(err_flag, LSTEP_FLAG_CSR_FULL);
        continue;
      }
      const int64_t i = c0 + (p >> 1);
      const double te = t[i];
      double prev = -CUDART_INF;
      if (rank > 0)
        prev = t[c0 + (int64_t)((s_key[j - 1] & kPosMask) >> 1)];
      else if (f > 0)
        prev = c_t[lo + f - 1];
      if (te < prev && err_flag) atomicOr(err_flag, LSTEP_FLAG_UNSORTED_STREAM);
      const int64_t at = lo + f + rank;
      c_nbr[at] = (int32_t)((p & 1) ? src[i] : dst[i]);
      c_eid[at] = (int32_t)(eid ? eid[i] : eid_base + i);
      c_t[at] = te;
    }
    __syncthreads();  // every entry of the chunk has read fill[] before any of it moves
    // the last entry of each row segment advances the row's fill (only that thread reads or writes it from here on)
    for (int j = tid; j < m; j += nt) {
      const unsigned long long key = s_key[j];
      if (key == kNone) continue;
      const int64_t row = (int64_t)(key >> kIngestPosBits);
      if (j + 1 < m && (s_key[j + 1] >> kIngestPosBits) == (unsigned long long)row) continue;
      const int cnt = j + 1 - lower_bound_smem(s_key, m, (unsigned long long)row << kIngestPosBits);
      const int32_t f = fill[row];
      if ((int64_t)f + cnt <= indptr[row + 1] - indptr[row]) fill[row] = f + cnt;
    }
    __syncthreads();  // the next chunk reads the new fill[] and s_key is rewritten
  }
}

// the CTA and its shared memory sized to the largest chunk (the first): 2n entries -> next power of two, half as many
// threads (one compare-exchange each per bitonic pass), 64 .. 1024
static int csr_ingest_launch(const lstep_csr* csr, int32_t* fill, const int64_t* src, const int64_t* dst, const int64_t* eid,
                             int64_t eid_base, const double* t, int64_t n_edges, uint32_t* err_flag, cudaStream_t st) {
  const int m = 2 * (int)(n_edges < kIngestChunkEdges ? n_edges : kIngestChunkEdges);
  int m2 = 2;
  while (m2 < m) m2 <<= 1;
  const int threads = m2 / 2 < 64 ? 64 : (m2 / 2 > 1024 ? 1024 : m2 / 2);
  // the CSR is caller-owned device memory; lstep_csr carries const pointers because every other entry point only reads it
  csr_ingest_kernel<<<1, threads, sizeof(unsigned long long) * (size_t)m2, st>>>(
      csr->indptr, const_cast<int32_t*>(csr->nbr), const_cast<int32_t*>(csr->eid), const_cast<double*>(csr->t), csr->num_rows, fill,
      src, dst, eid, eid_base, t, n_edges, err_flag);
  return check_launch("csr_ingest");
}

}  // namespace lstep

using namespace lstep;

extern "C" int lstep_csr_relayout(const lstep_csr* src, const int32_t* src_fill, const int64_t* new_indptr, int32_t* out_nbr,
                                  int32_t* out_eid, double* out_t, int32_t* out_fill, uint32_t* err_flag, void* stream) {
  if (!src || src->num_rows <= 0) return LSTEP_ERR_INVALID_ARG;
  return lstep_csr_relayout_rows(src, src_fill, src->num_rows, src->num_rows, new_indptr, -1, out_nbr, out_eid, out_t, out_fill, err_flag,
                                 stream);
}

extern "C" int lstep_csr_relayout_rows(const lstep_csr* src, const int32_t* src_fill, int64_t new_rows, int64_t row_cap,
                                       const int64_t* new_indptr, int64_t total, int32_t* out_nbr, int32_t* out_eid, double* out_t,
                                       int32_t* out_fill, uint32_t* err_flag, void* stream) {
  if (!src || !src->indptr || !new_indptr || !out_fill || src->num_rows <= 0) return LSTEP_ERR_INVALID_ARG;
  if (new_rows < src->num_rows || row_cap < new_rows) return LSTEP_ERR_INVALID_ARG;
  if (row_cap > 0x7fffffffLL) return LSTEP_ERR_ID_RANGE;
  if (!out_nbr || !out_eid || !out_t) return LSTEP_ERR_INVALID_ARG;
  cudaStream_t st = as_stream(stream);
  csr_relayout_kernel<<<(unsigned)ceil_div(row_cap * 32, 256), 256, 0, st>>>(src->indptr, src->nbr, src->eid, src->t, src_fill, src->num_rows,
                                                                             new_rows, row_cap, new_indptr, out_nbr, out_eid, out_t, out_fill,
                                                                             err_flag);
  int rc = check_launch("csr_relayout");
  if (rc != LSTEP_OK || total < 0) return rc;
  csr_pad_tail_kernel<<<num_sms() * 4, 256, 0, st>>>(new_indptr, new_rows, total, out_nbr, out_eid, out_t);
  return check_launch("csr_pad_tail");
}

extern "C" int lstep_csr_add_rows(lstep_csr* csr, int32_t* fill, int64_t n_rows, const int64_t* cap, void* stream) {
  if (!csr || !csr->indptr || !fill || n_rows < 0 || (n_rows > 0 && !cap)) return LSTEP_ERR_INVALID_ARG;
  if (csr->num_rows <= 0 || csr->num_rows + n_rows > 0x7fffffffLL) return LSTEP_ERR_ID_RANGE;
  if (n_rows == 0) return LSTEP_OK;
  // the CSR is caller-owned device memory; lstep_csr carries const pointers because the lookups only read it
  csr_add_rows_kernel<<<1, 1024, 0, as_stream(stream)>>>(const_cast<int64_t*>(csr->indptr), fill, csr->num_rows, n_rows, cap);
  const int rc = check_launch("csr_add_rows");
  if (rc == LSTEP_OK) csr->num_rows += n_rows;
  return rc;
}

extern "C" int lstep_csr_ingest(const lstep_csr* csr, int32_t* fill, const int64_t* src, const int64_t* dst, const int64_t* eid,
                                int64_t eid_base, const double* t, int64_t n_edges, uint32_t* err_flag, void* stream) {
  if (!csr || !csr->indptr || !fill || n_edges < 0) return LSTEP_ERR_INVALID_ARG;
  if (n_edges == 0) return LSTEP_OK;
  if (!src || !dst || !t || !csr->nbr || !csr->eid || !csr->t) return LSTEP_ERR_INVALID_ARG;
  if (csr->num_rows <= 0 || csr->num_rows > 0x7fffffffLL) return LSTEP_ERR_ID_RANGE;
  if (!eid && (eid_base < 0 || eid_base + n_edges - 1 > 0x7fffffffLL)) return LSTEP_ERR_ID_RANGE;
  return csr_ingest_launch(csr, fill, src, dst, eid, eid_base, t, n_edges, err_flag, as_stream(stream));
}
