// PE MLP:  out = base + tanh( [Ws base + bs] + W2 relu(W1 A + b1) + b2 )
// The arithmetic of models/LSTEP.py:240-247 (neighbourhood), :294-301 (update phase A, with the
// self term) and :329-336 (update phase B, where the self term is computed and discarded — Q3).
//
// launch_pe_mlp() dispatches to the cluster split-K kernel (csrc/mlp_cluster.cu, the default). This file holds the
// weight packing and the ALL-COLUMNS ring kernel it replaced, kept as the fallback for shapes the cluster kernel does
// not cover:
//
// fp32 FMA throughout: the parity bar (1e-5) rules out single-pass TF32/BF16 tensor-core math.
//   * weights are pre-packed (lstep_pack_linear) as [in_pad][ldo] row-major, in_pad = in rounded up
//     to 16, ldo = out rounded up to 32, zero filled — so a k-tile of 16 input rows is one contiguous
//     16*ldo*4-byte block (12 KB at d=172);
//   * one CTA owns R = 2*RT rows and all output columns. The three GEMM segments (W1 over the
//     aggregate, W2 over the hidden row, Ws over the base row) are walked as one flat sequence of
//     k-tiles that a single elected thread streams into a shared-memory ring with cp.async.bulk
//     (completion on an mbarrier);
//   * activations sit in shared memory k-major ([k][R]) so one 128-bit broadcast load feeds RT rows;
//     thread (rg, cp) keeps an RT x 2 register tile.
#include <cstdlib>

#include "common.cuh"
#include "mlp_job.cuh"

namespace lstep {

constexpr int kKTile = 16;

__global__ void pack_linear_kernel(const float* __restrict__ w, const float* __restrict__ b, int out_f, int in_f,
                                   int in_pad, int ldo, float* __restrict__ pw, float* __restrict__ pb) {
  const int64_t total = (int64_t)in_pad * ldo;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int k = (int)(i / ldo), c = (int)(i % ldo);
    pw[i] = (c < out_f && k < in_f) ? w[(size_t)c * in_f + k] : 0.f;
  }
  if (blockIdx.x == 0)
    for (int c = threadIdx.x; c < ldo; c += blockDim.x) pb[c] = (b && c < out_f) ? b[c] : 0.f;
}

__global__ void stream_order_fence_kernel() {}

// ---- mbarrier / bulk-copy primitives (PTX) ---------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t done = 0;
  uint32_t spins = 0;
  while (!done) {
    if (++spins > (1u << 24)) __trap();  // a lost bulk copy must fault, not hang the device
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
  }
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void consumer_sync(int nthreads) {  // named barrier 1: consumer warps only
  asm volatile("bar.sync 1, %0;" ::"r"(nthreads) : "memory");
}

// dynamic smem: [NS][kKTile][ldo] weight ring | As[in1_pad][R] | Hs[d_pad][R] | Bs[d_pad][R] | red[G][R][ldo]
//
// Warp-specialised: blockDim = G*ldo consumer threads + one producer warp.
//   producer  one lane streams the flat weight-tile sequence into the NS = 2G stage ring with
//             cp.async.bulk (full[s] mbarrier, expect_tx), waiting on empty[s] before reusing a stage;
//   consumers G k-split groups of ldo threads; group g takes every G-th tile of a segment into its
//             own partial accumulators and releases the stage (one arrive per warp on empty[s]); the
//             groups only meet at the end of a segment, where the partials are summed through smem.
template <int RT, int G>
__global__ void __launch_bounds__(G == 4 ? 800 : 288) pe_mlp_kernel(const float* __restrict__ A, int64_t lda, const float* pe,
                                                              RowIds base_ids, int64_t n_rows,
                                                              const int32_t* __restrict__ n_rows_dev, lstep_pe_mlp m,
                                                              int ldo, float* __restrict__ out, int64_t out_stride,
                                                              float* pe_inplace) {
  constexpr int R = 2 * RT;
  constexpr int NS = (RT >= 8 ? 2 : 3) * G;  // as many weight tiles in flight as shared memory allows
  extern __shared__ __align__(128) float smem[];
  __shared__ __align__(8) uint64_t full_bar[NS];
  __shared__ __align__(8) uint64_t empty_bar[NS];
  const int d = m.d, in1 = m.d + m.t;
  const int in1_pad = (in1 + kKTile - 1) / kKTile * kKTile;
  const int d_pad = (d + kKTile - 1) / kKTile * kKTile;
  if (n_rows_dev) {
    const int64_t nd = *n_rows_dev;
    n_rows = nd < n_rows ? nd : n_rows;
  }
  const int64_t n_row_tiles = (n_rows + R - 1) / R;
  if ((int64_t)blockIdx.x >= n_row_tiles) return;
  const int tile_elems = kKTile * ldo;
  float* Wst = smem;
  float* As = Wst + (size_t)NS * tile_elems;
  float* Hs = As + (size_t)in1_pad * R;   // Hs and Bs are adjacent: the second segment runs over [h ; base]
  float* Bs = Hs + (size_t)d_pad * R;
  float* red = Bs + (size_t)d_pad * R;    // [G][R][ldo]
  const int tid = threadIdx.x;
  const int ncons = G * ldo;
  const bool has_self = m.ws != nullptr;
  const int t1 = in1_pad / kKTile, t2 = d_pad / kKTile;
  const int ntiles = t1 + t2 + (has_self ? t2 : 0);
  const uint32_t tile_bytes = (uint32_t)tile_elems * 4u;
  // persistent: this CTA walks row tiles blockIdx.x, blockIdx.x + gridDim.x, ...; the weight-tile ring keeps
  // running across row tiles (global tile counter `it`), so the next row tile's first weights are already in
  // flight while the current epilogue runs.
  const int64_t my_tiles = (n_row_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x;

  if (tid == 0) {
    for (int s = 0; s < NS; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], (uint32_t)(ldo >> 5));  // one arrive per consumer warp of the owning group
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();

  if (tid >= ncons) {  // ---- producer warp
    if (tid == ncons) {
      int64_t it = 0;
      for (int64_t rt = 0; rt < my_tiles; ++rt) {
        for (int i = 0; i < ntiles; ++i, ++it) {
          const int s = (int)(it % NS);
          if (it >= NS) mbar_wait(&empty_bar[s], (uint32_t)(((it / NS) - 1) & 1));
          const float* src = i < t1 ? m.w1 + (size_t)i * tile_elems
                                    : (i < t1 + t2 ? m.w2 + (size_t)(i - t1) * tile_elems : m.ws + (size_t)(i - t1 - t2) * tile_elems);
          mbar_expect_tx(&full_bar[s], tile_bytes);
          bulk_g2s(Wst + (size_t)s * tile_elems, src, tile_bytes, &full_bar[s]);
        }
      }
    }
    return;
  }

  const int g = tid / ldo, lt = tid % ldo;  // k-split group, thread within group
  const int npairs = ldo >> 1;
  const int rg = lt / npairs, cp = lt % npairs;
  const int c0 = 2 * cp;
  const int lane = tid & 31;
  float acc[RT][2];
  auto fma_tile = [&](const float* wt, const float* in) {
    // wt: [kKTile][ldo] weight tile; in: [kKTile][R] activations (k-major)
#pragma unroll
    for (int k = 0; k < kKTile; ++k) {
      const float2 w = *reinterpret_cast<const float2*>(wt + k * ldo + c0);
      const float* ap = in + k * R + rg * RT;
      float av[RT];
      if (RT >= 4) {
#pragma unroll
        for (int q = 0; q < RT / 4; ++q) {
          const float4 v = *reinterpret_cast<const float4*>(ap + 4 * q);
          av[4 * q + 0] = v.x;
          av[4 * q + 1] = v.y;
          av[4 * q + 2] = v.z;
          av[4 * q + 3] = v.w;
        }
      } else {
        const float2 v = *reinterpret_cast<const float2*>(ap);
        av[0] = v.x;
        av[RT - 1] = v.y;
      }
#pragma unroll
      for (int r = 0; r < RT; ++r) {
        acc[r][0] = fmaf(av[r], w.x, acc[r][0]);
        acc[r][1] = fmaf(av[r], w.y, acc[r][1]);
      }
    }
  };
  // one segment: weight tiles [first, first+count) of the current row tile (global ring index it0 + i)
  auto run_segment = [&](int64_t it0, int first, int count, const float* in) {
#pragma unroll
    for (int r = 0; r < RT; ++r) acc[r][0] = acc[r][1] = 0.f;
    for (int j = g; j < count; j += G) {
      const int64_t it = it0 + first + j;
      const int s = (int)(it % NS);
      mbar_wait(&full_bar[s], (uint32_t)((it / NS) & 1));
      fma_tile(Wst + (size_t)s * tile_elems, in + (size_t)j * kKTile * R);
      __syncwarp();
      if (lane == 0) mbar_arrive(&empty_bar[s]);  // this warp is done with the stage
    }
    float* rp = red + ((size_t)g * R + rg * RT) * ldo + c0;
#pragma unroll
    for (int r = 0; r < RT; ++r) *reinterpret_cast<float2*>(rp + (size_t)r * ldo) = make_float2(acc[r][0], acc[r][1]);
    consumer_sync(ncons);
  };
  auto reduced = [&](int r, int j) {  // sum of the G partials of element (row rg*RT + r, column c0 + j), fixed order
    float v = 0.f;
#pragma unroll
    for (int gg = 0; gg < G; ++gg) v += red[((size_t)gg * R + rg * RT + r) * ldo + c0 + j];
    return v;
  };

  for (int64_t rt = 0; rt < my_tiles; ++rt) {
    const int64_t row0 = ((int64_t)blockIdx.x + rt * gridDim.x) * R;
    const int64_t it0 = rt * ntiles;
    // ---- stage the activation tiles k-major (loads batched ahead of the stores)
    {
      const int totalA = R * in1_pad, totalB = R * d_pad;
      for (int base = 0; base < totalA; base += ncons * 4) {
        float v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int idx = base + u * ncons + tid;
          const int r = idx / in1_pad, k = idx % in1_pad;
          v[u] = (idx < totalA && row0 + r < n_rows && k < in1) ? A[(row0 + r) * lda + k] : 0.f;
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int idx = base + u * ncons + tid;
          if (idx < totalA) As[(idx % in1_pad) * R + idx / in1_pad] = v[u];
        }
      }
      for (int base = 0; base < totalB; base += ncons * 4) {
        float v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int idx = base + u * ncons + tid;
          const int r = idx / d_pad, k = idx % d_pad;
          v[u] = (idx < totalB && row0 + r < n_rows && k < d) ? pe[base_ids.at(row0 + r) * (int64_t)d + k] : 0.f;
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int idx = base + u * ncons + tid;
          if (idx < totalB) Bs[(idx % d_pad) * R + idx / d_pad] = v[u];
        }
      }
    }
    consumer_sync(ncons);

    // ---- layer 1: h = relu(W1 a + b1), written k-major; padded columns stay zero
    run_segment(it0, 0, t1, As);
    if (g == 0) {
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        const int c = c0 + j;
        if (c < d_pad) {
          const float b = c < d ? m.b1[c] : 0.f;
#pragma unroll
          for (int r = 0; r < RT; ++r) Hs[c * R + rg * RT + r] = c < d ? fmaxf(reduced(r, j) + b, 0.f) : 0.f;
        }
      }
    }
    consumer_sync(ncons);

    // ---- layer 2 (+ self term): z = W2 h + b2 [+ Ws base + bs] as one k-run over [h ; base]
    run_segment(it0, t1, ntiles - t1, Hs);
    if (g == 0) {
#pragma unroll
      for (int r = 0; r < RT; ++r) {
        const int rr = rg * RT + r;
        const int64_t row = row0 + rr;
        if (row >= n_rows) continue;
        float* dst = out ? out + row * out_stride : pe_inplace + base_ids.at(row) * (int64_t)d;
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          const int c = c0 + j;
          if (c < d) {
            const float z = reduced(r, j) + m.b2[c] + (has_self ? m.bs[c] : 0.f);
            dst[c] = Bs[c * R + rr] + tanhf(z);
          }
        }
      }
    }
    consumer_sync(ncons);  // red / As / Bs are reused by the next row tile
  }
}

template <int RT, int G>
static int launch_mlp_r(const float* A, int64_t lda, const float* pe, RowIds base_ids, int64_t n_rows,
                        const int32_t* n_rows_dev, const lstep_pe_mlp* m, float* out, int64_t out_stride,
                        float* pe_inplace, cudaStream_t st) {
  constexpr int R = 2 * RT;
  const int ldo = lstep_packed_ld(m->d);
  const int in1_pad = lstep_packed_rows(m->d + m->t), d_pad = lstep_packed_rows(m->d);
  const size_t smem = sizeof(float) * ((size_t)(RT >= 8 ? 2 : 3) * G * kKTile * ldo + (size_t)R * (in1_pad + 2 * (size_t)d_pad) + (size_t)G * R * ldo);
  if (smem > 220 * 1024 || G * ldo + 32 > 1024) return LSTEP_ERR_UNSUPPORTED;
  auto kern = pe_mlp_kernel<RT, G>;
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024);
    if (e != cudaSuccess) {
      set_cuda_error(e, "pe_mlp attr");
      return LSTEP_ERR_CUDA;
    }
    attr_set = true;
  }
  int64_t blocks = ceil_div(n_rows, R);
  if (blocks > num_sms()) blocks = num_sms();  // persistent: one CTA per SM walks the row tiles
  kern<<<(unsigned)blocks, G * ldo + 32, smem, st>>>(A, lda, pe, base_ids, n_rows, n_rows_dev, *m, ldo, out, out_stride, pe_inplace);
  return check_launch("pe_mlp");
}



// n_rows is the host-side upper bound of rows; *n_rows_dev (optional) the device-side count.
int launch_pe_mlp(const float* A, int64_t lda, const float* pe, RowIds base_ids, int64_t n_rows, int64_t expected_rows,
                  const int32_t* n_rows_dev, const lstep_pe_mlp* m, float* out, int64_t out_stride, float* pe_inplace,
                  cudaStream_t st, bool late_trigger) {
  if (n_rows <= 0) return LSTEP_OK;
  if (!A || !pe || !base_ids.p[0] || !m || (!out && !pe_inplace)) return LSTEP_ERR_INVALID_ARG;
  // the cluster split-K kernel (csrc/mlp_cluster.cu); the all-columns weight-ring kernel below serves the shapes it does not cover
  const int rc = launch_pe_mlp_cluster(A, lda, pe, base_ids, n_rows, expected_rows, n_rows_dev, m, out, out_stride, pe_inplace, nullptr, nullptr, st, late_trigger);
  if (rc != LSTEP_ERR_UNSUPPORTED) return rc;
  const int ldo = lstep_packed_ld(m->d);
  // rows per CTA: the largest tile that still gives about one CTA per SM; k-split while the CTA stays <= 1024 threads
  if (ldo <= 192) {  // 4 k-split groups of <= 192 threads + the producer warp = 800 threads
    if (expected_rows >= (int64_t)num_sms() * 24) return launch_mlp_r<8, 4>(A, lda, pe, base_ids, n_rows, n_rows_dev, m, out, out_stride, pe_inplace, st);
    if (expected_rows >= (int64_t)num_sms() * 5) return launch_mlp_r<4, 4>(A, lda, pe, base_ids, n_rows, n_rows_dev, m, out, out_stride, pe_inplace, st);
    return launch_mlp_r<2, 4>(A, lda, pe, base_ids, n_rows, n_rows_dev, m, out, out_stride, pe_inplace, st);
  }
  return launch_mlp_r<4, 1>(A, lda, pe, base_ids, n_rows, n_rows_dev, m, out, out_stride, pe_inplace, st);
}

}  // namespace lstep

using namespace lstep;

extern "C" int lstep_packed_ld(int out_features) { return (int)align_up((size_t)out_features, 32); }
extern "C" int lstep_packed_rows(int in_features) { return (int)align_up((size_t)in_features, kKTile); }

extern "C" int lstep_pack_linear(const float* weight, const float* bias, int out_features, int in_features,
                                 float* packed_w, float* packed_b, void* stream) {
  if (!weight || !packed_w || !packed_b || out_features <= 0 || in_features <= 0) return LSTEP_ERR_INVALID_ARG;
  const int ldo = lstep_packed_ld(out_features);
  pack_linear_kernel<<<64, 256, 0, as_stream(stream)>>>(weight, bias, out_features, in_features,
                                                        lstep_packed_rows(in_features), ldo, packed_w, packed_b);
  // The MLP kernels fetch the packed parameters BEFORE their programmatic-dependency wait (they are constants
  // of the step). A plainly launched empty kernel behind the pack kernel is a full stream-order barrier: whatever
  // is launched after it, early start or not, begins after the packed weights are complete and visible.
  stream_order_fence_kernel<<<1, 32, 0, as_stream(stream)>>>();
  return check_launch("pack_linear");
}

extern "C" int lstep_pe_mlp_apply(const float* A, const float* pe, const int64_t* base_ids, int64_t n_rows,
                                  const lstep_pe_mlp* mlp, float* out, int64_t out_stride, float* pe_inplace,
                                  void* stream) {
  if (n_rows < 0) return LSTEP_ERR_INVALID_ARG;
  if (!mlp) return LSTEP_ERR_INVALID_ARG;
  return launch_pe_mlp(A, mlp->d + mlp->t, pe, single_ids(base_ids), n_rows, n_rows, nullptr, mlp, out, out_stride, pe_inplace,
                       as_stream(stream), false);
}
