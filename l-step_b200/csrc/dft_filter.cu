// K3 — learnable DFT filter over each node's PE history.
// Replaces LSTEP.fourier_transform_pe (/root/reference/models/LSTEP.py:104-137).
//
// The reference computes, per batch node n and PE column c,
//   X = FFT_t(x[n,:,c]);  X *= m;  X *= W[:,c];  X *= m;  y = iFFT(X);  y *= m;
//   out[n,c] = sum_t a[t] * Re(y[t])
// with x zero-padded to T steps and m[j] = 1 for j < b (b = batch_idx when the history is
// shorter than T, else no mask). Every step is linear in x, so
//   out[n,c] = sum_s G[s,c] * x[n,s,c],
//   G[s,c]   = (1/T) * sum_{f<b} Re( W[f,c] * A[f] * exp(-2*pi*i*f*s/T) ),
//   A[f]     = sum_{t<b} a[t] * exp(+2*pi*i*f*t/T).
// lstep_dft_collapse builds G in fp64 (phase reduced as an integer mod T, so the twiddles are
// exact to fp64 rounding); lstep_dft_filter is then a pure streaming reduction: 2 flop per 4
// bytes of history, bound by HBM bandwidth. It reads each node's history once with 128-bit
// loads that bypass L1, keeps G in L1/L2 (68.8 KB at T=100, d=172), and reduces the per-thread
// partial sums over time through shared memory in a fixed order (deterministic).
#include <cstdlib>

#include "common.cuh"

namespace lstep {

// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) dft_collapse_kernel(const float2* __restrict__ W, const float* __restrict__ a,
                                                           int T, int d, int b, float* __restrict__ G) {
  extern __shared__ double sm[];
  double* tw_c = sm;           // [T] cos(2*pi*m/T)
  double* tw_s = sm + T;       // [T] sin(2*pi*m/T)
  double* A_re = sm + 2 * T;   // [T]
  double* A_im = sm + 3 * T;   // [T]
  for (int m = threadIdx.x; m < T; m += blockDim.x) {
    double s, c;
    sincospi(2.0 * (double)m / (double)T, &s, &c);
    tw_c[m] = c;
    tw_s[m] = s;
  }
  __syncthreads();
  for (int f = threadIdx.x; f < T; f += blockDim.x) {
    double re = 0.0, im = 0.0;
    if (f < b) {
      for (int t = 0; t < b; ++t) {
        const int m = (int)(((long long)f * t) % T);
        const double at = (double)a[t];
        re += at * tw_c[m];
        im += at * tw_s[m];
      }
    }
    A_re[f] = re;
    A_im[f] = im;
  }
  __syncthreads();
  const double invT = 1.0 / (double)T;
  for (int s = blockIdx.x; s < T; s += gridDim.x) {
    for (int c = threadIdx.x; c < d; c += blockDim.x) {
      double acc = 0.0;
      for (int f = 0; f < b; ++f) {
        const float2 w = W[(size_t)f * d + c];
        const double br = (double)w.x * A_re[f] - (double)w.y * A_im[f];
        const double bi = (double)w.x * A_im[f] + (double)w.y * A_re[f];
        const int m = (int)(((long long)f * s) % T);
        acc += br * tw_c[m] + bi * tw_s[m];  // Re( B * exp(-i*theta) )
      }
      G[(size_t)s * d + c] = (float)(acc * invT);
    }
  }
}

// ---------------------------------------------------------------------------------------------
template <int VEC>
struct VecT;
template <>
struct VecT<4> {
  using type = float4;
};
template <>
struct VecT<1> {
  using type = float;
};

__device__ __forceinline__ void fma_acc(float4& acc, const float4& g, const float4& x) {
  acc.x = fmaf(g.x, x.x, acc.x);
  acc.y = fmaf(g.y, x.y, acc.y);
  acc.z = fmaf(g.z, x.z, acc.z);
  acc.w = fmaf(g.w, x.w, acc.w);
}
__device__ __forceinline__ void fma_acc(float& acc, const float& g, const float& x) { acc = fmaf(g, x, acc); }
__device__ __forceinline__ void add_acc(float4& a, const float4& b) {
  a.x += b.x;
  a.y += b.y;
  a.z += b.z;
  a.w += b.w;
}
__device__ __forceinline__ void add_acc(float& a, const float& b) { a += b; }
__device__ __forceinline__ float4 ld_stream(const float4* p) { return ld_stream_f4(p); }
__device__ __forceinline__ float ld_stream(const float* p) { return ld_stream_f(p); }
template <typename V>
__device__ __forceinline__ V vzero();
template <>
__device__ __forceinline__ float4 vzero<float4>() {
  return make_float4(0.f, 0.f, 0.f, 0.f);
}
template <>
__device__ __forceinline__ float vzero<float>() {
  return 0.f;
}

constexpr int kDftThreads = 256;

// threads = groups x dvec; thread (g, cv) owns vector column cv and history steps s = g, g+groups, ...
template <int VEC>
__global__ void __launch_bounds__(kDftThreads) dft_filter_kernel(const float* __restrict__ hist, int64_t node_stride,
                                                                 int64_t time_stride, int s0, int ring, int Th, int d,
                                                                 const int64_t* __restrict__ ids, int64_t n_ids,
                                                                 const float* __restrict__ G, float* __restrict__ out,
                                                                 int64_t out_stride, const int64_t* __restrict__ out_ids) {
  pdl_wait();
  pdl_launch_dependents();  // late trigger (see dft_filter_bulk_kernel)
  using V = typename VecT<VEC>::type;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  V* red = reinterpret_cast<V*>(smem_raw);  // [groups][dvec]
  const int dvec = d / VEC;
  const int groups = kDftThreads / dvec;
  const int g = threadIdx.x / dvec, cv = threadIdx.x % dvec;
  const bool active = g < groups;
  const V* Gv = reinterpret_cast<const V*>(G);
  for (int64_t n = blockIdx.x; n < n_ids; n += gridDim.x) {
    const float* base = hist + ids[n] * node_stride;
    V acc = vzero<V>();
    if (active) {
      int s = g;
      // 4 independent loads in flight per thread
      for (; s + 3 * groups < Th; s += 4 * groups) {
        V x[4], w[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int ss = s + u * groups;
          int ps = s0 + ss;
          if (ps >= ring) ps -= ring;
          x[u] = ld_stream(reinterpret_cast<const V*>(base + (int64_t)ps * time_stride) + cv);
          w[u] = __ldg(Gv + (size_t)ss * dvec + cv);
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) fma_acc(acc, w[u], x[u]);
      }
      for (; s < Th; s += groups) {
        int ps = s0 + s;
        if (ps >= ring) ps -= ring;
        const V x = ld_stream(reinterpret_cast<const V*>(base + (int64_t)ps * time_stride) + cv);
        const V w = __ldg(Gv + (size_t)s * dvec + cv);
        fma_acc(acc, w, x);
      }
      red[g * dvec + cv] = acc;
    }
    __syncthreads();
    if (active && g == 0) {
      V tot = red[cv];
      for (int gg = 1; gg < groups; ++gg) add_acc(tot, red[gg * dvec + cv]);
      reinterpret_cast<V*>(out + (out_ids ? out_ids[n] : n) * out_stride)[cv] = tot;
    }
    __syncthreads();
  }
}


// ---- node-major history (time_stride == d: the streaming ring, or a contiguous [V1,Th,d] tensor) ----------
// A node's Th steps are one contiguous block (68.8 KB at T=100, d=172) apart from the ring wrap. One CTA per
// node pulls the whole block into shared memory with a handful of cp.async.bulk copies (SASS UBLKCP), issued
// up front, in LOGICAL time order (the wrap is resolved by the copy addresses), one mbarrier per chunk of
// rows, and multiplies chunk c by G while chunks c+1.. are still in flight. With 3 CTAs resident per SM every
// byte of the launch is requested within the first microsecond, so the kernel runs at the HBM rate instead of
// paying one load latency per register-sized batch (the generic kernel above: 4 loads in flight per thread).
constexpr int kDftChunks = 4;

__device__ __forceinline__ uint32_t dft_s_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// prefetch (streaming step): the kernel in front is the previous step's ring append, and everything before THAT has
// completed by the time this kernel is resident (late triggers, see csrc/common.cuh), so the only rows of the ring
// still being written are those of the NEWEST slot. The first kDftChunks-1 chunks then cover the Th-1 older rows and
// are requested BEFORE the dependency wait — 99 % of the kernel's HBM traffic overlaps the tail of the previous
// step — and the last chunk is the newest row alone, requested after the wait.
__global__ void __launch_bounds__(kDftThreads, 5) dft_filter_bulk_kernel(const float* __restrict__ hist, int64_t node_stride, int s0,
                                                                      int ring, int Th, int d, const int64_t* __restrict__ ids,
                                                                      int64_t n_ids, const float* __restrict__ G,
                                                                      float* __restrict__ out, int64_t out_stride,
                                                                      const int64_t* __restrict__ out_ids, int prefetch) {
  extern __shared__ __align__(16) unsigned char smem_raw[];  // (bulk-copy destinations need 16-byte alignment)
  __shared__ __align__(8) uint64_t bar[kDftChunks];
  float4* xs = reinterpret_cast<float4*>(smem_raw);  // [Th][dvec] logical time order
  const int dvec = d >> 2;
  float4* red = xs + (size_t)Th * dvec;               // [groups][dvec]
  const int groups = kDftThreads / dvec;
  const int g = threadIdx.x / dvec, cv = threadIdx.x % dvec;
  const bool active = g < groups;
  // chunks 0 .. kDftChunks-2: the Th-1 older rows; last chunk: the newest row alone (the same partition with and
  // without prefetch, so both forms add in the same order and agree bit for bit)
  TL_ENTRY(0);
  const int rc = (Th - 1 + kDftChunks - 2) / (kDftChunks - 1);  // rows per chunk
  auto bounds = [&](int c, int& a, int& b) {
    if (c == kDftChunks - 1) {
      a = Th - 1;
      b = Th;
    } else {
      a = c * rc;
      b = min(Th - 1, a + rc);
    }
  };
  auto request = [&](const float* base, int c) {  // one elected thread: bulk copies of chunk c, logical order in smem
    int a, b;
    bounds(c, a, b);
    if (a >= b) return;
    const uint32_t bytes = (uint32_t)(b - a) * (uint32_t)d * 4u;
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(dft_s_u32(&bar[c])), "r"(bytes) : "memory");
    int ps = s0 + a;
    if (ps >= ring) ps -= ring;
    const int first = min(b - a, ring - ps);  // rows before the ring wraps
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     dft_s_u32(xs + (size_t)a * dvec)),
                 "l"(base + (int64_t)ps * d), "r"((uint32_t)first * (uint32_t)d * 4u), "r"(dft_s_u32(&bar[c]))
                 : "memory");
    if (first < b - a)
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                       dft_s_u32(xs + (size_t)(a + first) * dvec)),
                   "l"(base), "r"((uint32_t)(b - a - first) * (uint32_t)d * 4u), "r"(dft_s_u32(&bar[c]))
                   : "memory");
  };
  if (threadIdx.x == 0) {
    for (int c = 0; c < kDftChunks; ++c)
      asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(dft_s_u32(&bar[c])), "r"(1));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    if (prefetch && (int64_t)blockIdx.x < n_ids) {  // ids: the batch's node list, not written by any kernel of the chain
      const float* base = hist + ids[blockIdx.x] * node_stride;
      for (int c = 0; c < kDftChunks - 1; ++c) request(base, c);
    }
  }
  __syncthreads();
  pdl_wait();
  TL_WAITED(0);
  // late trigger: the next kernel of the step (the fused gather) does its lookups and cosines before its own wait;
  // it may only become resident once everything before this filter has completed
  pdl_launch_dependents();
  const float4* Gv = reinterpret_cast<const float4*>(G);
  uint32_t it = 0;
  // Streaming across the nodes of a CTA (launches with more nodes than resident CTAs: B = 2000): chunk c of the NEXT node
  // is requested as soon as every thread has finished with chunk c of the current one, so a CTA always has up to kDftChunks
  // copies in flight instead of draining its buffer between nodes (Flights shape, 2 500 nodes: 62.2 -> 58.9 us, 0.44 ->
  // 0.47 of the measured copy peak; with 30 MB outstanding the pattern itself — random 17 KB reads — tops out near 3 TB/s).
  for (int64_t n = blockIdx.x; n < n_ids; n += gridDim.x, ++it) {
    const int64_t n_next = n + gridDim.x;
    if (threadIdx.x == 0 && it == 0) {
      const float* base = hist + ids[n] * node_stride;
      for (int c = prefetch ? kDftChunks - 1 : 0; c < kDftChunks; ++c) request(base, c);
    }
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int c = 0; c < kDftChunks; ++c) {
      int a, b;
      bounds(c, a, b);
      if (a >= b) continue;
      // this thread's rows of the chunk: a + g, a + g + groups, ...; fetch their filter rows before waiting
      constexpr int kMaxRows = 5;  // (25-row chunks over 5 time groups; 48 registers: the step's next kernel shares the SM)
      float4 w[kMaxRows];
      if (active) {
#pragma unroll
        for (int u = 0; u < kMaxRows; ++u) {
          const int s = a + g + u * groups;
          if (s < b) w[u] = __ldg(Gv + (size_t)s * dvec + cv);
        }
      }
      {  // wait for the chunk (parity flips once per node this CTA handles)
        uint32_t done = 0, spins = 0;
        while (!done) {
          if (++spins > (1u << 24)) __trap();
          asm volatile(
              "{\n\t.reg .pred p;\n\t"
              "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
              "selp.u32 %0, 1, 0, p;\n\t}"
              : "=r"(done)
              : "r"(dft_s_u32(&bar[c])), "r"(it & 1u)
              : "memory");
        }
      }
      if (active) {
#pragma unroll
        for (int u = 0; u < kMaxRows; ++u) {
          const int s = a + g + u * groups;
          if (s < b) fma_acc(acc, w[u], xs[(size_t)s * dvec + cv]);
        }
        for (int s = a + g + kMaxRows * groups; s < b; s += groups) fma_acc(acc, __ldg(Gv + (size_t)s * dvec + cv), xs[(size_t)s * dvec + cv]);
      }
      if (n_next < n_ids) {  // (uniform over the CTA) the chunk's buffer is free once every thread has read it: refill it
        __syncthreads();
        if (threadIdx.x == 0) request(hist + ids[n_next] * node_stride, c);
      }
    }
    if (active) red[g * dvec + cv] = acc;
    __syncthreads();
    if (active && g == 0) {
      float4 tot = red[cv];
      for (int gg = 1; gg < groups; ++gg) add_acc(tot, red[gg * dvec + cv]);
      reinterpret_cast<float4*>(out + (out_ids ? out_ids[n] : n) * out_stride)[cv] = tot;
    }
    __syncthreads();  // xs / red are reused by the next node of this CTA
  }
  TL_EXIT(0);
}

// dG[s,c] += sum_{n in slice} x[n,s,c] * dout[n,c]; grid = (time groups, node slices)
template <int VEC>
__global__ void __launch_bounds__(kDftThreads) dft_filter_bwd_kernel(const float* __restrict__ hist,
                                                                     int64_t node_stride, int64_t time_stride, int s0,
                                                                     int ring, int Th, int d,
                                                                     const int64_t* __restrict__ ids, int64_t n_ids,
                                                                     const float* __restrict__ dout,
                                                                     float* __restrict__ dG) {
  using V = typename VecT<VEC>::type;
  const int dvec = d / VEC;
  const int groups = kDftThreads / dvec;
  const int g = threadIdx.x / dvec, cv = threadIdx.x % dvec;
  if (g >= groups) return;
  const int s = blockIdx.x * groups + g;
  if (s >= Th) return;
  int ps = s0 + s;
  if (ps >= ring) ps -= ring;
  V acc = vzero<V>();
  for (int64_t n = blockIdx.y; n < n_ids; n += gridDim.y) {
    const V x = ld_stream(reinterpret_cast<const V*>(hist + ids[n] * node_stride + (int64_t)ps * time_stride) + cv);
    const V go = __ldg(reinterpret_cast<const V*>(dout + n * (int64_t)d) + cv);
    fma_acc(acc, go, x);
  }
  float* dst = dG + (size_t)s * d + (size_t)cv * VEC;
  const float* a = reinterpret_cast<const float*>(&acc);
#pragma unroll
  for (int i = 0; i < VEC; ++i) atomicAdd(dst + i, a[i]);
}

static bool vec4_ok(const void* p, int64_t a, int64_t b, int d) {
  return (reinterpret_cast<uintptr_t>(p) % 16 == 0) && a % 4 == 0 && b % 4 == 0 && d % 4 == 0;
}

}  // namespace lstep

using namespace lstep;

extern "C" int lstep_dft_collapse(const float* W_c64, const float* a, int T, int d, int b, float* G, void* stream) {
  if (!W_c64 || !a || !G || T <= 0 || d <= 0) return LSTEP_ERR_INVALID_ARG;
  if (b < 0) b = 0;
  if (b > T) b = T;
  const size_t smem = sizeof(double) * 4 * (size_t)T;
  if (smem > 48 * 1024) return LSTEP_ERR_UNSUPPORTED;
  dft_collapse_kernel<<<T < num_sms() ? T : num_sms(), 256, smem, as_stream(stream)>>>(
      reinterpret_cast<const float2*>(W_c64), a, T, d, b, G);
  return check_launch("dft_collapse");
}

namespace lstep {
int launch_dft_filter(const float* hist, int64_t node_stride, int64_t time_stride, int s0, int ring, int Th, int d,
                      const int64_t* ids, int64_t n_ids, const float* G, float* out, int64_t out_stride,
                      const int64_t* out_ids, void* stream, bool prefetch_old_rows) {
  if (n_ids < 0 || Th < 0 || d <= 0 || ring < Th || s0 < 0 || (ring > 0 && s0 >= ring)) return LSTEP_ERR_INVALID_ARG;
  if (n_ids == 0) return LSTEP_OK;
  if (!ids || !out || !G || (Th > 0 && !hist)) return LSTEP_ERR_INVALID_ARG;
  const bool v4 = vec4_ok(hist, node_stride, time_stride, d) && vec4_ok(G, 0, 0, d) && vec4_ok(out, out_stride, 0, d);
  const int dvec = v4 ? d / 4 : d;
  if (dvec > kDftThreads) return LSTEP_ERR_UNSUPPORTED;
  const int groups = kDftThreads / dvec;
  const size_t smem = (size_t)groups * dvec * (v4 ? 16 : 4);
  const int64_t grid = n_ids < (int64_t)num_sms() * 6 ? n_ids : (int64_t)num_sms() * 6;
  cudaStream_t st = as_stream(stream);
  {
    // node-major history: bulk-async kernel (one CTA stages a node's whole block in shared memory)
    constexpr int kBulkCtasPerSm = 3;  // what <= 74 KB of shared memory per CTA leaves room for
    const size_t bulk_smem = ((size_t)Th * dvec + (size_t)groups * dvec) * 16;
    if (v4 && time_stride == d && Th > 0 && bulk_smem <= 74 * 1024) {
      static bool attr_set = false;
      if (!attr_set) {
        cudaError_t e = cudaFuncSetAttribute(dft_filter_bulk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 74 * 1024);
        if (e != cudaSuccess) {
          set_cuda_error(e, "dft_filter_bulk attr");
          return LSTEP_ERR_CUDA;
        }
        attr_set = true;
      }
      const int64_t bgrid = n_ids < (int64_t)num_sms() * kBulkCtasPerSm ? n_ids : (int64_t)num_sms() * kBulkCtasPerSm;
      launch_k(dft_filter_bulk_kernel, dim3((unsigned)bgrid), dim3(kDftThreads), bulk_smem, st, hist, node_stride, s0, ring, Th, d, ids,
               n_ids, G, out, out_stride, out_ids, prefetch_old_rows ? 1 : 0);
      return check_launch("dft_filter_bulk");
    }
  }
  if (v4)
    launch_k(dft_filter_kernel<4>, dim3((unsigned)grid), dim3(kDftThreads), smem, st, hist, node_stride, time_stride, s0, ring, Th, d,
             ids, n_ids, G, out, out_stride, out_ids);
  else
    launch_k(dft_filter_kernel<1>, dim3((unsigned)grid), dim3(kDftThreads), smem, st, hist, node_stride, time_stride, s0, ring, Th, d,
             ids, n_ids, G, out, out_stride, out_ids);
  return check_launch("dft_filter");
}
}  // namespace lstep

extern "C" int lstep_dft_filter(const float* hist, int64_t node_stride, int64_t time_stride, int s0, int ring, int Th,
                                int d, const int64_t* ids, int64_t n_ids, const float* G, float* out,
                                int64_t out_stride, void* stream) {
  return lstep::launch_dft_filter(hist, node_stride, time_stride, s0, ring, Th, d, ids, n_ids, G, out, out_stride, nullptr, stream, false);
}

/* Same filter with the result row n written to out + out_ids[n]*out_stride (history rows and table rows
 * may use different id spaces: local ring rows vs global table rows in the sharded layout). */
extern "C" int lstep_dft_filter_scatter(const float* hist, int64_t node_stride, int64_t time_stride, int s0, int ring, int Th,
                                        int d, const int64_t* ids, const int64_t* out_ids, int64_t n_ids, const float* G,
                                        float* out, int64_t out_stride, void* stream) {
  if (!out_ids && n_ids > 0) return LSTEP_ERR_INVALID_ARG;
  return lstep::launch_dft_filter(hist, node_stride, time_stride, s0, ring, Th, d, ids, n_ids, G, out, out_stride, out_ids, stream, false);
}

extern "C" int lstep_dft_filter_bwd(const float* hist, int64_t node_stride, int64_t time_stride, int s0, int ring,
                                    int Th, int d, const int64_t* ids, int64_t n_ids, const float* dout, float* dG,
                                    void* stream) {
  if (n_ids < 0 || Th < 0 || d <= 0 || ring < Th || s0 < 0) return LSTEP_ERR_INVALID_ARG;
  if (n_ids == 0 || Th == 0) return LSTEP_OK;
  if (!hist || !ids || !dout || !dG) return LSTEP_ERR_INVALID_ARG;
  const bool v4 = vec4_ok(hist, node_stride, time_stride, d) && vec4_ok(dout, 0, 0, d);
  const int dvec = v4 ? d / 4 : d;
  if (dvec > kDftThreads) return LSTEP_ERR_UNSUPPORTED;
  const int groups = kDftThreads / dvec;
  int64_t slices = ceil_div((int64_t)num_sms() * 4, ceil_div(Th, groups));
  if (slices > n_ids) slices = n_ids;
  if (slices < 1) slices = 1;
  dim3 grid((unsigned)ceil_div(Th, groups), (unsigned)slices);
  if (v4)
    dft_filter_bwd_kernel<4><<<grid, kDftThreads, 0, as_stream(stream)>>>(hist, node_stride, time_stride, s0, ring, Th,
                                                                          d, ids, n_ids, dout, dG);
  else
    dft_filter_bwd_kernel<1><<<grid, kDftThreads, 0, as_stream(stream)>>>(hist, node_stride, time_stride, s0, ring, Th,
                                                                          d, ids, n_ids, dout, dG);
  return check_launch("dft_filter_bwd");
}

LSTEP_TIMELINE_DEFINE(dft)
