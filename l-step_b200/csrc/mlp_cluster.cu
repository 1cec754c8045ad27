// PE MLP, cluster split-K form (the default path of launch_pe_mlp):
//
//   out = base + tanh( [Ws base + bs] + W2 relu(W1 A + b1) + b2 )        (same function as csrc/mlp.cu;
//   models/LSTEP.py:240-247, :294-301, :329-336)
//
// Why: a launch has 300..1200 rows (B=200) and 0.42 MB of fp32 weights. With all output columns in one CTA
// every CTA has to stream every weight through its shared memory for a handful of rows (csrc/mlp.cu: 423 KB
// per 8 rows, measured 36 % of issued instructions being FMAs). Here a thread-block CLUSTER of 4 CTAs owns a
// tile of RB = 4*TR rows and splits the REDUCTION dimension: CTA j keeps the k-slice j of all three weight
// matrices resident in shared memory (one cp.async.bulk each, 120 KB, loaded once per launch and reused by
// every row tile the cluster walks), computes partial sums of its slice for all output columns, and the
// partials are reduce-scattered over distributed shared memory: CTA j receives, from its three peers and
// itself, the partial sums of output columns [j*kc, (j+1)*kc) — which is exactly the k-slice of the hidden
// row it needs for the second layer, so no all-gather follows. 4x less weight traffic per row than the
// all-columns kernel, weights never leave shared memory, and the inner loop is 4*TR FMAs per (1 + TR/4)
// 128-bit shared loads.
//
//   thread  = (row group rg of 4, column group of 4 outputs, k half ks of 2): TR x 4 register tile; the two k
//             halves are the two half-warps and are combined with one shuffle per accumulator
//   smem    = W1[k1][ldo] | W2[k2][ldo] | Ws[k2][ldo] | A^T[k1][RBp] | H^T[k2][RBp] | B^T[k2][RBp] | Red1 | Red2
//             k1 = rows(d+t)/4, k2 = rows(d)/4; activations k-major so one 128-bit broadcast load feeds 4 rows
//   Red1/2  = [4 source CTAs][RB][kc] receive buffers of the two reduce-scatters (summed in source order:
//             deterministic). Partials travel as st.async (SASS STAS.128) that complete transaction bytes on an
//             mbarrier of the RECEIVING CTA, so a reduce-scatter costs no cluster barrier and no memory fence:
//             the owner simply waits until 4*RB*kc*4 bytes have landed. (The first version used
//             st.shared::cluster + barrier.cluster release/acquire: ncu showed 20 % of the kernel in
//             MEMBAR / UCGABAR_WAIT.)
#include <cstdlib>

#include "common.cuh"
#include "mlp_job.cuh"

namespace lstep {
namespace {

__device__ __forceinline__ uint32_t cluster_rank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
// address of the same shared-memory offset in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t map_to_rank(uint32_t local_addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_addr), "r"(rank));
  return r;
}
// 16-byte store into a peer's shared memory that completes 16 transaction bytes on the peer's mbarrier
__device__ __forceinline__ void st_async_f4(uint32_t addr, float4 v, uint32_t remote_bar) {
  asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v4.f32 [%0], {%1, %2, %3, %4}, [%5];" ::"r"(addr),
               "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w), "r"(remote_bar)
               : "memory");
}
__device__ __forceinline__ void cluster_arrive() { asm volatile("barrier.cluster.arrive.relaxed;" ::: "memory"); }
__device__ __forceinline__ void cluster_wait() { asm volatile("barrier.cluster.wait.acquire;" ::: "memory"); }

constexpr int kCl = 4;  // CTAs per cluster = k slices

#ifdef LSTEP_MLP_TIMING
__device__ long long g_mlp_clk[16];
#define MLP_T(i) do { if (blockIdx.x == 0 && threadIdx.x == 0) g_mlp_clk[i] = clock64(); } while (0)
#else
#define MLP_T(i)
#endif

struct ClShape {
  int ldo, k1, k2, ncg, wpr, nthreads, kc;
  size_t smem_floats;
};

// rows per thread TR need not be a multiple of 4: in the k-major activation rows every row group owns a segment of
// TRP = TR rounded up to 4 floats, so the 128-bit loads of a thread stay aligned (TR = 10: 40-row tiles, which
// cover ~1200 rows in 30 of the 33 co-resident clusters and save a sixth of the inner loop against TR = 12)
__host__ __device__ constexpr int cl_trp(int TR) { return (TR + 3) / 4 * 4; }

__host__ __device__ inline ClShape cl_shape(int d, int t, bool has_self, int RB) {
  ClShape s;
  s.ldo = (int)align_up((size_t)d, 32);
  const int in1_pad = (int)align_up((size_t)(d + t), 16), d_pad = (int)align_up((size_t)d, 16);
  s.k1 = in1_pad / kCl;
  s.k2 = d_pad / kCl;
  s.ncg = d_pad / 4;       // column groups of 4 outputs (padded columns have zero weights and zero bias)
  s.kc = d_pad / kCl;      // output columns owned by one CTA == its k slice of the hidden row
  s.wpr = (s.ncg + 15) / 16;  // warps per row group: 16 column groups x 2 k halves per warp
  s.nthreads = 4 * s.wpr * 32;
  const int RBp = 4 * cl_trp(RB / 4) + 4;
  s.smem_floats = (size_t)(s.k1 + s.k2 + (has_self ? s.k2 : 0)) * s.ldo + (size_t)(s.k1 + 2 * s.k2) * RBp + (size_t)2 * kCl * RB * s.kc +
                  (size_t)2 * s.kc;  // + the owned slices of b1 and b2 (+ bs)
  return s;
}

// one k-run over `kn` weight rows (this thread's half), TR x 4 register tile. The operands of step k+1 are
// fetched before the FMAs of step k (register double buffering: with 3 warps per scheduler the 29-cycle
// shared-memory latency is otherwise exposed); the fetch past the last row reads the next buffer in
// shared memory, never out of the allocation, and its values are not used.
template <int TR>
__device__ __forceinline__ void k_run(const float* __restrict__ w, int ldo, const float* __restrict__ a, int RBp, int kn,
                                      float (&acc)[TR][4]) {
  // Accumulators are kept as row PAIRS so that one packed FFMA2 (fma.rn.f32x2, sm_100: two IEEE fp32 FMAs per
  // issue slot, each bit-identical to fmaf) updates rows 2p and 2p+1 of a column: the activation pair comes
  // straight out of the 128-bit shared load, the weight is duplicated once per column and k step. The loop is
  // issue bound (32 FMAs + 3 loads per k step and warp), so halving the FMA instructions is the lever.
  float2 acc2[TR / 2][4];
#pragma unroll
  for (int p = 0; p < TR / 2; ++p)
#pragma unroll
    for (int c = 0; c < 4; ++c) acc2[p][c] = make_float2(acc[2 * p][c], acc[2 * p + 1][c]);
  float4 wv = *reinterpret_cast<const float4*>(w);
  constexpr int NQ = cl_trp(TR) / 4;  // 128-bit activation loads per k step (the last may carry unused padding)
  float4 av[NQ];
#pragma unroll
  for (int q = 0; q < NQ; ++q) av[q] = *reinterpret_cast<const float4*>(a + 4 * q);
#pragma unroll 2
  for (int k = 0; k < kn; ++k) {
    w += ldo;
    a += RBp;
    const float4 wn = *reinterpret_cast<const float4*>(w);
    float4 an[NQ];
#pragma unroll
    for (int q = 0; q < NQ; ++q) an[q] = *reinterpret_cast<const float4*>(a + 4 * q);
    const float2 wd[4] = {make_float2(wv.x, wv.x), make_float2(wv.y, wv.y), make_float2(wv.z, wv.z), make_float2(wv.w, wv.w)};
#pragma unroll
    for (int q = 0; q < NQ; ++q) {
      const float2 lo = make_float2(av[q].x, av[q].y), hi = make_float2(av[q].z, av[q].w);
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        if (2 * q < TR / 2) acc2[2 * q][c] = __ffma2_rn(lo, wd[c], acc2[2 * q][c]);
        if (2 * q + 1 < TR / 2) acc2[2 * q + 1][c] = __ffma2_rn(hi, wd[c], acc2[2 * q + 1][c]);
      }
    }
    wv = wn;
#pragma unroll
    for (int q = 0; q < NQ; ++q) av[q] = an[q];
  }
#pragma unroll
  for (int p = 0; p < TR / 2; ++p)
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      acc[2 * p][c] = acc2[p][c].x;
      acc[2 * p + 1][c] = acc2[p][c].y;
    }
}

template <int TR>
__global__ void __cluster_dims__(kCl, 1, 1) __launch_bounds__(512, 1)
    pe_mlp_cluster_kernel(const __grid_constant__ MlpJob job0, const __grid_constant__ MlpJob job1, int split, const float* pe,
                          FixedRows fx) {
  constexpr int RB = 4 * TR, TRP = cl_trp(TR), RBp = 4 * TRP + 4;
  auto col_of = [](int r) { return (r / TR) * TRP + r % TR; };  // position of tile row r in a k-major activation row
  const int64_t cluster_raw = blockIdx.x / kCl;
  const bool second = cluster_raw >= split;
  const MlpJob& jb = second ? job1 : job0;
  const float* __restrict__ A = jb.A;
  const int64_t lda = jb.lda;
  const RowIds& base_ids = jb.base_ids;
  int64_t n_rows = jb.n_rows;
  const int32_t* __restrict__ n_rows_dev = jb.n_rows_dev;
  const lstep_pe_mlp& m = jb.m;
  float* __restrict__ out = jb.out;
  const int64_t out_stride = jb.out_stride;
  float* pe_inplace = jb.pe_inplace;
  extern __shared__ __align__(128) float smem[];
  __shared__ __align__(8) uint64_t wbar[2];  // weight slices landed (layer 1, layer 2)
  __shared__ __align__(8) uint64_t rbar[2];  // reduce-scatter 1 / 2 of the current row tile landed
  __shared__ int64_t s_node[RB];             // base node id of every row of the tile
  const int d = m.d, in1 = m.d + m.t;
  const bool has_self = m.ws != nullptr;
  const ClShape sh = cl_shape(d, m.t, has_self, RB);
  const int ldo = sh.ldo, k1 = sh.k1, k2 = sh.k2, kc = sh.kc, ncg = sh.ncg;
  const uint32_t j = cluster_rank();
  const int64_t pe_rows = fx.pe_rows;
  auto clamp_row = [pe_rows](int64_t node) { return (pe_rows > 0 && (node < 0 || node >= pe_rows)) ? (int64_t)0 : node; };
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int nthr = blockDim.x;

  float* W1s = smem;
  float* W2s = W1s + (size_t)k1 * ldo;  // W2 slice, then (contiguous) the Ws slice: layer 2 is one k-run over [h ; base]
  float* As = W2s + (size_t)(has_self ? 2 : 1) * k2 * ldo;
  float* Hs = As + (size_t)k1 * RBp;
  float* Bs = Hs + (size_t)k2 * RBp;
  float* Red1 = Bs + (size_t)k2 * RBp;
  float* Red2 = Red1 + (size_t)kCl * RB * kc;
  float* bias1 = Red2 + (size_t)kCl * RB * kc;  // [kc] b1 of the owned columns
  float* bias2 = bias1 + kc;                    // [kc] b2 (+ bs)
  const uint32_t red_bytes = (uint32_t)(kCl * RB * kc * sizeof(float));  // what one reduce-scatter delivers to this CTA

  // ---- everything that does not depend on the preceding kernel: barriers, the weight slices (parameters),
  // the bias slices, the cluster rendezvous. With programmatic dependent launch this overlaps the tail of
  // the kernel in front.
  TL_ENTRY(fx.acc ? 4 : 2);
  if (!fx.late_trigger) pdl_launch_dependents();
  if (tid == 0) {
    mb_init(&wbar[0], 1);
    mb_init(&wbar[1], 1);
    mb_init(&rbar[0], 1);
    mb_init(&rbar[1], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    // this CTA's k slices of the packed weights: contiguous row blocks
    const uint32_t b1 = (uint32_t)k1 * ldo * 4u, b2 = (uint32_t)k2 * ldo * 4u;
    mb_expect_tx(&wbar[0], b1);
    bulk_load(W1s, m.w1 + (size_t)j * k1 * ldo, b1, &wbar[0]);
    mb_expect_tx(&wbar[1], has_self ? 2 * b2 : b2);
    bulk_load(W2s, m.w2 + (size_t)j * k2 * ldo, b2, &wbar[1]);
    if (has_self) bulk_load(W2s + (size_t)k2 * ldo, m.ws + (size_t)j * k2 * ldo, b2, &wbar[1]);
    mb_expect_tx(&rbar[0], red_bytes);
    mb_expect_tx(&rbar[1], red_bytes);
  }
  for (int c = tid; c < kc; c += nthr) {
    const int col = (int)j * kc + c;  // packed biases are zero padded to ldo >= d_pad
    bias1[c] = m.b1[col];
    bias2[c] = m.b2[col] + (has_self ? m.bs[col] : 0.f);
  }
  __syncthreads();
  // every CTA of the cluster must be running, with its barriers initialised, before a peer stores into it:
  // arrive now, wait right before the first remote store (the staging and layer 1 run in between)
  cluster_arrive();
  const bool ids_early = fx.ids_stable && !n_rows_dev;
  if (ids_early && tid < RB) {
    const int64_t cl = second ? cluster_raw - split : cluster_raw;
    const int64_t row = cl * RB + tid;
    s_node[tid] = row < n_rows ? clamp_row(base_ids.at(row)) : 0;
  }
  pdl_wait();  // from here on the kernel reads what the preceding kernels wrote
  TL_WAITED(fx.acc ? 4 : 2);
  MLP_T(0);
  if (n_rows_dev) {
    const int64_t nd = ld_dep(n_rows_dev);
    n_rows = nd < n_rows ? nd : n_rows;
  }
  // (after the row-count read: a kernel that becomes resident on this trigger may reset the counter)
  if (fx.late_trigger) pdl_launch_dependents();
  const int64_t n_tiles = (n_rows + RB - 1) / RB;
  const int64_t cluster_id = second ? cluster_raw - split : cluster_raw;
  const int64_t n_clusters = second ? (int64_t)(gridDim.x / kCl) - split : (int64_t)split;
  const bool idle = cluster_id >= n_tiles;  // a cluster without a row tile still completes the rendezvous and drains its copies
  if (!ids_early && tid < RB) {  // first dependent load chain of the kernel (id -> base row)
    const int64_t row = cluster_id * RB + tid;
    s_node[tid] = (!idle && row < n_rows) ? clamp_row(base_ids.at_dep(row)) : 0;
  }
  __syncthreads();
  if (idle) {
    cluster_wait();
    mb_wait(&wbar[0], 0);
    mb_wait(&wbar[1], 0);
    return;
  }
  MLP_T(1);

  // thread coordinates
  const int rg = warp / sh.wpr;
  const int cg_raw = (warp % sh.wpr) * 16 + (lane & 15);
  const bool col_ok = cg_raw < ncg;
  const int cg = col_ok ? cg_raw : ncg - 1;
  const int ks = lane >> 4;
  const int cgs_per_owner = ncg / kCl;
  const uint32_t owner = (uint32_t)(cg / cgs_per_owner);
  const int oc = (cg % cgs_per_owner) * 4;  // column inside the owner's slice
  // where this thread's partial tile lands in the owner's receive buffers (source slot j)
  const uint32_t red_off = (uint32_t)((((size_t)j * RB + rg * TR) * kc + oc) * sizeof(float));
  const uint32_t red1_remote = map_to_rank(s_u32(Red1), owner) + red_off;
  const uint32_t red2_remote = map_to_rank(s_u32(Red2), owner) + red_off;
  const uint32_t rbar1_remote = map_to_rank(s_u32(&rbar[0]), owner);
  const uint32_t rbar2_remote = map_to_rank(s_u32(&rbar[1]), owner);
  const bool a_vec = (lda % 4 == 0) && ((reinterpret_cast<uintptr_t>(A) & 15) == 0);
  const bool p_vec = (d % 4 == 0) && ((reinterpret_cast<uintptr_t>(pe) & 15) == 0);
  const int kA0 = (int)j * k1, kB0 = (int)j * k2;  // first global k of this CTA's slices

  auto send = [&](uint32_t base, uint32_t bar, const float (&acc)[TR][4]) {
    if (ks == 0 && col_ok) {
#pragma unroll
      for (int r = 0; r < TR; ++r)
        st_async_f4(base + (uint32_t)(r * kc * sizeof(float)), make_float4(acc[r][0], acc[r][1], acc[r][2], acc[r][3]), bar);
    }
  };
  auto load4 = [&](const float* p, int kg, int lim, bool vec) {
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (vec && kg + 3 < lim) {  // ld_dep: both operands are written by earlier kernels of the step
      v = ld_dep(reinterpret_cast<const float4*>(p));
    } else {
      if (kg + 0 < lim) v.x = ld_dep(p + 0);
      if (kg + 1 < lim) v.y = ld_dep(p + 1);
      if (kg + 2 < lim) v.z = ld_dep(p + 2);
      if (kg + 3 < lim) v.w = ld_dep(p + 3);
    }
    return v;
  };
  auto load4_fixed = [&](const unsigned long long* p, int kg, int lim) {
    constexpr float kInv = 2.3283064365386963e-10f;  // 2^-32
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (kg + 3 < lim && (reinterpret_cast<uintptr_t>(p) & 15) == 0) {
      const ulonglong2 a = __ldcg(reinterpret_cast<const ulonglong2*>(p)), b = __ldcg(reinterpret_cast<const ulonglong2*>(p) + 1);
      v.x = (float)(long long)a.x * kInv;
      v.y = (float)(long long)a.y * kInv;
      v.z = (float)(long long)b.x * kInv;
      v.w = (float)(long long)b.y * kInv;
    } else {
      if (kg + 0 < lim) v.x = (float)(long long)__ldcg(p + 0) * kInv;
      if (kg + 1 < lim) v.y = (float)(long long)__ldcg(p + 1) * kInv;
      if (kg + 2 < lim) v.z = (float)(long long)__ldcg(p + 2) * kInv;
      if (kg + 3 < lim) v.w = (float)(long long)__ldcg(p + 3) * kInv;
    }
    return v;
  };
  auto put4 = [&](float* dst, float4 v) {
    dst[0] = v.x;
    dst[RBp] = v.y;
    dst[2 * RBp] = v.z;
    dst[3 * RBp] = v.w;
  };

  const int nA = RB * (k1 / 4), nB = RB * (k2 / 4);
  uint32_t it = 0;  // row tiles done by this cluster: parity of the reduce-scatter barriers
  for (int64_t tile = cluster_id; tile < n_tiles; tile += n_clusters, ++it) {
    const int64_t row0 = tile * RB;
    if (it > 0) {
      if (tid < RB) {
        const int64_t row = row0 + tid;
        s_node[tid] = row < n_rows ? clamp_row(base_ids.at_dep(row)) : 0;
      }
      __syncthreads();
    }
    // ---- stage this CTA's k slices of the aggregate rows and of the base rows, transposed to k-major.
    // lane -> row, so the transposing shared stores are conflict free; each thread moves 4 consecutive k.
    // All global loads of a pass are issued before the first store (one latency, not one per element).
    for (int base = 0; base < nA + nB; base += 4 * nthr) {
      float4 v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int idx = base + u * nthr + tid;
        v[u] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (idx < nA) {
          const int r = idx % RB, q = idx / RB;
          const int64_t row = row0 + r;
          const int kg = kA0 + 4 * q;
          if (row < n_rows) v[u] = fx.acc ? load4_fixed(fx.acc + row * (int64_t)in1 + kg, kg, in1) : load4(A + row * lda + kg, kg, in1, a_vec);
        } else if (idx < nA + nB) {
          const int r = (idx - nA) % RB, q = (idx - nA) / RB;
          const int kg = kB0 + 4 * q;
          // plain (not read-only-cache) loads: the table is written by this kernel when it runs in place
          if (row0 + r < n_rows) v[u] = load4(pe + s_node[r] * (int64_t)d + kg, kg, d, p_vec);
        }
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int idx = base + u * nthr + tid;
        if (idx < nA) {
          put4(As + (size_t)(4 * (idx / RB)) * RBp + col_of(idx % RB), v[u]);
        } else if (idx < nA + nB) {
          put4(Bs + (size_t)(4 * ((idx - nA) / RB)) * RBp + col_of((idx - nA) % RB), v[u]);
        }
      }
    }
    __syncthreads();
    MLP_T(2);
    if (it == 0) mb_wait(&wbar[0], 0);
    MLP_T(3);

    // ---- layer 1: partial sums of this CTA's k slice, all output columns
    float acc[TR][4];
#pragma unroll
    for (int r = 0; r < TR; ++r) acc[r][0] = acc[r][1] = acc[r][2] = acc[r][3] = 0.f;
    {
      const int kh = k1 / 2;
      k_run<TR>(W1s + (size_t)(ks * kh) * ldo + 4 * cg, ldo, As + (size_t)(ks * kh) * RBp + rg * TRP, RBp, kh, acc);
    }
#pragma unroll
    for (int r = 0; r < TR; ++r)
#pragma unroll
      for (int c = 0; c < 4; ++c) acc[r][c] += __shfl_xor_sync(kFull, acc[r][c], 16);  // combine the two k halves
    MLP_T(4);
    if (it == 0) cluster_wait();
    MLP_T(5);
    send(red1_remote, rbar1_remote, acc);
    MLP_T(6);

    // ---- hidden slice owned by this CTA: h = relu(sum of the 4 partials + b1), k-major
    mb_wait(&rbar[0], it & 1);
    MLP_T(7);
    for (int idx = tid; idx < RB * (kc / 4); idx += nthr) {  // lane -> row: conflict-free 128-bit reads and k-major stores
      const int r = idx % RB, c = 4 * (idx / RB);
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int s = 0; s < kCl; ++s) {
        const float4 p = *reinterpret_cast<const float4*>(Red1 + ((size_t)s * RB + r) * kc + c);
        v.x += p.x;
        v.y += p.y;
        v.z += p.z;
        v.w += p.w;
      }
      const float4 b = *reinterpret_cast<const float4*>(bias1 + c);
      const int col = (int)j * kc + c;
      float* dst = Hs + (size_t)c * RBp + col_of(r);
      dst[0] = col + 0 < d ? fmaxf(v.x + b.x, 0.f) : 0.f;
      dst[RBp] = col + 1 < d ? fmaxf(v.y + b.y, 0.f) : 0.f;
      dst[2 * RBp] = col + 2 < d ? fmaxf(v.z + b.z, 0.f) : 0.f;
      dst[3 * RBp] = col + 3 < d ? fmaxf(v.w + b.w, 0.f) : 0.f;
    }
    __syncthreads();
    if (tid == 0) mb_expect_tx(&rbar[0], red_bytes);  // arm the next tile's phase (every reader is past Red1)
    MLP_T(8);
    if (it == 0) mb_wait(&wbar[1], 0);
    MLP_T(9);

    // ---- layer 2 (+ self term): one k-run over [h slice ; base slice] against [W2 slice ; Ws slice]
#pragma unroll
    for (int r = 0; r < TR; ++r) acc[r][0] = acc[r][1] = acc[r][2] = acc[r][3] = 0.f;
    {
      const int kn = has_self ? 2 * k2 : k2;  // Hs and Bs are adjacent, so are the two weight slices
      const int kh = kn / 2;
      k_run<TR>(W2s + (size_t)(ks * kh) * ldo + 4 * cg, ldo, Hs + (size_t)(ks * kh) * RBp + rg * TRP, RBp, kh, acc);
    }
#pragma unroll
    for (int r = 0; r < TR; ++r)
#pragma unroll
      for (int c = 0; c < 4; ++c) acc[r][c] += __shfl_xor_sync(kFull, acc[r][c], 16);
    MLP_T(10);
    send(red2_remote, rbar2_remote, acc);

    // ---- epilogue on the owned columns: out = base + tanh(z)
    mb_wait(&rbar[1], it & 1);
    MLP_T(11);
    const bool o_vec = (d % 4 == 0) && (out ? (out_stride % 4 == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0)
                                           : (reinterpret_cast<uintptr_t>(pe_inplace) & 15) == 0);
    for (int idx = tid; idx < RB * (kc / 4); idx += nthr) {
      const int r = idx % RB, c = 4 * (idx / RB);
      const int col = (int)j * kc + c;
      const int64_t row = row0 + r;
      if (row < n_rows && col < d) {
        float4 z = *reinterpret_cast<const float4*>(bias2 + c);
#pragma unroll
        for (int s = 0; s < kCl; ++s) {
          const float4 p = *reinterpret_cast<const float4*>(Red2 + ((size_t)s * RB + r) * kc + c);
          z.x += p.x;
          z.y += p.y;
          z.z += p.z;
          z.w += p.w;
        }
        const float* bp = Bs + (size_t)c * RBp + col_of(r);
        float4 o;
        o.x = bp[0] + tanhf(z.x);
        o.y = bp[RBp] + tanhf(z.y);
        o.z = bp[2 * RBp] + tanhf(z.z);
        o.w = bp[3 * RBp] + tanhf(z.w);
        if (fx.ring_slot) {  // (d % 4 == 0 and 16-byte rows are preconditions of the streaming step)
          *reinterpret_cast<float4*>(fx.ring_slot + s_node[r] * fx.ring_stride + col) = o;
        }
        auto store = [&](float* dst) {
          if (o_vec && col + 3 < d) {
            *reinterpret_cast<float4*>(dst) = o;
          } else {
            dst[0] = o.x;
            if (col + 1 < d) dst[1] = o.y;
            if (col + 2 < d) dst[2] = o.z;
            if (col + 3 < d) dst[3] = o.w;
          }
        };
        if (out && jb.fan.n_out > 0) {  // identical query sets were computed once: fan the row out
          const int64_t u = row / jb.fan.period, i = row % jb.fan.period;
          for (int c = 0; c < jb.fan.n_out; ++c)
            if (jb.fan.src_of[c] == u) store(out + (c * jb.fan.period + i) * out_stride + col);
        } else {
          store((out ? out + row * out_stride : pe_inplace + s_node[r] * (int64_t)d) + col);
        }
      }
    }
    if (fx.reset_map && j == 0 && tid < RB && row0 + tid < n_rows) fx.reset_map[s_node[tid]] = 0;
    MLP_T(12);
    __syncthreads();  // As / Hs / Bs / s_node are restaged by the next row tile; every reader is past Red2
    if (tid == 0) mb_expect_tx(&rbar[1], red_bytes);
  }
  TL_EXIT(fx.acc ? 4 : 2);
}

template <int TR>
int launch_cl(const MlpJob& j0, const MlpJob* j1, const float* pe, FixedRows fx, cudaStream_t st) {
  constexpr int RB = 4 * TR;
  const lstep_pe_mlp* m = &j0.m;
  const ClShape sh = cl_shape(m->d, m->t, m->ws != nullptr, RB);
  const size_t smem = sh.smem_floats * sizeof(float);
  if (smem > 226 * 1024 || sh.nthreads > 512 || sh.ncg % kCl != 0) return LSTEP_ERR_UNSUPPORTED;
  if (j1 && (j1->m.d != m->d || j1->m.t != m->t || (j1->m.ws != nullptr) != (m->ws != nullptr))) return LSTEP_ERR_UNSUPPORTED;
  auto kern = pe_mlp_cluster_kernel<TR>;
  static int max_clusters = 0;  // co-resident clusters of 4 (B200: 33 — some GPCs strand SMs), queried once
  if (max_clusters == 0) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 226 * 1024);
    if (e != cudaSuccess) {
      set_cuda_error(e, "pe_mlp_cluster attr");
      return LSTEP_ERR_CUDA;
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(num_sms() / kCl * kCl);
    cfg.blockDim = dim3(sh.nthreads);
    cfg.dynamicSmemBytes = 226 * 1024;
    cudaLaunchAttribute attr;
    attr.id = cudaLaunchAttributeClusterDimension;
    attr.val.clusterDim.x = kCl;
    attr.val.clusterDim.y = 1;
    attr.val.clusterDim.z = 1;
    cfg.attrs = &attr;
    cfg.numAttrs = 1;
    int n = 0;
    e = cudaOccupancyMaxActiveClusters(&n, kern, &cfg);
    if (e != cudaSuccess || n <= 0) {
      (void)cudaGetLastError();
      n = 32;
    }
    max_clusters = n;
  }
  int64_t c0 = ceil_div(j0.n_rows, RB), c1 = j1 ? ceil_div(j1->n_rows, RB) : 0;
  if (j1) {
    if (c0 + c1 > max_clusters) return LSTEP_ERR_UNSUPPORTED;  // a pair must fit one round (the caller picks a larger tile or splits)
  } else if (c0 > max_clusters) {
    c0 = max_clusters;  // persistent: the cluster walks row tiles, weights stay resident
  }
  launch_k(kern, dim3((unsigned)((c0 + c1) * kCl)), dim3(sh.nthreads), smem, st, j0, j1 ? *j1 : j0, (int)c0, pe, fx);
  return check_launch("pe_mlp_cluster");
}

}  // namespace

// expected_rows: the typical row count (n_rows is only an upper bound when n_rows_dev carries the real one).
// acc_fixed / reset_map: see FixedRows (both NULL: the aggregate is the float matrix A).
int launch_pe_mlp_cluster(const float* A, int64_t lda, const float* pe, RowIds base_ids, int64_t n_rows, int64_t expected_rows,
                          const int32_t* n_rows_dev, const lstep_pe_mlp* m, float* out, int64_t out_stride, float* pe_inplace,
                          const unsigned long long* acc_fixed, int32_t* reset_map, cudaStream_t st, bool late_trigger,
                          float* ring_slot, int64_t ring_stride, const OutFan* fan, int64_t pe_rows) {
  const FixedRows fx{acc_fixed, reset_map, late_trigger ? 1 : 0, ring_slot, ring_stride, pe_rows, 0};
  const MlpJob j{A, lda, base_ids, n_rows, n_rows_dev, *m, out, out_stride, pe_inplace, fan ? *fan : OutFan{}};
  if (pe_mlp_umma_wanted(m, expected_rows)) {  // large launches: tcgen05 3xTF32 kernel (csrc/mlp_umma.cu)
    const int rc = launch_pe_mlp_umma(j, nullptr, pe, fx, st);
    if (rc != LSTEP_ERR_UNSUPPORTED) return rc;
  }
  // rows per cluster tile: the smallest tile that covers the launch in one round of ~32 co-resident clusters
  if (expected_rows <= 32 * 16) return launch_cl<4>(j, nullptr, pe, fx, st);
  if (expected_rows <= 32 * 32) return launch_cl<8>(j, nullptr, pe, fx, st);
  if (expected_rows <= 33 * 40) {
    const int rc10 = launch_cl<10>(j, nullptr, pe, fx, st);
    if (rc10 != LSTEP_ERR_UNSUPPORTED) return rc10;
  }
  const int rc = launch_cl<12>(j, nullptr, pe, fx, st);
  if (rc != LSTEP_ERR_UNSUPPORTED) return rc;
  return launch_cl<8>(j, nullptr, pe, fx, st);
}

// Two float-input jobs in one launch (see MlpJob); LSTEP_ERR_UNSUPPORTED when they do not fit one round of clusters.
int launch_pe_mlp_cluster_pair(const float* pe, const float* A0, int64_t lda0, RowIds ids0, int64_t rows0, const lstep_pe_mlp* m0,
                               float* out0, int64_t out_stride0, const float* A1, int64_t lda1, RowIds ids1, int64_t rows1,
                               const lstep_pe_mlp* m1, float* out1, int64_t out_stride1, cudaStream_t st, bool late_trigger,
                               int64_t pe_rows, const OutFan* fan0) {
  if (rows0 <= 0 || rows1 <= 0 || !out0 || !out1) return LSTEP_ERR_UNSUPPORTED;
  const FixedRows fx{nullptr, nullptr, late_trigger ? 1 : 0, nullptr, 0, pe_rows, 1};  // (the step's id lists are stable)
  const MlpJob j0{A0, lda0, ids0, rows0, nullptr, *m0, out0, out_stride0, nullptr, fan0 ? *fan0 : OutFan{}};
  const MlpJob j1{A1, lda1, ids1, rows1, nullptr, *m1, out1, out_stride1, nullptr, OutFan{}};
  if (pe_mlp_umma_wanted(m0, rows0 + rows1)) {
    const int rc = launch_pe_mlp_umma(j0, &j1, pe, fx, st);
    if (rc != LSTEP_ERR_UNSUPPORTED) return rc;
  }
  int rc = launch_cl<4>(j0, &j1, pe, fx, st);
  if (rc == LSTEP_ERR_UNSUPPORTED) rc = launch_cl<8>(j0, &j1, pe, fx, st);
  if (rc == LSTEP_ERR_UNSUPPORTED) rc = launch_cl<10>(j0, &j1, pe, fx, st);
  if (rc == LSTEP_ERR_UNSUPPORTED) rc = launch_cl<12>(j0, &j1, pe, fx, st);
  return rc;
}

// true when the cluster kernel covers this MLP shape (the push form of update_pe phase B depends on it)
bool pe_mlp_cluster_supports(const lstep_pe_mlp* m) {
  if (!m) return false;
  const ClShape sh = cl_shape(m->d, m->t, m->ws != nullptr, 32);
  return sh.smem_floats * sizeof(float) <= 226 * 1024 && sh.nthreads <= 512 && sh.ncg % kCl == 0;
}

LSTEP_TIMELINE_DEFINE(mlp)

#ifdef LSTEP_MLP_TIMING
extern "C" int lstep_debug_mlp_clocks(long long* out16) {
  return cudaMemcpyFromSymbol(out16, g_mlp_clk, sizeof(long long) * 16) == cudaSuccess ? 0 : 4;
}
#endif

}  // namespace lstep
