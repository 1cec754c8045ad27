// Shared device/host helpers for the lstep_b200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <cmath>
#include <utility>

#include "lstep_b200.h"

namespace lstep {

constexpr int kWarp = 32;
constexpr unsigned kFull = 0xffffffffu;
// SM count of the current device (B200: 148 = 2 dies x 74), queried once per process; grids are sized in multiples of it
int num_sms();

// Runtime switches, each the way a test reaches a shipped path or its reference on the same inputs. Initialised ONCE
// (first use) from the LSTEP_* environment variables DESIGN.md lists and changed with lstep_set_option(); the launch paths
// read plain ints. Every default is the shipped path.
struct Tuning {
  int pdl = 1;                // programmatic dependent launch along the step's kernel chain      (LSTEP_NO_PDL=1 -> 0)
  int phaseb_push = 1;        // push form of phase B (0: count / scan / fill / gather pull form)  (LSTEP_PHASEB_PULL)
  int gather_pipe = 1;        // multi-row gather CTAs with a look-ahead lookup warp (B = 2000)     (LSTEP_NO_GATHER_PIPE)
  int mlp_umma = 1;           // tcgen05 tensor-core MLP for launches with >= mlp_umma_min_rows rows (LSTEP_NO_MLP_UMMA)
  int mlp_umma_min_rows = 1536;  //                                                                (LSTEP_MLP_UMMA_MIN_ROWS)
  int profile = 0;            // lstep_step_profile(): CUDA events around every kernel of the streaming step
};
Tuning& tuning();

// lstep_step_profile(1): the streaming step records a CUDA event on its launch stream before its first kernel and after
// each of its kernels (slots below). Events between kernels also serialise the chain (no programmatic overlap across an
// event), so the durations are those of the step's own kernels run back to back on live data — the per-kernel roofline
// figures of bench.py — while the step time itself is always measured with profiling off.
// (peer group step, csrc/peer.cu: kProfDft = owned filter + announcement of barrier 1, kProfWait1 / kProfWait2 = time spent waiting
// for the other ranks, kProfBcast = phase-A rows into every rank's buffer + announcement of barrier 2)
enum ProfSlot { kProfStart = 0, kProfDft, kProfWait1, kProfGather, kProfMlpPair, kProfBcast, kProfWait2, kProfPush, kProfMlpB, kProfAppend, kProfSlots };
void prof_mark(cudaStream_t st, int slot);

// last CUDA error text, for lstep_last_cuda_error()
void set_cuda_error(cudaError_t e, const char* where);
int check_launch(const char* where);

inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }

__host__ __device__ inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }
__host__ __device__ inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// ---- programmatic dependent launch (PDL) ------------------------------------------------------------
// The step is a chain of ~11 short, dependent kernels; a plain stream launch starts kernel n+1 only after
// kernel n has drained (2-4 us of launch latency each, a fifth of the step). Every kernel of the chain
// therefore (a) lets its successor be scheduled early (pdl_launch_dependents, first instruction) and
// (b) calls pdl_wait() before its first access to global memory that a predecessor may have written or may
// still read; griddepcontrol.wait returns when all preceding grids have completed and their writes are
// visible, so the memory ordering is that of a plain launch. Launch with launch_k(); kernels that are
// launched with <<<>>> execute both instructions as no-ops.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// ---- opt-in timeline instrumentation (-DLSTEP_TIMELINE): first CTA entry, first return from the dependency wait and
// last CTA exit of every kernel of a step on the global nanosecond timer, read back with lstep_debug_timeline().
#ifdef LSTEP_TIMELINE
static __device__ unsigned long long g_timeline[64];  // one copy per translation unit (no relocatable device code)
// defines the reader of this translation unit's copy: mode 0 resets (min slots to ~0, max slots to 0), mode 1 reads
#define LSTEP_TIMELINE_DEFINE(name)                                                                   \
  extern "C" int lstep_debug_timeline_##name(int mode, unsigned long long* out64) {                   \
    unsigned long long h[64];                                                                         \
    if (mode == 0) {                                                                                  \
      for (int i = 0; i < 64; ++i) h[i] = (i % 4 == 2) ? 0ull : ~0ull;                                \
      return cudaMemcpyToSymbol(lstep::g_timeline, h, sizeof(h)) == cudaSuccess ? 0 : 4;              \
    }                                                                                                 \
    return cudaMemcpyFromSymbol(out64, lstep::g_timeline, sizeof(h)) == cudaSuccess ? 0 : 4;          \
  }
__device__ __forceinline__ unsigned long long gtimer() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
#define TL_ENTRY(k) do { if (threadIdx.x == 0) atomicMin(&g_timeline[(k) * 4 + 0], gtimer()); } while (0)
#define TL_WAITED(k) do { if (threadIdx.x == 0) atomicMin(&g_timeline[(k) * 4 + 1], gtimer()); } while (0)
#define TL_EXIT(k) do { if (threadIdx.x == 0) atomicMax(&g_timeline[(k) * 4 + 2], gtimer()); } while (0)
#else
#define LSTEP_TIMELINE_DEFINE(name)
#define TL_ENTRY(k)
#define TL_WAITED(k)
#define TL_EXIT(k)
#endif

// A kernel launched this way is resident BEFORE its predecessor has finished, so it misses the L1
// invalidation a kernel boundary normally gives: a line that a predecessor CTA on the same SM pulled into L1
// (or the read-only path) and that was then rewritten from another SM would be read stale. Every load of data
// that an earlier kernel of the step WRITES therefore goes through ld_dep() = ld.global.cg (served by L2,
// the point of coherence). Plain / __ldg loads are kept for data no kernel of the step writes (CSR, packed
// parameters, the batch arrays, query ids).
__device__ __forceinline__ float ld_dep(const float* p) { return __ldcg(p); }
__device__ __forceinline__ float4 ld_dep(const float4* p) { return __ldcg(p); }
__device__ __forceinline__ int32_t ld_dep(const int32_t* p) { return __ldcg(p); }
__device__ __forceinline__ int64_t ld_dep(const int64_t* p) { return (int64_t)__ldcg(reinterpret_cast<const long long*>(p)); }

inline bool pdl_enabled() { return tuning().pdl != 0; }  // (LSTEP_NO_PDL=1 / lstep_set_option("pdl", 0): A/B measurements)

template <typename... KArgs, typename... Args>
inline cudaError_t launch_k(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at;
  cfg.numAttrs = pdl_enabled() ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kern, KArgs(std::forward<Args>(args))...);
}

// streaming 128-bit load served by L2 (history rows are read once; also see ld_dep above)
__device__ __forceinline__ float4 ld_stream_f4(const float4* p) {
  float4 v;
  asm volatile("ld.global.cg.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
               : "l"(p));
  return v;
}
__device__ __forceinline__ float ld_stream_f(const float* p) {
  float v;
  asm volatile("ld.global.cg.f32 %0, [%1];" : "=f"(v) : "l"(p));
  return v;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
  return v;
}

// Row -> node id for kernels that serve several query sets in one launch (the eval loop's C calls of
// compute_neighborhood_pe share one batch of edge times): row r belongs to set r / period.
struct RowIds {
  const int64_t* p[8];
  int64_t period;  // 0: single set, p[0][row]
  __device__ __forceinline__ int64_t at(int64_t row) const { return period ? p[row / period][row % period] : p[0][row]; }
  // ids that an earlier kernel of the step wrote (update_pe phase B: the list of distinct destinations)
  __device__ __forceinline__ int64_t at_dep(int64_t row) const {
    return period ? __ldcg(reinterpret_cast<const long long*>(p[row / period]) + row % period)
                  : __ldcg(reinterpret_cast<const long long*>(p[0]) + row);
  }
  __device__ __forceinline__ int64_t time_index(int64_t row) const { return period ? row % period : row; }
};
// push form of update_pe's phase B (csrc/update_push.cu): the padding row 0 collects a contribution from EVERY batch node with
// a padded slot (most nodes of a 10 M-node graph): thousands of 64-bit atomics per column on one accumulator row. They go to
// kPushRow0Parts partial rows instead (selected by the batch row), which the last CTA of the kernel folds into row 0's
// accumulator and returns to zero. Part of the update workspace's zero-initialised head.
constexpr int kPushRow0Parts = 32;
constexpr int kPushRow0Cols = 256;  // >= d
constexpr size_t kPushRow0Bytes = sizeof(unsigned long long) * kPushRow0Parts * kPushRow0Cols;
// Range of phase B's 32.32 fixed-point sums (both forms): a call adds at most n_ids*K contributions to one column, each
// converted as round(x * 2^32). With |x| < 2^31 / (n_ids*K + 1) every converted value is below 2^63 / (n_ids*K + 1) + 1/2,
// so every column sum (and z * fx of the padding row) stays inside int64 for any n_ids*K < 2^31 (check_update_args). The
// kernels raise LSTEP_FLAG_FIXED_POINT_RANGE for a contribution that fails `|x| < bound` (NaN included); they only compare,
// the values they add are unchanged. Rounded toward zero to fp32 (l-step_b200/_lib.py::fixed_point_bound computes the same).
inline float fixed_point_bound(int64_t n_ids, int K) {
  const double b = 2147483648.0 / ((double)n_ids * K + 1.0);
  const float f = (float)b;
  return (double)f > b ? std::nextafter(f, 0.f) : f;
}
// update_pe inside a peer group (csrc/peer.cu): this rank accumulates / rewrites only the phase-B destinations u with
// u % mul == add and applies only the phase-A rows of the batch nodes it owns; new_rows holds phase A's rows of ALL batch
// nodes (row i = ids[i], written by their owners through peer memory).
struct PushOwner {
  int mul = 1, add = 0;
  const float* new_rows = nullptr;
};
inline RowIds single_ids(const int64_t* ids) {
  RowIds r{};
  r.p[0] = ids;
  r.period = 0;
  return r;
}

// Most-recent-K lookup of one (node, time) query by a full warp over the time-sorted CSR row of `node`
// (utils/utils.py:129-146): c = #entries with t < tq (strict, fp64) by a 32-ary search — each step the 32
// lanes probe 32 interior pivots and a ballot shrinks the range 33x — then the last take = min(K, c) entries
// are [first, first + take). All 32 lanes must call it with the same arguments.
__device__ __forceinline__ void warp_recent_range(const int64_t* __restrict__ indptr, const double* __restrict__ c_t, int64_t node,
                                                  double tq, int K, int lane, int64_t& first, int& take) {
  const int64_t lo = indptr[node];
  int64_t a = lo, b = indptr[node + 1];
  // invariant: entries < a are earlier than tq, entries >= b are not
  while (b - a > 32) {
    const int64_t len = b - a;
    const int64_t p = a + (len * (lane + 1)) / 33;
    const int j = __popc(__ballot_sync(kFull, c_t[p] < tq));
    const int64_t pa = a + (len * j) / 33, pb = a + (len * (j + 1)) / 33;
    if (j < 32) b = pb;
    if (j > 0) a = pa + 1;
  }
  const int64_t p = a + lane;
  const bool less = (p < b) && (c_t[p] < tq);
  const int64_t end = a + __popc(__ballot_sync(kFull, less));
  const int64_t cnt = end - lo;
  take = (int)(cnt < K ? cnt : K);
  first = end - take;
}

// Optional tail of the lookup kernel used by update_pe phase B: while a row's K neighbours are still in
// registers, count them per destination (integer atomics on the per-node map), record the arrival rank
// and the list of distinct destinations, flag padding; block 0 also zeroes pe[0] (LSTEP.py:317).
struct PhaseBHook {
  int32_t* cnt_of;
  int32_t* rank;
  int64_t* U;
  int32_t* counters;  // [0] = number of distinct destinations, [1] = any padded slot
  float* pe0;
  int d;
};

// TimeEncoder (models/modules.py:37): cos(fp32(dt) * w_j + 0). The product is a separately rounded fp32
// multiply (that is what Linear(1->t) computes), then an accurate cosine. Arguments reach 1e6..1e8 rad
// (dt in seconds times w_0 = 1), where cosf() takes its slow Payne-Hanek path (hundreds of instructions,
// divergent: only the low-frequency lanes need it) and where an fp64 reduction is no alternative (the
// scalar fp64 pipe of this part issues ~4 lanes/clk/SM: measured, it made one hub CTA the step's long
// pole). accurate_cos() does the Payne-Hanek reduction in 64-bit integer arithmetic instead: with
// |x| = m * 2^E (m the 24-bit significand), (x * 2/pi) mod 4 in 2.62 fixed point is m * W mod 2^64, where
// W is the 64-bit window of the bits of 2/pi that starts E+62 bits after the binary point (bits further
// left only contribute multiples of 4 quadrants). The top two bits are the quadrant, the rest the
// fraction of a quadrant (error < 2^-38), folded to [-1/2, 1/2), scaled by pi/2 and fed to the Cephes
// single-precision minimax polynomials: ~35 integer / fp32 instructions, absolute error <= 1.1e-7. (That general form
// now serves |x| >= 2^32 only; below it the window selection is replaced by two fixed multiplies, see accurate_cos.)
// (checked against libm on 15 000 arguments up to 2e9). Arguments below 2^14 — 72 % of the (dt, w_j)
// pairs, all of them for j >= 28 — take a 3-term Cody-Waite reduction in fp32 FMAs instead (6 instructions).
__device__ __forceinline__ float cos_poly(float rf, int q) {
  const float z = rf * rf;
  // sin(r) = r + r^3 * S(z),  cos(r) = 1 - z/2 + z^2 * C(z)   on |r| <= pi/4
  const float s = fmaf(rf * z, fmaf(fmaf(-1.9515295891e-4f, z, 8.3321608736e-3f), z, -1.6666654611e-1f), rf);
  const float c = fmaf(z * z, fmaf(fmaf(2.443315711809948e-5f, z, -1.388731625493765e-3f), z, 4.166664568298827e-2f),
                       fmaf(-0.5f, z, 1.0f));
  // cos(r + q*pi/2): q mod 4 = 0: c, 1: -s, 2: -c, 3: s
  const float v = (q & 1) ? s : c;
  return (((q + 1) & 2) ? -v : v);
}

__device__ __forceinline__ float accurate_cos(float x) {
  if (fabsf(x) < 16384.f) {
    const float k = rintf(x * 0.63661977236758134f);
    float r = fmaf(-k, 1.5703125f, x);                 // pi/2 = 1.5703125 + 4.837512969970703125e-4 + 7.549789954891882e-8 + ...
    r = fmaf(-k, 4.837512969970703125e-4f, r);
    r = fmaf(-k, 7.549789954891882e-8f, r);
    return cos_poly(r, (int)k);
  }
  const float ax = fabsf(x);
  if (ax < 4294967296.f) {
    // 2^14 <= |x| < 2^32 — every large argument a timestamp difference produces: |x| = xi + xf with xi an exact 32-bit
    // integer and xf an exact multiple of 2^-9 in [0, 1), so (|x| * 2/pi) mod 4 in 2.62 fixed point is
    // xi * C + (xf * 2^9) * (C >> 9) mod 2^64 with C = floor(2/pi * 2^62): two integer multiplies instead of selecting a
    // window of 2/pi by the exponent (error < 2^-30 of a quadrant). The top 32 bits of the folded fraction are all the
    // fp32 polynomial can use.
    const uint32_t xi = __float2uint_rz(ax);
    const uint32_t xfi = __float2uint_rz((ax - __uint2float_rn(xi)) * 512.f);
    const unsigned long long C = 0x28be60db9391054aull;
    const unsigned long long R = (unsigned long long)xi * C + (unsigned long long)xfi * (C >> 9);
    int q = (int)(R >> 62);
    long long f = (long long)(R & 0x3fffffffffffffffull);
    if (f >= (1ll << 61)) {
      f -= (1ll << 62);
      q += 1;
    }
    return cos_poly((float)(int)(f >> 30) * 3.6572951981678992e-10f /* (pi/2) * 2^-32 */, q);
  }
  const uint32_t bits = __float_as_uint(x);
  int e = (int)((bits >> 23) & 0xffu);
  if (e >= 214) return cosf(x);  // inf / nan / beyond the 128 stored bits of 2/pi (never a real timestamp)
  const uint32_t m = (bits & 0x7fffffu) | (e ? 0x800000u : 0u);
  e = e ? e : 1;
  const int sh = e - 88;  // E + 62 with E = e - 150
  const unsigned long long P_hi = 0xa2f9836e4e441529ull, P_lo = 0xfc2757d1f534ddc0ull;  // floor(2/pi * 2^128)
  unsigned long long W = 0ull;
  if (sh > 64)
    W = (P_hi << (sh - 64)) | (P_lo >> (128 - sh));
  else if (sh > 0)
    W = P_hi >> (64 - sh);
  const unsigned long long R = (unsigned long long)m * W;  // mod 2^64: 2 quadrant bits . 62 fraction bits
  int q = (int)(R >> 62);
  long long f = (long long)(R & 0x3fffffffffffffffull);
  if (f >= (1ll << 61)) {
    f -= (1ll << 62);
    q += 1;
  }
  return cos_poly((float)f * 3.4061215800865545e-19f /* (pi/2) * 2^-62 */, q);
}

__device__ __forceinline__ float time_feature(float dt, float w) { return accurate_cos(__fmul_rn(dt, w)); }

}  // namespace lstep
