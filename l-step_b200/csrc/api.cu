// Status / error plumbing of the C ABI (include/lstep_b200.h).
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "common.cuh"

namespace lstep {

static thread_local char g_cuda_err[256] = "";

void set_cuda_error(cudaError_t e, const char* where) {
  snprintf(g_cuda_err, sizeof(g_cuda_err), "%s: %s", where, cudaGetErrorString(e));
}

int num_sms() {
  static int n = 0;
  if (n == 0) {
    int dev = 0, v = 0;
    if (cudaGetDevice(&dev) == cudaSuccess && cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && v > 0)
      n = v;
    else
      return 148;  // B200; not cached: the next call asks again
  }
  return n;
}

namespace {
struct OptName {
  const char* name;
  int Tuning::*field;
  const char* env;   // environment variable read once at first use
  int env_value;     // value the field takes when the variable is set (-1: atoi of the variable)
};
const OptName kOpts[] = {
    {"pdl", &Tuning::pdl, "LSTEP_NO_PDL", 0},
    {"phaseb_push", &Tuning::phaseb_push, "LSTEP_PHASEB_PULL", 0},
    {"gather_pipe", &Tuning::gather_pipe, "LSTEP_NO_GATHER_PIPE", 0},
    {"mlp_umma", &Tuning::mlp_umma, "LSTEP_NO_MLP_UMMA", 0},
    {"mlp_umma_min_rows", &Tuning::mlp_umma_min_rows, "LSTEP_MLP_UMMA_MIN_ROWS", -1},
    {"profile", &Tuning::profile, nullptr, 0},
};
}  // namespace

namespace {
cudaEvent_t g_prof_ev[kProfSlots];
bool g_prof_have = false;
unsigned g_prof_seen = 0;  // slots recorded since the last read
}  // namespace

void prof_mark(cudaStream_t st, int slot) {
  if (!tuning().profile) return;
  if (!g_prof_have) {
    for (int i = 0; i < kProfSlots; ++i)
      if (cudaEventCreate(&g_prof_ev[i]) != cudaSuccess) return;
    g_prof_have = true;
  }
  if (slot == kProfStart) g_prof_seen = 0;
  if (cudaEventRecord(g_prof_ev[slot], st) == cudaSuccess) g_prof_seen |= 1u << slot;
}

Tuning& tuning() {
  static Tuning t = [] {
    Tuning v;
    for (const OptName& o : kOpts) {
      const char* e = o.env ? getenv(o.env) : nullptr;
      if (e) v.*(o.field) = o.env_value >= 0 ? o.env_value : atoi(e);
    }
    return v;
  }();
  return t;
}

int check_launch(const char* where) {
  const cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) return LSTEP_OK;
  set_cuda_error(e, where);
  return LSTEP_ERR_CUDA;
}

}  // namespace lstep

extern "C" const char* lstep_strerror(int status) {
  switch (status) {
    case LSTEP_OK: return "ok";
    case LSTEP_ERR_INVALID_ARG: return "invalid argument";
    case LSTEP_ERR_UNSUPPORTED: return "shape not supported by the sm_100a kernels";
    case LSTEP_ERR_WORKSPACE: return "workspace too small";
    case LSTEP_ERR_CUDA: return "CUDA runtime error";
    case LSTEP_ERR_ID_RANGE: return "id does not fit the int32 device encoding";
    default: return "unknown status";
  }
}

extern "C" const char* lstep_last_cuda_error(void) { return lstep::g_cuda_err; }

extern "C" int lstep_abi_version(void) { return LSTEP_ABI_VERSION; }

extern "C" int lstep_device_ok(void) {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 0;
  cudaDeviceProp p;
  if (cudaGetDeviceProperties(&p, dev) != cudaSuccess) return 0;
  return p.major == 10 ? 1 : 0;
}

extern "C" int lstep_set_option(const char* name, int value) {
  if (!name) return LSTEP_ERR_INVALID_ARG;
  for (const lstep::OptName& o : lstep::kOpts)
    if (strcmp(o.name, name) == 0) {
      lstep::tuning().*(o.field) = value;
      return LSTEP_OK;
    }
  return LSTEP_ERR_INVALID_ARG;
}

extern "C" int lstep_get_option(const char* name, int* value) {
  if (!name || !value) return LSTEP_ERR_INVALID_ARG;
  for (const lstep::OptName& o : lstep::kOpts)
    if (strcmp(o.name, name) == 0) {
      *value = lstep::tuning().*(o.field);
      return LSTEP_OK;
    }
  return LSTEP_ERR_INVALID_ARG;
}

extern "C" int lstep_step_profile(int enable) {
  lstep::tuning().profile = enable ? 1 : 0;
  return LSTEP_OK;
}

/* ms[i - 1] = time between the previous recorded mark and mark i of the LAST profiled step, for every slot of ProfSlot
 * (csrc/common.cuh): 0 DFT filter, 1 wait on barrier 1 (peer group), 2 fused gather, 3 paired MLP, 4 phase-A row broadcast (peer
 * group), 5 wait on barrier 2 (peer group), 6 phase-B push, 7 phase-B MLP, 8 append; -1 where no mark was recorded. */
extern "C" int lstep_step_profile_read_all(float* ms, int n) {
  using namespace lstep;
  if (!ms || n < kProfSlots - 1) return LSTEP_ERR_INVALID_ARG;
  for (int i = 0; i < n; ++i) ms[i] = -1.f;
  if (!g_prof_have || !(g_prof_seen & 1u)) return LSTEP_ERR_INVALID_ARG;
  int last = 0;
  for (int i = 1; i < kProfSlots; ++i)
    if (g_prof_seen & (1u << i)) last = i;
  if (cudaEventSynchronize(g_prof_ev[last]) != cudaSuccess) return LSTEP_ERR_CUDA;
  int prev = 0;
  for (int i = 1; i < kProfSlots; ++i) {
    if (!(g_prof_seen & (1u << i))) continue;
    float v = 0.f;
    if (cudaEventElapsedTime(&v, g_prof_ev[prev], g_prof_ev[i]) != cudaSuccess) return LSTEP_ERR_CUDA;
    ms[i - 1] = v;
    prev = i;
  }
  return LSTEP_OK;
}

/* ms6[i] = duration of kernel i of the LAST profiled step: 0 DFT filter, 1 fused gather, 2 paired MLP, 3 phase-B push,
 * 4 phase-B MLP, 5 ring append; -1 where that kernel was not launched. Synchronises on the step's last event. */
extern "C" int lstep_step_profile_read(float* ms6) {
  using namespace lstep;
  if (!ms6) return LSTEP_ERR_INVALID_ARG;
  float all[kProfSlots];
  const int rc = lstep_step_profile_read_all(all, kProfSlots);
  static const int pick[6] = {kProfDft, kProfGather, kProfMlpPair, kProfPush, kProfMlpB, kProfAppend};
  for (int i = 0; i < 6; ++i) ms6[i] = rc == LSTEP_OK ? all[pick[i] - 1] : -1.f;
  return rc;
}
