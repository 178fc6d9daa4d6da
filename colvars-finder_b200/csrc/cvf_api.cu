// cvf_api.cu -- version, error reporting and device queries of libcvf_sm100.so.
#include <stdarg.h>

#include <atomic>
#include <mutex>

#include "cvf_common.cuh"

namespace cvf {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int check_cuda(cudaError_t e, const char* what) {
  if (e == cudaSuccess) return 0;
  set_error("%s: %s", what, cudaGetErrorString(e));
  return (int)e;
}

static int g_sms[64];
static int g_smem[64];

static int device_attr(int* cache, cudaDeviceAttr attr, int fallback) {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return fallback;
  if (cache[dev] == 0) {
    int v = 0;
    if (cudaDeviceGetAttribute(&v, attr, dev) != cudaSuccess || v <= 0) return fallback;
    cache[dev] = v;
  }
  return cache[dev];
}

// ---- launch accounting -------------------------------------------------------------------------------------
static const char* const g_kernel_names[K_COUNT] = {
    "align_fwd", "features_fwd", "eigen_stats(general)", "eigen_grad(general)", "eigen_combine", "reduce_partials", "ae_step",
    "fast_pack", "fast_prep", "fast_pass1", "fast_stats", "fast_pass2", "(unused)", "fma_probe", "fast_jjt", "ae_fast_prep", "ae_fast_main", "ae_fast_dw", "weights_filter",
    "align_vjp", "features_vjp"};
static std::atomic<long long> g_launches[K_COUNT];
static std::atomic<int> g_prof_on{0};
static std::mutex g_prof_mutex;   // guards g_recs / g_n_recs (timed launches are a profiling mode, not the hot path)
struct ProfRec {
  int id;
  cudaEvent_t e0, e1;
};
static ProfRec g_recs[4096];
static int g_n_recs = 0;

void prof_begin(int id, cudaStream_t stream) {
  g_launches[id].fetch_add(1, std::memory_order_relaxed);
  if (!g_prof_on.load(std::memory_order_relaxed)) return;
  std::lock_guard<std::mutex> lock(g_prof_mutex);
  if (g_n_recs >= 4096) return;
  ProfRec& r = g_recs[g_n_recs];
  r.id = id;
  if (cudaEventCreate(&r.e0) != cudaSuccess || cudaEventCreate(&r.e1) != cudaSuccess) return;
  cudaEventRecord(r.e0, stream);
}
void prof_end(int id, cudaStream_t stream) {
  if (!g_prof_on.load(std::memory_order_relaxed)) return;
  std::lock_guard<std::mutex> lock(g_prof_mutex);
  if (g_n_recs >= 4096 || g_recs[g_n_recs].id != id) return;
  cudaEventRecord(g_recs[g_n_recs].e1, stream);
  ++g_n_recs;
}

int sm_count() { return device_attr(g_sms, cudaDevAttrMultiProcessorCount, 148); }
int max_smem_optin() { return device_attr(g_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, 232448); }

}  // namespace cvf

extern "C" int cvf_version(void) { return CVF_VERSION; }

#ifndef CVF_SOURCE_HASH
#define CVF_SOURCE_HASH "unstamped"
#endif
static const char g_source_stamp[] = "CVF_SOURCE_HASH=" CVF_SOURCE_HASH;
extern "C" const char* cvf_source_hash(void) { return g_source_stamp + 16; }

extern "C" int cvf_profile_enable(int32_t on) {
  cvf::g_prof_on.store(on ? 1 : 0);
  return 0;
}
extern "C" int32_t cvf_profile_num_kernels(void) { return cvf::K_COUNT; }
extern "C" const char* cvf_profile_kernel_name(int32_t id) { return id >= 0 && id < cvf::K_COUNT ? cvf::g_kernel_names[id] : ""; }
extern "C" int cvf_profile_read(double* ms_out, int64_t* timed_out, int64_t* launches_out, int32_t reset) {
  using namespace cvf;
  if (!ms_out || !timed_out || !launches_out) {
    set_error("cvf_profile_read: null pointer");
    return CVF_E_ARG;
  }
  std::lock_guard<std::mutex> lock(g_prof_mutex);
  for (int i = 0; i < K_COUNT; ++i) ms_out[i] = 0.0, timed_out[i] = 0, launches_out[i] = g_launches[i].load();
  for (int i = 0; i < g_n_recs; ++i) {
    float ms = 0.f;
    if (cudaEventSynchronize(g_recs[i].e1) == cudaSuccess && cudaEventElapsedTime(&ms, g_recs[i].e0, g_recs[i].e1) == cudaSuccess) {
      ms_out[g_recs[i].id] += ms;
      ++timed_out[g_recs[i].id];
    }
    cudaEventDestroy(g_recs[i].e0);
    cudaEventDestroy(g_recs[i].e1);
  }
  g_n_recs = 0;
  if (reset)
    for (int i = 0; i < K_COUNT; ++i) g_launches[i].store(0);
  return 0;
}
extern "C" const char* cvf_last_error_string(void) { return cvf::g_err; }

extern "C" int64_t cvf_mlp_param_count(const cvf_mlp* net) {
  cvf::NetPlan np;
  if (cvf::make_net_plan(net, &np)) return -1;
  return np.n_params;
}

// ---- fp32 FMA probe ------------------------------------------------------------------------------------
namespace cvf {
__global__ void __launch_bounds__(256) fma_probe_kernel(float* sink, int iters) {
  float a[16];
  const float x = 1.0f + 1e-7f * threadIdx.x, y = 1e-9f * blockIdx.x;
#pragma unroll
  for (int i = 0; i < 16; ++i) a[i] = (float)i;
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int i = 0; i < 16; ++i) a[i] = fmaf(a[i], x, y);
  }
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < 16; ++i) s += a[i];
  if (s == 12345.678f) sink[0] = s;   // never true: keeps the chains alive
}
}  // namespace cvf

extern "C" int cvf_fma_probe(float* sink, int32_t iters, double* flops_out, void* stream) {
  if (!sink || iters < 1 || !flops_out) {
    cvf::set_error("cvf_fma_probe: bad argument");
    return CVF_E_ARG;
  }
  const int grid = cvf::sm_count() * 8;
  CVF_LAUNCH(cvf::K_FMA_PROBE, (cudaStream_t)stream, cvf::fma_probe_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(sink, iters));
  *flops_out = 2.0 * 16.0 * (double)iters * 256.0 * (double)grid;
  CVF_CUDA(cudaGetLastError());
  return 0;
}
extern "C" size_t cvf_sizeof_preproc(void) { return sizeof(cvf_preproc); }
extern "C" size_t cvf_sizeof_mlp(void) { return sizeof(cvf_mlp); }
