// Error reporting, launch accounting, driver entry points and boundary layout helpers of libmvsf_b200.
#include <stdarg.h>
#include <string.h>

#include <mutex>
#include <string>
#include <utility>
#include <vector>

#include "common.cuh"
#include "umma.cuh"

namespace mvsf {
static thread_local char g_err[1024] = "";
static thread_local long long g_launches = 0;

int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}
void count_launch(int n) { g_launches += n; }

int current_device() {
  int d = 0;
  if (cudaGetDevice(&d) != cudaSuccess || d < 0) d = 0;
  return d;
}
int device_sm_count(int dev) {
  static std::atomic<int> cache[64];
  const int slot = dev & 63;
  int v = cache[slot].load(std::memory_order_relaxed);
  if (v <= 0) {
    if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || v <= 0) v = 148;
    cache[slot].store(v, std::memory_order_relaxed);
  }
  return v;
}

// Opt-in per-kernel device timers (CUDA events on the launching stream around selected launches): bench.py needs the
// duration of single kernels that are launched from inside a multi-kernel entry point.
struct KTimer { std::string name; std::vector<std::pair<cudaEvent_t, cudaEvent_t>> ev; };
static std::atomic<bool> g_ktimer_on{false};
static std::vector<KTimer> g_ktimers;
static std::mutex g_ktimer_mu;   // the timers are process-global; calls may come from several host threads
bool ktimer_enabled() { return g_ktimer_on.load(std::memory_order_relaxed); }
cudaEvent_t ktimer_begin(const char* name, cudaStream_t s) {
  std::lock_guard<std::mutex> lk(g_ktimer_mu);
  KTimer* t = nullptr;
  for (auto& k : g_ktimers)
    if (k.name == name) t = &k;
  if (!t) { g_ktimers.push_back(KTimer{name, {}}); t = &g_ktimers.back(); }
  cudaEvent_t a = nullptr, b = nullptr;
  cudaEventCreate(&a);
  cudaEventCreate(&b);
  t->ev.push_back({a, b});
  cudaEventRecord(a, s);
  return b;
}
void ktimer_end(cudaEvent_t e, cudaStream_t s) { cudaEventRecord(e, s); }

umma::EncodeTiledFn umma::encode_tiled_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

// [N][C][HW] -> [N][HW][C] through a 32x32 shared-memory tile (coalesced on both sides)
__global__ void transpose_chw_hwc_kernel(const float* __restrict__ src, float* __restrict__ dst, int C, int HW) {
  __shared__ float tile[32][33];
  const int n = blockIdx.z;
  const float* s = src + (size_t)n * C * HW;
  float* d = dst + (size_t)n * C * HW;
  int p0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    int c = c0 + i, p = p0 + threadIdx.x;
    if (c < C && p < HW) tile[i][threadIdx.x] = s[(size_t)c * HW + p];
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    int p = p0 + i, c = c0 + threadIdx.x;
    if (c < C && p < HW) d[(size_t)p * C + c] = tile[threadIdx.x][i];
  }
}
// [N][HW][C] -> [N][C][HW]
__global__ void transpose_hwc_chw_kernel(const float* __restrict__ src, float* __restrict__ dst, int C, int HW) {
  __shared__ float tile[32][33];
  const int n = blockIdx.z;
  const float* s = src + (size_t)n * C * HW;
  float* d = dst + (size_t)n * C * HW;
  int p0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    int p = p0 + i, c = c0 + threadIdx.x;
    if (c < C && p < HW) tile[i][threadIdx.x] = s[(size_t)p * C + c];
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    int c = c0 + i, p = p0 + threadIdx.x;
    if (c < C && p < HW) d[(size_t)c * HW + p] = tile[threadIdx.x][i];
  }
}
}  // namespace mvsf

extern "C" {

const char* mvsf_last_error(void) { return mvsf::g_err; }
int mvsf_abi_version(void) { return 1; }
long long mvsf_launch_count(int reset) {
  long long v = mvsf::g_launches;
  if (reset) mvsf::g_launches = 0;
  return v;
}

int mvsf_ktimer_enable(int on) {
  mvsf::g_ktimer_on.store(on != 0);
  return MVSF_OK;
}
/* device milliseconds and launches recorded under `name` since the last read (synchronises the device, then resets) */
int mvsf_ktimer_read(const char* name, double* ms, long long* launches) {
  MVSF_REQUIRE(name && ms && launches, "ktimer_read: null pointer");
  *ms = 0.0;
  *launches = 0;
  std::lock_guard<std::mutex> lk(mvsf::g_ktimer_mu);
  for (auto& k : mvsf::g_ktimers) {
    if (k.name != name) continue;
    for (auto& pr : k.ev) {
      float t = 0.f;
      MVSF_CUDA_OK(cudaEventSynchronize(pr.second));
      MVSF_CUDA_OK(cudaEventElapsedTime(&t, pr.first, pr.second));
      *ms += t;
      *launches += 1;
      cudaEventDestroy(pr.first);
      cudaEventDestroy(pr.second);
    }
    k.ev.clear();
  }
  return MVSF_OK;
}

int mvsf_nchw_to_nhwc(const float* src, float* dst, int N, int C, int HW, mvsf_stream_t stream) {
  MVSF_REQUIRE(src && dst && N > 0 && C > 0 && HW > 0 && N <= 65535, "nchw_to_nhwc: bad arguments");
  dim3 grid(mvsf::cdiv(HW, 32), mvsf::cdiv(C, 32), N), block(32, 8);
  mvsf::transpose_chw_hwc_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(src, dst, C, HW);
  MVSF_LAUNCH_CHECK("nchw_to_nhwc");
  return MVSF_OK;
}
int mvsf_nhwc_to_nchw(const float* src, float* dst, int N, int C, int HW, mvsf_stream_t stream) {
  MVSF_REQUIRE(src && dst && N > 0 && C > 0 && HW > 0 && N <= 65535, "nhwc_to_nchw: bad arguments");
  dim3 grid(mvsf::cdiv(HW, 32), mvsf::cdiv(C, 32), N), block(32, 8);
  mvsf::transpose_hwc_chw_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(src, dst, C, HW);
  MVSF_LAUNCH_CHECK("nhwc_to_nchw");
  return MVSF_OK;
}
}
