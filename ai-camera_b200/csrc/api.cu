// Error state, version and launch accounting shared by every entry point of the C ABI.
#include <atomic>
#include <map>
#include <mutex>
#include <utility>
#include <vector>

#include "common.cuh"

namespace aicam {

static thread_local std::string g_error;
static std::atomic<uint64_t> g_launches{0};

void set_error(const std::string& msg) { g_error = msg; }
int fail(int code, const std::string& msg) {
  g_error = msg;
  return code;
}
void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }

static std::mutex g_attr_mutex;
static std::map<std::pair<int, const void*>, size_t> g_smem_limit;  // (device, kernel) -> bytes opted in to
static std::map<int, int> g_num_sms;

int ensure_dynamic_smem(const void* kernel, size_t bytes) {
  int dev = 0;
  AICAM_CUDA_OK(cudaGetDevice(&dev));
  std::lock_guard<std::mutex> lock(g_attr_mutex);
  size_t& have = g_smem_limit[std::make_pair(dev, kernel)];
  if (bytes > have) {
    if (bytes > 48 * 1024)
      AICAM_CUDA_OK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(bytes)));
    have = bytes;
  }
  return AICAM_OK;
}

int current_num_sms() {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 0;
  std::lock_guard<std::mutex> lock(g_attr_mutex);
  auto it = g_num_sms.find(dev);
  if (it != g_num_sms.end()) return it->second;
  int n = 0;
  if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return 0;
  g_num_sms[dev] = n;
  return n;
}

// ---- per-launch event timing of the convolution kernel ------------------------------------
static bool g_profile = false;
static std::vector<std::pair<cudaEvent_t, cudaEvent_t>> g_events;
static size_t g_events_used = 0;

bool profile_begin(cudaStream_t st, size_t* slot) {
  if (!g_profile) return false;
  if (g_events_used == g_events.size()) {
    cudaEvent_t a, b;
    if (cudaEventCreate(&a) != cudaSuccess || cudaEventCreate(&b) != cudaSuccess) return false;
    g_events.emplace_back(a, b);
  }
  *slot = g_events_used++;
  cudaEventRecord(g_events[*slot].first, st);
  return true;
}

// Step timeline (debug): while enabled, every conv_win launch is handed the next 4-slot record of a device buffer and
// its CTA 0 stamps %globaltimer there at entry, when its dependency on the previous kernel has resolved, and at exit;
// slot 3 holds a host-written tag (cout, cin, height).  A CUDA-graph capture made while the timeline is on keeps the
// records, so replays give the IN-GRAPH timing of every layer (aicam_debug_timeline).
static long long* g_tl_dev = nullptr;
static int g_tl_cap = 0, g_tl_next = 0;
static std::vector<long long> g_tl_tags;
long long* timeline_slot(long long tag) {
  if (!g_tl_dev || g_tl_next >= g_tl_cap) return nullptr;
  g_tl_tags.push_back(tag);
  return g_tl_dev + 4 * static_cast<size_t>(g_tl_next++);
}
void profile_end(cudaStream_t st, size_t slot) { cudaEventRecord(g_events[slot].second, st); }

}  // namespace aicam

extern "C" {

int aicam_version(void) { return 100; }
const char* aicam_last_error(void) { return aicam::g_error.c_str(); }
uint64_t aicam_launch_count(void) { return aicam::g_launches.load(); }

int aicam_debug_timeline(int op, long long* host_out, int capacity) {
  // op 1: start (allocate `capacity` records, restart numbering), op 2: copy the records to host_out ([n][4]: entry ns,
  // dependency-resolved ns, exit ns, tag), returns their number; op 0: stop and free
  using namespace aicam;
  if (op == 1) {
    if (g_tl_dev) cudaFree(g_tl_dev);
    g_tl_dev = nullptr; g_tl_next = 0; g_tl_tags.clear();
    if (capacity <= 0 || cudaMalloc(&g_tl_dev, sizeof(long long) * 4 * capacity) != cudaSuccess) return fail(AICAM_ERR_CUDA, "debug_timeline: allocation failed");
    cudaMemset(g_tl_dev, 0, sizeof(long long) * 4 * capacity);
    g_tl_cap = capacity;
    return AICAM_OK;
  }
  if (op == 2) {
    if (!g_tl_dev || !host_out) return fail(AICAM_ERR_INVALID_ARG, "debug_timeline: not started");
    const int n = std::min(g_tl_next, capacity);
    if (cudaDeviceSynchronize() != cudaSuccess ||
        cudaMemcpy(host_out, g_tl_dev, sizeof(long long) * 4 * n, cudaMemcpyDeviceToHost) != cudaSuccess)
      return fail(AICAM_ERR_CUDA, "debug_timeline: copy failed");
    for (int i = 0; i < n; ++i) host_out[4 * i + 3] = g_tl_tags[i];
    return n;
  }
  if (g_tl_dev) cudaFree(g_tl_dev);
  g_tl_dev = nullptr; g_tl_cap = 0; g_tl_next = 0; g_tl_tags.clear();
  return AICAM_OK;
}

int aicam_profile_enable(int on) {
  aicam::g_profile = on != 0;
  return AICAM_OK;
}

int aicam_profile_conv(double* total_ms, uint64_t* launches) {
  if (!total_ms || !launches) return aicam::fail(AICAM_ERR_INVALID_ARG, "profile_conv: null argument");
  cudaError_t e = cudaDeviceSynchronize();
  if (e != cudaSuccess) return aicam::fail(AICAM_ERR_CUDA, std::string("profile_conv: ") + cudaGetErrorString(e));
  double sum = 0.0;
  for (size_t i = 0; i < aicam::g_events_used; ++i) {
    float ms = 0.0f;
    cudaEventElapsedTime(&ms, aicam::g_events[i].first, aicam::g_events[i].second);
    sum += ms;
  }
  *total_ms = sum;
  *launches = aicam::g_events_used;
  aicam::g_events_used = 0;
  return AICAM_OK;
}

}  // extern "C"
