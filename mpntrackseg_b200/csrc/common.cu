// Error reporting, device queries and a small device-wide exclusive scan.
#include <stdarg.h>
#include <string.h>

#include <atomic>
#include <mutex>
#include <vector>

#include "common.cuh"

namespace mpn {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

static std::atomic<long long> g_launches{0};
void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

struct ProfSpan { int kind; cudaEvent_t a, b; };
static bool g_prof = false;
static std::vector<ProfSpan> g_spans;
static std::mutex g_prof_mu;
bool profiling() { return g_prof; }
void profile_mark(int kind, bool begin, cudaStream_t s) {
  std::lock_guard<std::mutex> lk(g_prof_mu);
  if (begin) {
    ProfSpan sp; sp.kind = kind;
    cudaEventCreate(&sp.a); cudaEventCreate(&sp.b);
    cudaEventRecord(sp.a, s);
    g_spans.push_back(sp);
  } else if (!g_spans.empty()) {
    cudaEventRecord(g_spans.back().b, s);
  }
}

int sm_count() {
  // per device: one process may drive several GPUs (the cache is keyed by the current device)
  static int cached[64] = {0};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
  if (cached[dev] == 0) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) return 148;
    cached[dev] = n;
  }
  return cached[dev];
}

// ---------------------------------------------------------------- exclusive scan
// Three launches: per-chunk totals, scan of the totals by one CTA, per-chunk scan + offset.
constexpr int kScanThreads = 256;
constexpr int kScanItems = 8;                       // per thread
constexpr int kScanChunk = kScanThreads * kScanItems;

template <typename T>
__global__ void scan_chunk_totals(const T* __restrict__ in, T* __restrict__ totals, int64_t n) {
  __shared__ T sm[32];
  __shared__ T tot;
  const int64_t base = (int64_t)blockIdx.x * kScanChunk + (int64_t)threadIdx.x * kScanItems;
  T s = 0;
#pragma unroll
  for (int i = 0; i < kScanItems; ++i)
    if (base + i < n) s += in[base + i];
  block_exclusive_scan<T>(s, sm, &tot);
  if (threadIdx.x == 0) totals[blockIdx.x] = tot;
}

template <typename T>
__global__ void scan_totals_inplace(T* __restrict__ totals, int64_t m, T* __restrict__ grand) {
  __shared__ T sm[32];
  __shared__ T tot;
  T carry = 0;
  for (int64_t s = 0; s < m; s += blockDim.x) {
    int64_t i = s + threadIdx.x;
    T v = i < m ? totals[i] : T(0);
    T ex = block_exclusive_scan<T>(v, sm, &tot);
    if (i < m) totals[i] = carry + ex;
    carry += tot;
    __syncthreads();
  }
  if (threadIdx.x == 0) *grand = carry;
}

template <typename T>
__global__ void scan_chunks(const T* __restrict__ in, T* __restrict__ out,
                            const T* __restrict__ offsets, int64_t n) {
  __shared__ T sm[32];
  __shared__ T tot;
  const int64_t base = (int64_t)blockIdx.x * kScanChunk + (int64_t)threadIdx.x * kScanItems;
  T v[kScanItems];
  T s = 0;
#pragma unroll
  for (int i = 0; i < kScanItems; ++i) {
    v[i] = base + i < n ? in[base + i] : T(0);
    s += v[i];
  }
  T ex = block_exclusive_scan<T>(s, sm, &tot) + offsets[blockIdx.x];
#pragma unroll
  for (int i = 0; i < kScanItems; ++i) {
    if (base + i < n) out[base + i] = ex;
    ex += v[i];
  }
}

template <typename T>
static int exclusive_scan_impl(const T* in, T* out, int64_t n, cudaStream_t stream) {
  if (n <= 0) {
    MPN_CUDA(cudaMemsetAsync(out, 0, sizeof(T), stream));
    return MPN_OK;
  }
  const int64_t chunks = ceil_div(n, kScanChunk);
  {
    // keep the stream-ordered pool's memory across synchronisations (default threshold 0 would hand it
    // back to the OS at every sync and re-allocate on the next call)
    static bool pool_ready = false;
    if (!pool_ready) {
      int dev = 0;
      cudaMemPool_t pool;
      if (cudaGetDevice(&dev) == cudaSuccess && cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) {
        unsigned long long keep = ~0ull;
        cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
      }
      pool_ready = true;
    }
  }
  T* totals = nullptr;
  MPN_CUDA(cudaMallocAsync(&totals, sizeof(T) * (chunks + 1), stream));
  scan_chunk_totals<T><<<(unsigned)chunks, kScanThreads, 0, stream>>>(in, totals, n); count_launch();
  scan_totals_inplace<T><<<1, 1024, 0, stream>>>(totals, chunks, out + n); count_launch();
  scan_chunks<T><<<(unsigned)chunks, kScanThreads, 0, stream>>>(in, out, totals, n); count_launch();
  MPN_LAUNCH_CHECK();
  MPN_CUDA(cudaFreeAsync(totals, stream));
  return MPN_OK;
}

int exclusive_scan_i64(const int64_t* in, int64_t* out, int64_t n, cudaStream_t stream) {
  return exclusive_scan_impl<int64_t>(in, out, n, stream);
}
int exclusive_scan_i32(const int32_t* in, int32_t* out, int64_t n, cudaStream_t stream) {
  return exclusive_scan_impl<int32_t>(in, out, n, stream);
}

}  // namespace mpn

extern "C" {

const char* mpn_last_error(void) { return mpn::g_err; }

int mpn_abi_version(void) { return 4; }

long long mpn_launch_count(void) { return mpn::g_launches.load(); }

int mpn_profile_begin(void) {
  std::lock_guard<std::mutex> lk(mpn::g_prof_mu);
  for (auto& sp : mpn::g_spans) { cudaEventDestroy(sp.a); cudaEventDestroy(sp.b); }
  mpn::g_spans.clear();
  mpn::g_prof = true;
  return MPN_OK;
}

int mpn_profile_end(double* h_ms /*[2]*/, long long* h_launches /*[2]*/) {
  MPN_CUDA(cudaDeviceSynchronize());
  std::lock_guard<std::mutex> lk(mpn::g_prof_mu);
  mpn::g_prof = false;
  double ms[2] = {0, 0};
  long long cnt[2] = {0, 0};
  for (auto& sp : mpn::g_spans) {
    float t = 0.f;
    if (cudaEventElapsedTime(&t, sp.a, sp.b) == cudaSuccess && sp.kind >= 0 && sp.kind < 2) {
      ms[sp.kind] += t;
      cnt[sp.kind] += 1;
    }
    cudaEventDestroy(sp.a); cudaEventDestroy(sp.b);
  }
  mpn::g_spans.clear();
  if (h_ms) { h_ms[0] = ms[0]; h_ms[1] = ms[1]; }
  if (h_launches) { h_launches[0] = cnt[0]; h_launches[1] = cnt[1]; }
  return MPN_OK;
}

int mpn_device_arch(void) {
  int dev = 0;
  MPN_CUDA(cudaGetDevice(&dev));
  int major = 0, minor = 0;
  MPN_CUDA(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
  MPN_CUDA(cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, dev));
  return major * 10 + minor;
}

}  // extern "C"
