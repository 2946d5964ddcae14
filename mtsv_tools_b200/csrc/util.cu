// util.cu — error plumbing, device selection, memory allocation and the exclusive-scan primitive used between stages.
#include <stdio.h>

#include "ctx.h"

namespace mtsv {

static thread_local std::string g_last_error;
std::atomic<uint64_t> g_launches{0};

int set_error(int code, const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  g_last_error = buf;
  return code;
}

const char* last_error_cstr() { return g_last_error.c_str(); }

// SMs of the current device (grids of the worklist-driven kernels are sized in multiples of it); the attribute
// query is a driver call, so it is made once per device
unsigned sm_count() {
  static std::atomic<int> cached[64];
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
  int n = cached[dev].load(std::memory_order_relaxed);
  if (n == 0) {
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) {
      (void)cudaGetLastError();
      n = 148;
    }
    cached[dev].store(n, std::memory_order_relaxed);
  }
  return (unsigned)n;
}

void CudaFree::operator()(void* p) const { cudaFree(p); }
void CudaFreeHost::operator()(void* p) const { cudaFreeHost(p); }

int device_alloc(void** p, size_t bytes) {
  const cudaError_t e = cudaMalloc(p, bytes);
  if (e == cudaSuccess) return 0;
  (void)cudaGetLastError();
  *p = nullptr;
  return set_error(MTSVGPU_ENOMEM, "cudaMalloc(%zu bytes) failed: %s", bytes, cudaGetErrorString(e));
}

int pinned_alloc(void** p, size_t bytes, unsigned flags) {
  const cudaError_t e = cudaHostAlloc(p, bytes, flags);
  if (e == cudaSuccess) return 0;
  (void)cudaGetLastError();
  *p = nullptr;
  return set_error(MTSVGPU_ENOMEM, "cudaHostAlloc(%zu bytes) failed: %s", bytes, cudaGetErrorString(e));
}

int use_device(int device) {
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    (void)cudaGetLastError();
    return set_error(MTSVGPU_ENODEVICE, "no CUDA device available (this library has no CPU path)");
  }
  if (device < 0 || device >= ndev) return set_error(MTSVGPU_EINVAL, "device %d out of range", device);
  MTSV_CUDA_TRY(cudaSetDevice(device));
  return 0;
}

int DevBuf::reserve(size_t bytes) {
  if (bytes <= cap && p) return 0;
  p.reset();
  cap = 0;
  size_t want = bytes + bytes / 4 + 256;  // headroom so slowly growing batches do not realloc
  if (dev_alloc(p, want) != 0) {
    want = bytes ? bytes : 256;
    MTSV_TRY(dev_alloc(p, want));
  }
  cap = want;
  return 0;
}

// ---------------------------------------------------------------------------------------------
// exclusive scan of u32 -> u32 (n+1 outputs, out[n] = total), u64 total for overflow detection
// ---------------------------------------------------------------------------------------------
constexpr int kScanThreads = 256;
constexpr int kScanItems = 8;
constexpr int kScanTile = kScanThreads * kScanItems;

__device__ __forceinline__ uint64_t warp_inclusive_u64(uint64_t v) {
  const unsigned lane = threadIdx.x & 31;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    uint64_t o = __shfl_up_sync(0xffffffffu, v, d);
    if (lane >= (unsigned)d) v += o;
  }
  return v;
}

// exclusive prefix of `v` across the block; *total gets the block sum (valid in every thread)
__device__ __forceinline__ uint64_t block_exclusive_u64(uint64_t v, uint64_t* total) {
  __shared__ uint64_t warp_sums[32];
  const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = (blockDim.x + 31) >> 5;
  uint64_t inc = warp_inclusive_u64(v);
  if (lane == 31) warp_sums[warp] = inc;
  __syncthreads();
  if (warp == 0) {
    uint64_t w = lane < nwarps ? warp_sums[lane] : 0;
    uint64_t winc = warp_inclusive_u64(w);
    warp_sums[lane] = winc;  // inclusive over warps
  }
  __syncthreads();
  uint64_t base = warp ? warp_sums[warp - 1] : 0;
  *total = warp_sums[nwarps - 1];
  uint64_t r = base + inc - v;
  __syncthreads();
  return r;
}

__global__ void __launch_bounds__(kScanThreads) scan_tile_sums(const uint32_t* __restrict__ in,
                                                               uint64_t n,
                                                               uint64_t* __restrict__ sums) {
  uint64_t base = (uint64_t)blockIdx.x * kScanTile + (uint64_t)threadIdx.x * kScanItems;
  uint64_t s = 0;
#pragma unroll
  for (int i = 0; i < kScanItems; ++i)
    if (base + i < n) s += in[base + i];
  uint64_t total;
  block_exclusive_u64(s, &total);
  if (threadIdx.x == 0) sums[blockIdx.x] = total;
}

__global__ void __launch_bounds__(1024) scan_sums_inplace(uint64_t* __restrict__ sums, uint32_t nb,
                                                          uint64_t* __restrict__ total_out) {
  uint64_t carry = 0;
  for (uint32_t base = 0; base < nb; base += blockDim.x) {
    uint32_t i = base + threadIdx.x;
    uint64_t v = i < nb ? sums[i] : 0;
    uint64_t total;
    uint64_t ex = block_exclusive_u64(v, &total);
    if (i < nb) sums[i] = carry + ex;
    carry += total;
  }
  if (threadIdx.x == 0 && total_out) *total_out = carry;
}

__global__ void __launch_bounds__(kScanThreads) scan_apply(const uint32_t* __restrict__ in,
                                                           uint32_t* __restrict__ out, uint64_t n,
                                                           const uint64_t* __restrict__ sums) {
  uint64_t base = (uint64_t)blockIdx.x * kScanTile + (uint64_t)threadIdx.x * kScanItems;
  uint32_t v[kScanItems];
  uint64_t s = 0;
#pragma unroll
  for (int i = 0; i < kScanItems; ++i) {
    v[i] = base + i < n ? in[base + i] : 0;
    s += v[i];
  }
  uint64_t total;
  uint64_t ex = block_exclusive_u64(s, &total) + sums[blockIdx.x];
#pragma unroll
  for (int i = 0; i < kScanItems; ++i) {
    if (base + i < n) out[base + i] = (uint32_t)ex;
    ex += v[i];
    if (base + i + 1 == n) out[n] = (uint32_t)ex;
  }
}

__global__ void scan_empty(uint32_t* out, uint64_t* total_out) {
  out[0] = 0;
  if (total_out) *total_out = 0;
}

int exclusive_scan_u32(const uint32_t* d_in, uint32_t* d_out, uint64_t n, DevBuf& tmp,
                       uint64_t* d_total, cudaStream_t stream) {
  if (n == 0) {
    MTSV_LAUNCH(scan_empty, 1, 1, 0, stream, d_out, d_total);
    MTSV_CUDA_TRY(cudaGetLastError());
    return 0;
  }
  uint64_t nb = (n + kScanTile - 1) / kScanTile;
  if (nb > 0xffffffffull) return set_error(MTSVGPU_ELIMIT, "scan too large");
  if (tmp.cap < nb * sizeof(uint64_t)) {
    MTSV_CUDA_TRY(cudaStreamSynchronize(stream));
    MTSV_TRY(tmp.reserve(nb * sizeof(uint64_t)));
  }
  uint64_t* sums = tmp.as<uint64_t>();
  MTSV_LAUNCH(scan_tile_sums, (unsigned)nb, kScanThreads, 0, stream, d_in, n, sums);
  MTSV_LAUNCH(scan_sums_inplace, 1, 1024, 0, stream, sums, (uint32_t)nb, d_total);
  MTSV_LAUNCH(scan_apply, (unsigned)nb, kScanThreads, 0, stream, d_in, d_out, n, sums);
  MTSV_CUDA_TRY(cudaGetLastError());
  return 0;
}

}  // namespace mtsv
