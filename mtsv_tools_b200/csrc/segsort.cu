// segsort.cu — segmented sort of u64 keys, for the binner's seed hits per read-strand and the (TaxID, edit) merge of
// collapse.cu.  Bitonic network in its "all ascending" form (first step of each merge compares i with its mirror
// i ^ (k-1)), which tolerates virtual +inf padding, so segment lengths need not be powers of two.  Segment q =
// keys[seg_off[q] .. + seg_cnt[q]).
//   <= 32 keys : one warp, registers + shuffles
//   <= 4096    : one CTA, shared memory
//   larger     : one CTA, in place in global memory (rare: > 4096 seed hits for one read-strand)
#include "ctx.h"

namespace mtsv {

struct SortCounts {  // lengths of the three work lists
  unsigned int n_warp, n_medium, n_large;
};

constexpr uint32_t kSortMedium = 4096;

__device__ __forceinline__ uint64_t warp_sort_u64(uint64_t v, unsigned lane) {
#pragma unroll
  for (int k = 2; k <= 32; k <<= 1) {
    {
      uint64_t o = __shfl_xor_sync(0xffffffffu, v, k - 1);
      bool low = (lane & (k - 1)) < ((lane ^ (k - 1)) & (k - 1));
      v = low ? (v < o ? v : o) : (v > o ? v : o);
    }
#pragma unroll
    for (int j = k >> 2; j > 0; j >>= 1) {
      uint64_t o = __shfl_xor_sync(0xffffffffu, v, j);
      bool low = (lane & j) == 0;
      v = low ? (v < o ? v : o) : (v > o ? v : o);
    }
  }
  return v;
}

// Segments are classified once (warp-aggregated appends to three work lists); segments of at most
// `min_count` keys are left to their consumer (the per-lane paths of coalesce / rank_emit order a
// handful of keys themselves, which beats launching a warp per query).
__global__ void __launch_bounds__(256) sort_classify_kernel(const uint32_t* __restrict__ seg_cnt, uint32_t nq,
                                                            uint32_t min_count, uint32_t* __restrict__ warp_list,
                                                            uint32_t* __restrict__ medium_list,
                                                            uint32_t* __restrict__ large_list,
                                                            SortCounts* __restrict__ ctr) {
  uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
  const unsigned lane = threadIdx.x & 31;
  uint32_t n = q < nq ? seg_cnt[q] : 0;
  int cls = n <= min_count || n < 2 ? -1 : (n <= 32 ? 0 : (n <= kSortMedium ? 1 : 2));
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    unsigned m = __ballot_sync(0xffffffffu, cls == c);
    if (!m) continue;
    unsigned int* counter = c == 0 ? &ctr->n_warp : (c == 1 ? &ctr->n_medium : &ctr->n_large);
    uint32_t* list = c == 0 ? warp_list : (c == 1 ? medium_list : large_list);
    uint32_t base = 0;
    if (lane == (unsigned)(__ffs(m) - 1)) base = atomicAdd(counter, (unsigned)__popc(m));
    base = __shfl_sync(0xffffffffu, base, __ffs(m) - 1);
    if (cls == c) list[base + __popc(m & ((1u << lane) - 1))] = q;
  }
}

__global__ void __launch_bounds__(256) sort_warp_kernel(uint64_t* __restrict__ keys,
                                                        const uint32_t* __restrict__ seg_off,
                                                        const uint32_t* __restrict__ seg_cnt,
                                                        const uint32_t* __restrict__ list,
                                                        const SortCounts* __restrict__ ctr) {
  const unsigned lane = threadIdx.x & 31;
  const uint32_t n_list = ctr->n_warp;
  const uint32_t warps = (gridDim.x * blockDim.x) >> 5;
  for (uint32_t it = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; it < n_list; it += warps) {
    uint32_t q = list[it];
    uint32_t n = seg_cnt[q];
    uint64_t* base = keys + seg_off[q];
    uint64_t v = lane < n ? base[lane] : ~0ull;
    v = warp_sort_u64(v, lane);
    if (lane < n) base[lane] = v;
  }
}

__global__ void __launch_bounds__(512) sort_medium_kernel(uint64_t* __restrict__ keys,
                                                          const uint32_t* __restrict__ seg_off,
                                                          const uint32_t* __restrict__ seg_cnt,
                                                          const uint32_t* __restrict__ list,
                                                          const SortCounts* __restrict__ ctr) {
  __shared__ uint64_t sk[kSortMedium];
  const uint32_t n_list = ctr->n_medium;
  for (uint32_t it = blockIdx.x; it < n_list; it += gridDim.x) {
    uint32_t q = list[it];
    uint32_t n = seg_cnt[q];
    uint64_t* base = keys + seg_off[q];
    uint32_t N = 64;
    while (N < n) N <<= 1;
    for (uint32_t i = threadIdx.x; i < N; i += blockDim.x) sk[i] = i < n ? base[i] : ~0ull;
    __syncthreads();
    for (uint32_t k = 2; k <= N; k <<= 1) {
      for (uint32_t i = threadIdx.x; i < N; i += blockDim.x) {
        uint32_t l = i ^ (k - 1);
        if (l > i) {
          uint64_t a = sk[i], b = sk[l];
          if (a > b) {
            sk[i] = b;
            sk[l] = a;
          }
        }
      }
      __syncthreads();
      for (uint32_t j = k >> 2; j > 0; j >>= 1) {
        for (uint32_t i = threadIdx.x; i < N; i += blockDim.x) {
          uint32_t l = i ^ j;
          if (l > i) {
            uint64_t a = sk[i], b = sk[l];
            if (a > b) {
              sk[i] = b;
              sk[l] = a;
            }
          }
        }
        __syncthreads();
      }
    }
    for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) base[i] = sk[i];
    __syncthreads();
  }
}

__global__ void __launch_bounds__(1024) sort_large_kernel(uint64_t* __restrict__ keys,
                                                          const uint32_t* __restrict__ seg_off,
                                                          const uint32_t* __restrict__ seg_cnt,
                                                          const uint32_t* __restrict__ list,
                                                          const SortCounts* __restrict__ ctr) {
  const uint32_t n_list = ctr->n_large;
  for (uint32_t it = blockIdx.x; it < n_list; it += gridDim.x) {
    uint32_t q = list[it];
    uint32_t n = seg_cnt[q];
    uint64_t* base = keys + seg_off[q];
    uint64_t N = 64;
    while (N < n) N <<= 1;
    for (uint64_t k = 2; k <= N; k <<= 1) {
      for (uint64_t i = threadIdx.x; i < n; i += blockDim.x) {
        uint64_t l = i ^ (k - 1);
        if (l > i && l < n) {
          uint64_t a = base[i], b = base[l];
          if (a > b) {
            base[i] = b;
            base[l] = a;
          }
        }
      }
      __syncthreads();
      for (uint64_t j = k >> 2; j > 0; j >>= 1) {
        for (uint64_t i = threadIdx.x; i < n; i += blockDim.x) {
          uint64_t l = i ^ j;
          if (l > i && l < n) {
            uint64_t a = base[i], b = base[l];
            if (a > b) {
              base[i] = b;
              base[l] = a;
            }
          }
        }
        __syncthreads();
      }
    }
  }
}

int SegSortScratch::reserve(uint32_t nq) {
  MTSV_TRY(lists.reserve((size_t)3 * nq * 4));
  return counts.reserve(sizeof(SortCounts));
}

int run_segmented_sort(cudaStream_t st, SegSortScratch& s, uint64_t* keys, const uint32_t* seg_off,
                       const uint32_t* seg_cnt, uint32_t nq, uint32_t min_count) {
  if (s.lists.cap < (size_t)3 * nq * 4 || !s.counts.p) {
    MTSV_CUDA_TRY(cudaStreamSynchronize(st));
    MTSV_TRY(s.reserve(nq));
  }
  uint32_t* lists = s.lists.as<uint32_t>();
  SortCounts* d_ctr = s.counts.as<SortCounts>();
  MTSV_CUDA_TRY(cudaMemsetAsync(d_ctr, 0, sizeof(SortCounts), st));
  MTSV_LAUNCH(sort_classify_kernel, (nq + 255) / 256, 256, 0, st, seg_cnt, nq, min_count, lists, lists + nq,
              lists + 2 * (size_t)nq, d_ctr);
  MTSV_LAUNCH(sort_warp_kernel, sm_count() * 8, 256, 0, st, keys, seg_off, seg_cnt, lists, d_ctr);
  MTSV_LAUNCH(sort_medium_kernel, sm_count() * 4, 512, 0, st, keys, seg_off, seg_cnt, lists + nq, d_ctr);
  MTSV_LAUNCH(sort_large_kernel, sm_count(), 1024, 0, st, keys, seg_off, seg_cnt, lists + 2 * (size_t)nq, d_ctr);
  MTSV_CUDA_TRY(cudaGetLastError());
  return 0;
}

}  // namespace mtsv
