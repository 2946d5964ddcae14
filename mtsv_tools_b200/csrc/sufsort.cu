// sufsort.cu — suffix array of the '$'-terminated reference text, on the device.
//
// Replaces the `suffix_array(&seq)` call of mtsv-build (MGIndex::new, src/index.rs:560-561; rust-bio wraps a
// single-threaded SA-IS).  The suffix array of a text that ends in a unique smallest sentinel is unique, so any
// correct construction yields the same BWT / samples / `.index` bytes.
//
// Method: prefix doubling with discarding (Manber-Myers / Larsson-Sadakane) on hand-written LSD radix sorts.
//   round 0   key = the first 21 symbols (3 bits each: $ < A < C < G < N < T), value = suffix start; one
//             8-pass radix sort of all n pairs; groups of equal keys get their first SA position as rank
//   round r   only suffixes in groups of >= 2 stay active; an active suffix i is re-sorted inside its group by
//             rank[i + h] (key = group head << 32 | rank[i+h] + 1), h = 21 * 2^(r-1); groups split, singletons
//             leave.  The active list is processed in slabs cut at group boundaries so the scratch is bounded.
// All arrays are 32-bit (n < 2^32 - 64, the limit of the device index); nothing here depends on n < 2^31.
// HBM streaming bound: a radix pass moves 32 B per pair (8 B histogram read, 12 B in, 12 B out).
#include <stdlib.h>
#include <string.h>

#include "ctx.h"

namespace mtsv {
namespace {

// ---------------------------------------------------------------------------------------------
// LSD radix sort of (u64 key, u32 value) pairs, 8-bit digits, stable
// ---------------------------------------------------------------------------------------------
constexpr int kRsThreads = 256;
constexpr int kRsItems = 16;
constexpr int kRsTile = kRsThreads * kRsItems;  // 4096 pairs
constexpr int kRsWarps = kRsThreads / 32;
constexpr int kRsBins = 257;  // 256 digits + one bin for the padding of the last tile

struct RsPlan {
  uint32_t tiles_per_chunk, n_chunks;
};

RsPlan rs_plan(uint64_t n) {
  const uint64_t tiles = (n + kRsTile - 1) / kRsTile;
  uint64_t tpc = tiles / ((uint64_t)sm_count() * 16);  // >= 16 chunks per SM when the input is large enough
  if (tpc < 1) tpc = 1;
  if (tpc > 64) tpc = 64;
  RsPlan p;
  p.tiles_per_chunk = (uint32_t)tpc;
  p.n_chunks = (uint32_t)((tiles + tpc - 1) / tpc);
  if (p.n_chunks == 0) p.n_chunks = 1;
  return p;
}

// per-chunk digit histogram: hist[digit * n_chunks + chunk]
__global__ void __launch_bounds__(kRsThreads) rs_hist_kernel(const uint64_t* __restrict__ keys, uint64_t n,
                                                             uint32_t shift, uint32_t tiles_per_chunk,
                                                             uint32_t n_chunks, uint32_t* __restrict__ hist) {
  __shared__ uint32_t h[256];
  h[threadIdx.x] = 0;
  __syncthreads();
  const uint64_t begin = (uint64_t)blockIdx.x * tiles_per_chunk * kRsTile;
  uint64_t end = begin + (uint64_t)tiles_per_chunk * kRsTile;
  if (end > n) end = n;
  const unsigned lane = threadIdx.x & 31;
  for (uint64_t base = begin + (threadIdx.x & ~31u); base < end; base += kRsThreads) {
    const uint64_t i = base + lane;
    const uint32_t d = i < end ? (uint32_t)((keys[i] >> shift) & 0xff) : 0xffffffffu;
    const unsigned peers = __match_any_sync(0xffffffffu, d);  // equal digits of a warp add once
    if (d != 0xffffffffu && lane == (unsigned)(__ffs(peers) - 1)) atomicAdd(&h[d], (uint32_t)__popc(peers));
  }
  __syncthreads();
  hist[(uint64_t)threadIdx.x * n_chunks + blockIdx.x] = h[threadIdx.x];
}

// scatter: a CTA walks the tiles of its chunk; inside a tile a pair's destination is
//   base(digit, chunk) + pairs of that digit in earlier tiles + in earlier warps of the tile + earlier in its warp
__global__ void __launch_bounds__(kRsThreads) rs_scatter_kernel(
    const uint64_t* __restrict__ keys_in, const uint32_t* __restrict__ vals_in, uint64_t* __restrict__ keys_out,
    uint32_t* __restrict__ vals_out, uint64_t n, uint32_t shift, uint32_t tiles_per_chunk, uint32_t n_chunks,
    const uint32_t* __restrict__ base) {
  __shared__ uint32_t gbase[256];
  __shared__ uint32_t whist[kRsWarps * kRsBins];
  const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  gbase[threadIdx.x] = base[(uint64_t)threadIdx.x * n_chunks + blockIdx.x];
  const uint64_t chunk_begin = (uint64_t)blockIdx.x * tiles_per_chunk * kRsTile;
  for (uint32_t t = 0; t < tiles_per_chunk; ++t) {
    const uint64_t tile0 = chunk_begin + (uint64_t)t * kRsTile;
    if (tile0 >= n) break;
    for (uint32_t i = threadIdx.x; i < kRsWarps * kRsBins; i += kRsThreads) whist[i] = 0;
    __syncthreads();
    uint64_t k[kRsItems];
    uint32_t v[kRsItems], r[kRsItems];
    const uint64_t wbase = tile0 + (uint64_t)warp * (kRsItems * 32);
    uint32_t* wh = whist + warp * kRsBins;
#pragma unroll
    for (int j = 0; j < kRsItems; ++j) {
      const uint64_t i = wbase + (uint64_t)j * 32 + lane;
      const bool ok = i < n;
      k[j] = ok ? keys_in[i] : 0;
      v[j] = ok ? vals_in[i] : 0;
      const uint32_t d = ok ? (uint32_t)((k[j] >> shift) & 0xff) : 256u;
      const unsigned peers = __match_any_sync(0xffffffffu, d);
      const unsigned leader = (unsigned)(__ffs(peers) - 1);
      uint32_t old = 0;
      if (lane == leader) {
        old = wh[d];
        wh[d] = old + (uint32_t)__popc(peers);
      }
      old = __shfl_sync(0xffffffffu, old, leader);
      r[j] = old + (uint32_t)__popc(peers & ((1u << lane) - 1u));
      __syncwarp();
    }
    __syncthreads();
    uint32_t tile_cnt = 0;
    {
      const uint32_t d = threadIdx.x;  // one digit per thread: exclusive prefix over the warps
#pragma unroll
      for (int w = 0; w < kRsWarps; ++w) {
        const uint32_t c = whist[w * kRsBins + d];
        whist[w * kRsBins + d] = tile_cnt;
        tile_cnt += c;
      }
    }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < kRsItems; ++j) {
      const uint64_t i = wbase + (uint64_t)j * 32 + lane;
      if (i < n) {
        const uint32_t d = (uint32_t)((k[j] >> shift) & 0xff);
        const uint32_t pos = gbase[d] + wh[d] + r[j];
        keys_out[pos] = k[j];
        vals_out[pos] = v[j];
      }
    }
    __syncthreads();
    gbase[threadIdx.x] += tile_cnt;
  }
}

struct SortScratch {
  DevBuf hist, scan_tmp;
};

// Sorts n pairs by the 8-bit digits at `shifts` (least significant first).  *where = 0 when the result is in
// (k0, v0), 1 when it is in (k1, v1).
int radix_sort_pairs(cudaStream_t st, uint64_t* k0, uint64_t* k1, uint32_t* v0, uint32_t* v1, uint64_t n,
                     const std::vector<uint32_t>& shifts, SortScratch& sc, int* where) {
  *where = 0;
  if (n == 0) return 0;
  const RsPlan pl = rs_plan(n);
  const uint64_t hn = (uint64_t)256 * pl.n_chunks;
  if (sc.hist.cap < (hn + 1) * 4) {
    MTSV_CUDA_TRY(cudaStreamSynchronize(st));
    MTSV_TRY(sc.hist.reserve((hn + 1) * 4));
  }
  uint32_t* hist = sc.hist.as<uint32_t>();
  uint64_t* ki = k0;
  uint64_t* ko = k1;
  uint32_t* vi = v0;
  uint32_t* vo = v1;
  for (uint32_t shift : shifts) {
    MTSV_LAUNCH(rs_hist_kernel, pl.n_chunks, kRsThreads, 0, st, ki, n, shift, pl.tiles_per_chunk, pl.n_chunks, hist);
    MTSV_TRY(exclusive_scan_u32(hist, hist, hn, sc.scan_tmp, nullptr, st));
    MTSV_LAUNCH(rs_scatter_kernel, pl.n_chunks, kRsThreads, 0, st, ki, vi, ko, vo, n, shift, pl.tiles_per_chunk,
                pl.n_chunks, hist);
    std::swap(ki, ko);
    std::swap(vi, vo);
    *where ^= 1;
  }
  MTSV_CUDA_TRY(cudaGetLastError());
  return 0;
}

// ---------------------------------------------------------------------------------------------
// inclusive max-scan of u32 in place (three phases, like util.cu's sum scan)
// ---------------------------------------------------------------------------------------------
constexpr int kMsThreads = 256;
constexpr int kMsItems = 8;
constexpr int kMsTile = kMsThreads * kMsItems;

__device__ __forceinline__ uint32_t warp_incl_max(uint32_t v) {
  const unsigned lane = threadIdx.x & 31;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const uint32_t o = __shfl_up_sync(0xffffffffu, v, d);
    if (lane >= (unsigned)d) v = max(v, o);
  }
  return v;
}

// inclusive max over the block of one value per thread; *total = block max (valid in every thread)
__device__ __forceinline__ uint32_t block_incl_max(uint32_t v, uint32_t* total) {
  __shared__ uint32_t wmax[32];
  const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = (blockDim.x + 31) >> 5;
  uint32_t inc = warp_incl_max(v);
  if (lane == 31) wmax[warp] = inc;
  __syncthreads();
  if (warp == 0) {
    uint32_t w = lane < nwarps ? wmax[lane] : 0;
    wmax[lane] = warp_incl_max(w);
  }
  __syncthreads();
  if (warp) inc = max(inc, wmax[warp - 1]);
  *total = wmax[nwarps - 1];
  __syncthreads();
  return inc;
}

__global__ void __launch_bounds__(kMsThreads) ms_tile_max(const uint32_t* __restrict__ a, uint64_t n,
                                                          uint32_t* __restrict__ tmax) {
  const uint64_t base = (uint64_t)blockIdx.x * kMsTile + (uint64_t)threadIdx.x * kMsItems;
  uint32_t m = 0;
#pragma unroll
  for (int i = 0; i < kMsItems; ++i)
    if (base + i < n) m = max(m, a[base + i]);
  uint32_t total;
  block_incl_max(m, &total);
  if (threadIdx.x == 0) tmax[blockIdx.x] = total;
}

// exclusive max-scan of the tile maxima, in place, by one block
__global__ void __launch_bounds__(1024) ms_scan_tiles(uint32_t* __restrict__ tmax, uint32_t nb) {
  __shared__ uint32_t incs[1024];
  uint32_t carry = 0;
  for (uint32_t base = 0; base < nb; base += blockDim.x) {
    const uint32_t i = base + threadIdx.x;
    const uint32_t v = i < nb ? tmax[i] : 0;
    uint32_t total;
    incs[threadIdx.x] = block_incl_max(v, &total);
    __syncthreads();
    const uint32_t ex = threadIdx.x ? incs[threadIdx.x - 1] : 0u;
    if (i < nb) tmax[i] = max(carry, ex);
    carry = max(carry, total);
    __syncthreads();
  }
}

__global__ void __launch_bounds__(kMsThreads) ms_apply(uint32_t* __restrict__ a, uint64_t n,
                                                       const uint32_t* __restrict__ tmax) {
  const uint64_t base = (uint64_t)blockIdx.x * kMsTile + (uint64_t)threadIdx.x * kMsItems;
  uint32_t v[kMsItems];
  uint32_t m = 0;
#pragma unroll
  for (int i = 0; i < kMsItems; ++i) {
    v[i] = base + i < n ? a[base + i] : 0;
    m = max(m, v[i]);
  }
  uint32_t total;
  const uint32_t inc = block_incl_max(m, &total);
  // exclusive over threads: inclusive of the previous thread
  __shared__ uint32_t incs[kMsThreads];
  incs[threadIdx.x] = inc;
  __syncthreads();
  uint32_t run = max(tmax[blockIdx.x], threadIdx.x ? incs[threadIdx.x - 1] : 0u);
#pragma unroll
  for (int i = 0; i < kMsItems; ++i) {
    run = max(run, v[i]);
    if (base + i < n) a[base + i] = run;
  }
}

int inclusive_max_scan_u32(uint32_t* d_a, uint64_t n, DevBuf& tmp, cudaStream_t st) {
  if (n == 0) return 0;
  const uint64_t nb = (n + kMsTile - 1) / kMsTile;
  if (tmp.cap < nb * 4) {
    MTSV_CUDA_TRY(cudaStreamSynchronize(st));
    MTSV_TRY(tmp.reserve(nb * 4));
  }
  uint32_t* tmax = tmp.as<uint32_t>();
  MTSV_LAUNCH(ms_tile_max, (unsigned)nb, kMsThreads, 0, st, d_a, n, tmax);
  MTSV_LAUNCH(ms_scan_tiles, 1, 1024, 0, st, tmax, (uint32_t)nb);
  MTSV_LAUNCH(ms_apply, (unsigned)nb, kMsThreads, 0, st, d_a, n, tmax);
  MTSV_CUDA_TRY(cudaGetLastError());
  return 0;
}

// ---------------------------------------------------------------------------------------------
// prefix doubling
// ---------------------------------------------------------------------------------------------
// byte order of the text's symbols: $ < A < C < G < N < T  (anything else sorts as N; the caller normalises)
__device__ __forceinline__ uint64_t sym3(uint8_t b) {
  switch (b) {
    case '$': return 0;
    case 'A': return 1;
    case 'C': return 2;
    case 'G': return 3;
    case 'T': return 5;
    default: return 4;
  }
}

// round 0: key of suffix i = its first K symbols, 3 bits each (0 past the end); 8 suffixes per thread
__global__ void __launch_bounds__(256) sfx_init_kernel(const uint8_t* __restrict__ text, uint64_t n, uint32_t K,
                                                       uint64_t* __restrict__ keys, uint32_t* __restrict__ vals) {
  const uint64_t i0 = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) * 8;
  if (i0 >= n) return;
  const uint64_t mask = K >= 21 ? 0x7fffffffffffffffull : ((1ull << (3 * K)) - 1);
  uint64_t key = 0;
  for (uint32_t j = 0; j < K; ++j) key = (key << 3) | (i0 + j < n ? sym3(text[i0 + j]) : 0);
#pragma unroll
  for (uint32_t t = 0; t < 8; ++t) {
    const uint64_t i = i0 + t;
    if (i < n) {
      keys[i] = key;
      vals[i] = (uint32_t)i;
    }
    key = ((key << 3) & mask) | (i + K < n ? sym3(text[i + K]) : 0);
  }
}

// after a sort: headv[j] = own SA position when pair j opens a group of equal keys, else 0
// (pos == nullptr: the pairs cover the whole array and j itself is the position)
__global__ void __launch_bounds__(256) sfx_heads_kernel(const uint64_t* __restrict__ keys, const uint32_t* __restrict__ pos,
                                                        uint64_t m, uint32_t* __restrict__ headv) {
  const uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= m) return;
  const bool open = j == 0 || keys[j] != keys[j - 1];
  headv[j] = open ? (pos ? pos[j] : (uint32_t)j) : 0u;
}

// headv is now the group head of every pair: publish ranks (and, for slabs, the new order into sa)
__global__ void __launch_bounds__(256) sfx_publish_kernel(const uint32_t* __restrict__ vals, const uint32_t* __restrict__ pos,
                                                          const uint32_t* __restrict__ headv, uint64_t m,
                                                          uint32_t* __restrict__ sa, uint32_t* __restrict__ rank) {
  const uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= m) return;
  const uint32_t v = vals[j];
  if (pos) sa[pos[j]] = v;
  rank[v] = headv[j];
}

// stays[j] = 1 when pair j is in a group of two or more
__global__ void __launch_bounds__(256) sfx_stays_kernel(const uint32_t* __restrict__ headv, const uint32_t* __restrict__ pos,
                                                        uint64_t m, uint32_t* __restrict__ stays) {
  const uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= m) return;
  const uint32_t pj = pos ? pos[j] : (uint32_t)j;
  const bool open = headv[j] == pj;
  bool next_open = true;
  if (j + 1 < m) next_open = headv[j + 1] == (pos ? pos[j + 1] : (uint32_t)(j + 1));
  stays[j] = (open && next_open) ? 0u : 1u;
}

__global__ void __launch_bounds__(256) sfx_compact_kernel(const uint32_t* __restrict__ idx, const uint32_t* __restrict__ pos,
                                                          uint64_t m, uint32_t* __restrict__ out) {
  const uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= m) return;
  if (idx[j + 1] != idx[j]) out[idx[j]] = pos ? pos[j] : (uint32_t)j;
}

// round r >= 1, one slab of the active list: key = group head << 32 | (rank[i + h] + 1, or 0 past the end)
__global__ void __launch_bounds__(256) sfx_slab_keys_kernel(const uint32_t* __restrict__ pos, uint64_t m,
                                                            const uint32_t* __restrict__ sa, const uint32_t* __restrict__ rank,
                                                            uint64_t n, uint64_t h, uint64_t* __restrict__ keys,
                                                            uint32_t* __restrict__ vals) {
  const uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= m) return;
  const uint32_t v = sa[pos[j]];
  const uint64_t nxt = (uint64_t)v + h;
  const uint64_t r2 = nxt < n ? (uint64_t)rank[nxt] + 1 : 0;
  keys[j] = ((uint64_t)rank[v] << 32) | r2;
  vals[j] = v;
}

// Where the slab that starts at active index a ends: at most `want` pairs, cut back to a group boundary; a
// group larger than `want` is taken whole.
__global__ void sfx_slab_cut_kernel(const uint32_t* __restrict__ pos, uint64_t m, uint64_t a, uint64_t want,
                                    const uint32_t* __restrict__ sa, const uint32_t* __restrict__ rank,
                                    unsigned long long* __restrict__ out) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  uint64_t b = a + want < m ? a + want : m;
  if (b < m) {
    const uint32_t hd = rank[sa[pos[b]]];
    uint64_t lo = a, hi = b;  // first active index whose position is >= hd
    while (lo < hi) {
      const uint64_t mid = (lo + hi) >> 1;
      if (pos[mid] < hd) lo = mid + 1;
      else hi = mid;
    }
    if (lo > a) {
      b = lo;
    } else {  // the group of pair b starts at a: find its end
      lo = b;
      hi = m;
      while (lo < hi) {
        const uint64_t mid = (lo + hi) >> 1;
        if (rank[sa[pos[mid]]] == hd) lo = mid + 1;
        else hi = mid;
      }
      b = lo;
    }
  }
  *out = b;
}

__global__ void __launch_bounds__(256) sfx_bwt_kernel(const uint8_t* __restrict__ text, const uint32_t* __restrict__ sa,
                                                      uint64_t n, uint8_t* __restrict__ bwt) {
  const uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n) return;
  const uint32_t p = sa[r];
  bwt[r] = text[p ? p - 1 : n - 1];  // bwt[r] = text[SA[r] - 1], the sentinel for SA[r] == 0 (bio::bwt)
}

uint32_t bits_of(uint64_t v) {  // bits needed to hold values 0..v
  uint32_t b = 1;
  while (b < 64 && (v >> b)) ++b;
  return b;
}

unsigned grid_for(uint64_t items, unsigned threads) { return (unsigned)((items + threads - 1) / threads); }

}  // namespace

// Suffix array (u32, n entries) of the n symbols at d_text, the last of which must be the only '$'.  `verbose` prints
// one line per round on stderr.
int suffix_array_device(const uint8_t* d_text, uint64_t n, cudaStream_t st, DevPtr<uint32_t>& sa_out, int verbose) {
  if (!d_text || n < 1) return set_error(MTSVGPU_EINVAL, "suffix sort: bad argument");
  if (n >= (1ull << 32) - 64) return set_error(MTSVGPU_ELIMIT, "suffix sort: %llu symbols (limit 2^32-64)", (unsigned long long)n);
  // test knobs: symbols in the round-0 key, pairs per slab
  uint32_t K = 21;
  uint64_t slab = 1ull << 29;
  if (const char* e = getenv("MTSV_B200_SUFSORT_K")) K = (uint32_t)std::min(21, std::max(1, atoi(e)));
  if (const char* e = getenv("MTSV_B200_SUFSORT_SLAB")) slab = (uint64_t)std::max(1ll, atoll(e));

  SortScratch sc;
  DevBuf ms_tmp, sum_tmp;
  DevPtr<uint32_t> sa, rank, apos, apos_next;
  DevPtr<unsigned long long> d_scalar;
  MTSV_TRY(dev_alloc(sa, n + 1));  // (+1: may trade places with the scan buffer of round 0)
  MTSV_TRY(dev_alloc(rank, n));
  MTSV_TRY(dev_alloc(d_scalar, 2));
  uint64_t m = 0;  // active pairs

  // ---- round 0 ----
  {
    DevPtr<uint64_t> k0, k1;
    DevPtr<uint32_t> v1;
    MTSV_TRY(dev_alloc(k0, n));
    MTSV_TRY(dev_alloc(k1, n));
    MTSV_TRY(dev_alloc(v1, n + 1));
    MTSV_LAUNCH(sfx_init_kernel, grid_for((n + 7) / 8, 256), 256, 0, st, d_text, n, K, k0.get(), sa.get());
    std::vector<uint32_t> shifts;
    for (uint32_t s = 0; s < 3 * K; s += 8) shifts.push_back(s);
    int where = 0;
    MTSV_TRY(radix_sort_pairs(st, k0.get(), k1.get(), sa.get(), v1.get(), n, shifts, sc, &where));
    uint64_t* ks = where ? k1.get() : k0.get();
    uint64_t* kfree = where ? k0.get() : k1.get();
    if (where) std::swap(sa, v1);  // the sorted suffix starts are the suffix array so far
    uint32_t* headv = reinterpret_cast<uint32_t*>(kfree);  // n u32 fit in the idle key buffer
    uint32_t* idx = v1.get();
    MTSV_LAUNCH(sfx_heads_kernel, grid_for(n, 256), 256, 0, st, ks, (const uint32_t*)nullptr, n, headv);
    MTSV_TRY(inclusive_max_scan_u32(headv, n, ms_tmp, st));
    MTSV_LAUNCH(sfx_publish_kernel, grid_for(n, 256), 256, 0, st, sa.get(), (const uint32_t*)nullptr, headv, n, sa.get(), rank.get());
    MTSV_LAUNCH(sfx_stays_kernel, grid_for(n, 256), 256, 0, st, headv, (const uint32_t*)nullptr, n, idx);
    MTSV_TRY(exclusive_scan_u32(idx, idx, n, sum_tmp, (uint64_t*)d_scalar.get(), st));
    MTSV_CUDA_TRY(cudaMemcpyAsync(&m, d_scalar.get(), 8, cudaMemcpyDeviceToHost, st));
    MTSV_CUDA_TRY(cudaStreamSynchronize(st));
    if (m) {
      MTSV_TRY(dev_alloc(apos, m));
      MTSV_LAUNCH(sfx_compact_kernel, grid_for(n, 256), 256, 0, st, idx, (const uint32_t*)nullptr, n, apos.get());
      MTSV_CUDA_TRY(cudaStreamSynchronize(st));
    }
    MTSV_CUDA_TRY(cudaGetLastError());
  }
  if (verbose) fprintf(stderr, "[mtsv_b200 sufsort] round 0: h=%u, %llu of %llu suffixes still tied\n", K, (unsigned long long)m, (unsigned long long)n);

  // ---- rounds r >= 1 ----
  uint64_t h = K;
  const uint32_t lo_passes = (bits_of(n) + 7) / 8, hi_passes = (bits_of(n - 1) + 7) / 8;
  std::vector<uint32_t> shifts;
  for (uint32_t i = 0; i < lo_passes; ++i) shifts.push_back(8 * i);
  for (uint32_t i = 0; i < hi_passes; ++i) shifts.push_back(32 + 8 * i);
  uint64_t ws_cap = 0;
  DevPtr<uint64_t> k0, k1;
  DevPtr<uint32_t> v0, v1, headv, idx;
  auto reserve_ws = [&](uint64_t need) -> int {
    if (need <= ws_cap) return 0;
    k0.reset(); k1.reset(); v0.reset(); v1.reset(); headv.reset(); idx.reset();
    MTSV_TRY(dev_alloc(k0, need));
    MTSV_TRY(dev_alloc(k1, need));
    MTSV_TRY(dev_alloc(v0, need));
    MTSV_TRY(dev_alloc(v1, need));
    MTSV_TRY(dev_alloc(headv, need));
    MTSV_TRY(dev_alloc(idx, need + 1));
    ws_cap = need;
    return 0;
  };
  for (uint32_t round = 1; m > 0; ++round) {
    if (round > 40) return set_error(MTSVGPU_ECUDA, "suffix sort: internal error, no convergence");
    MTSV_TRY(dev_alloc(apos_next, m));
    uint64_t m_next = 0, a = 0, n_slabs = 0;
    while (a < m) {
      unsigned long long b = 0;
      MTSV_LAUNCH(sfx_slab_cut_kernel, 1, 1, 0, st, apos.get(), m, a, slab, sa.get(), rank.get(), d_scalar.get());
      MTSV_CUDA_TRY(cudaMemcpyAsync(&b, d_scalar.get(), 8, cudaMemcpyDeviceToHost, st));
      MTSV_CUDA_TRY(cudaStreamSynchronize(st));
      if (b <= a || b > m) return set_error(MTSVGPU_ECUDA, "suffix sort: internal error, bad slab [%llu,%llu)", (unsigned long long)a, b);
      const uint64_t ms = b - a;
      MTSV_TRY(reserve_ws(std::max<uint64_t>(ms, std::min(slab, m))));
      const uint32_t* pos = apos.get() + a;
      MTSV_LAUNCH(sfx_slab_keys_kernel, grid_for(ms, 256), 256, 0, st, pos, ms, sa.get(), rank.get(), n, h, k0.get(), v0.get());
      int where = 0;
      MTSV_TRY(radix_sort_pairs(st, k0.get(), k1.get(), v0.get(), v1.get(), ms, shifts, sc, &where));
      const uint64_t* ks = where ? k1.get() : k0.get();
      const uint32_t* vs = where ? v1.get() : v0.get();
      MTSV_LAUNCH(sfx_heads_kernel, grid_for(ms, 256), 256, 0, st, ks, pos, ms, headv.get());
      MTSV_TRY(inclusive_max_scan_u32(headv.get(), ms, ms_tmp, st));
      MTSV_LAUNCH(sfx_publish_kernel, grid_for(ms, 256), 256, 0, st, vs, pos, headv.get(), ms, sa.get(), rank.get());
      MTSV_LAUNCH(sfx_stays_kernel, grid_for(ms, 256), 256, 0, st, headv.get(), pos, ms, idx.get());
      MTSV_TRY(exclusive_scan_u32(idx.get(), idx.get(), ms, sum_tmp, (uint64_t*)d_scalar.get() + 1, st));
      MTSV_LAUNCH(sfx_compact_kernel, grid_for(ms, 256), 256, 0, st, idx.get(), pos, ms, apos_next.get() + m_next);
      unsigned long long kept = 0;
      MTSV_CUDA_TRY(cudaMemcpyAsync(&kept, d_scalar.get() + 1, 8, cudaMemcpyDeviceToHost, st));
      MTSV_CUDA_TRY(cudaStreamSynchronize(st));
      MTSV_CUDA_TRY(cudaGetLastError());
      m_next += kept;
      a = b;
      ++n_slabs;
    }
    if (verbose)
      fprintf(stderr, "[mtsv_b200 sufsort] round %u: h=%llu, %llu pairs in %llu slab(s), %llu still tied\n", round,
              (unsigned long long)h, (unsigned long long)m, (unsigned long long)n_slabs, (unsigned long long)m_next);
    std::swap(apos, apos_next);
    apos_next.reset();
    m = m_next;
    h *= 2;
  }
  sa_out = std::move(sa);
  return 0;
}

// bwt[r] = text[SA[r] - 1] (bio::bwt, src/index.rs:566-567) on the device
int bwt_from_sa_device(const uint8_t* d_text, const uint32_t* d_sa, uint64_t n, cudaStream_t st, uint8_t* d_bwt) {
  MTSV_LAUNCH(sfx_bwt_kernel, grid_for(n, 256), 256, 0, st, d_text, d_sa, n, d_bwt);
  MTSV_CUDA_TRY(cudaGetLastError());
  return 0;
}

}  // namespace mtsv
