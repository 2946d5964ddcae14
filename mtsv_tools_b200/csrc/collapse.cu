// collapse.cu — chunk-sharded operation (SURVEY §8e): merge the hit lists that several MG-index
// chunks produced for the SAME reads.  This is the reduction mtsv-collapse performs on results files
// (src/collapse.rs:543-654); mode TaxId: for equal read ids keep the minimum edit per TaxID
// (:597-602), hits listed by ascending TaxID (write_collapsed_taxid, :278-279); mode TaxIdGi further down.
//
// Inputs: n_parts device arrays of mtsvgpu_hit, each with a per-read u32 count array for the same
// n_reads reads (after the NCCL exchange every rank holds all parts for its own range of reads).
// All kernels are flat over reads / hits; the per-read sort reuses the binner's segmented sorts.
#include <mutex>

#include "ctx.h"

namespace mtsv {

struct PartsView {
  const mtsvgpu_hit* hits[16];
  const uint32_t* counts[16];
  const uint32_t* offs[16];  // exclusive scans of counts
  uint32_t n_parts;
};

__global__ void collapse_total_kernel(PartsView pv, uint32_t n_reads, uint32_t* __restrict__ total) {
  uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n_reads) return;
  uint32_t t = 0;
  for (uint32_t p = 0; p < pv.n_parts; ++p) t += pv.counts[p][r];
  total[r] = t;
}

// key = tax << 32 | edit: ascending order groups a TaxID's hits with the smallest edit first
__global__ void collapse_scatter_kernel(PartsView pv, uint32_t n_reads, const uint32_t* __restrict__ comb_off,
                                        uint64_t* __restrict__ keys) {
  uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t r = t / pv.n_parts, p = t % pv.n_parts;
  if (r >= n_reads) return;
  uint32_t dst = comb_off[r];
  for (uint32_t q = 0; q < p; ++q) dst += pv.counts[q][r];
  const mtsvgpu_hit* src = pv.hits[p] + pv.offs[p][r];
  uint32_t n = pv.counts[p][r];
  for (uint32_t i = 0; i < n; ++i) keys[dst + i] = ((uint64_t)src[i].tax_id << 32) | src[i].edit;
}

__global__ void collapse_count_kernel(const uint64_t* __restrict__ keys, const uint32_t* __restrict__ comb_off,
                                      uint32_t n_reads, uint32_t* __restrict__ n_out) {
  uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n_reads) return;
  n_out[r] = taxid_count(keys, comb_off[r], comb_off[r + 1]);
}

__global__ void collapse_write_kernel(const uint64_t* __restrict__ keys, const uint32_t* __restrict__ comb_off,
                                      const uint32_t* __restrict__ out_off32, uint32_t n_reads,
                                      mtsvgpu_taxhit* __restrict__ out, uint64_t* __restrict__ out_off) {
  uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r > n_reads) return;
  out_off[r] = out_off32[r];
  if (r == n_reads) return;
  taxid_write(keys, comb_off[r], comb_off[r + 1], out, out_off32[r]);
}

// ------------------------------------------------------------------------------------------
// mode TaxIdGi (src/collapse.rs:603-625): per read and per (TaxID, GI) keep the hit with the smallest edit,
// ties to the smallest offset; listed by (TaxID, GI) (write_collapsed_taxid_gi, :311-318).
// The key (tax, gi, edit, offset) does not fit the 64-bit segmented sorts, and per-read lists are short, so
// this is done without sorting: a hit is a winner when no other hit of the read with the same (tax, gi)
// precedes it in (edit, offset, position); a winner's output slot is the number of winners with a smaller
// (tax, gi).  One warp per read, O(n^2) over the read's combined list.
// ------------------------------------------------------------------------------------------
__global__ void collapse_gather_kernel(PartsView pv, uint32_t n_reads, const uint32_t* __restrict__ comb_off,
                                       mtsvgpu_hit* __restrict__ comb) {
  uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t r = t / pv.n_parts, p = t % pv.n_parts;
  if (r >= n_reads) return;
  uint32_t dst = comb_off[r];
  for (uint32_t q = 0; q < p; ++q) dst += pv.counts[q][r];
  const mtsvgpu_hit* src = pv.hits[p] + pv.offs[p][r];
  uint32_t n = pv.counts[p][r];
  for (uint32_t i = 0; i < n; ++i) comb[dst + i] = src[i];
}

__device__ __forceinline__ bool same_group(const mtsvgpu_hit& a, const mtsvgpu_hit& b) {
  return a.tax_id == b.tax_id && a.gi == b.gi;
}
__device__ __forceinline__ bool group_less(const mtsvgpu_hit& a, const mtsvgpu_hit& b) {
  return a.tax_id != b.tax_id ? a.tax_id < b.tax_id : a.gi < b.gi;
}

// flag[i] = 1 when combined hit i is the winner of its (tax, gi) group; n_out[r] = winners of read r
__global__ void __launch_bounds__(128) collapse_long_flag_kernel(const mtsvgpu_hit* __restrict__ comb,
                                                                 const uint32_t* __restrict__ comb_off, uint32_t n_reads,
                                                                 uint8_t* __restrict__ flag, uint32_t* __restrict__ n_out) {
  const uint32_t r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const unsigned lane = threadIdx.x & 31;
  if (r >= n_reads) return;
  const uint32_t b = comb_off[r], e = comb_off[r + 1];
  uint32_t wins = 0;
  for (uint32_t i = b + lane; i < e; i += 32) {
    const mtsvgpu_hit hi = comb[i];
    bool win = true;
    for (uint32_t j = b; j < e && win; ++j) {
      if (j == i) continue;
      const mtsvgpu_hit hj = comb[j];
      if (!same_group(hi, hj)) continue;
      const bool before = hj.edit != hi.edit ? hj.edit < hi.edit
                                             : (hj.offset != hi.offset ? hj.offset < hi.offset : j < i);
      if (before) win = false;
    }
    flag[i] = win ? 1 : 0;
    wins += win;
  }
  for (int d = 16; d; d >>= 1) wins += __shfl_xor_sync(0xffffffffu, wins, d);
  if (lane == 0) n_out[r] = wins;
}

__global__ void __launch_bounds__(128) collapse_long_write_kernel(const mtsvgpu_hit* __restrict__ comb,
                                                                  const uint32_t* __restrict__ comb_off,
                                                                  const uint8_t* __restrict__ flag,
                                                                  const uint32_t* __restrict__ out_off32, uint32_t n_reads,
                                                                  mtsvgpu_hit* __restrict__ out, uint64_t* __restrict__ out_off) {
  const uint32_t r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const unsigned lane = threadIdx.x & 31;
  if (r > n_reads) return;
  if (lane == 0) out_off[r] = out_off32[r];
  if (r == n_reads) return;
  const uint32_t b = comb_off[r], e = comb_off[r + 1], w = out_off32[r];
  for (uint32_t i = b + lane; i < e; i += 32) {
    if (!flag[i]) continue;
    const mtsvgpu_hit hi = comb[i];
    uint32_t rank = 0;
    for (uint32_t j = b; j < e; ++j)
      if (flag[j] && group_less(comb[j], hi)) ++rank;
    out[w + rank] = hi;
  }
}

int collapse_device(int device, cudaStream_t st, uint32_t n_parts, const mtsvgpu_hit* const* d_hits,
                    const uint32_t* const* d_counts, uint64_t n_reads, mtsvgpu_taxhit** d_out,
                    uint64_t** d_out_off, uint64_t* n_out) {
  if (!d_hits || !d_counts || !d_out || !d_out_off || !n_out) return set_error(MTSVGPU_EINVAL, "null argument");
  if (n_parts == 0 || n_parts > 16) return set_error(MTSVGPU_EINVAL, "n_parts must be in [1,16]");
  if (n_reads > 0x7ffffff0ull) return set_error(MTSVGPU_ELIMIT, "too many reads in one collapse call");
  MTSV_TRY(use_device(device));
  if (device >= 16) return set_error(MTSVGPU_EINVAL, "device %d out of range", device);
  const uint32_t nr = (uint32_t)n_reads;
  // grow-only workspace per device (cudaMalloc / cudaFree per call would cost more than the kernels); never
  // destroyed: freeing at process exit would run after the CUDA runtime has been torn down
  static CollapseScratch* const g_ws = new CollapseScratch[16];
  static std::mutex g_mu;
  std::lock_guard<std::mutex> lock(g_mu);
  CollapseScratch& w = g_ws[device];
  DevBuf* offs = w.offs;
  DevBuf &total = w.total, &comb_off = w.comb_off, &keys = w.keys, &scan_tmp = w.scan_tmp,
         &counters = w.counters, &worklist = w.worklist, &cnt_out = w.cnt_out, &off_out32 = w.off_out32;

  PartsView pv{};
  pv.n_parts = n_parts;
  MTSV_TRY(counters.reserve(sizeof(BatchCounters) + 16));
  MTSV_CUDA_TRY(cudaMemsetAsync(counters.p.get(), 0, sizeof(BatchCounters) + 16, st));
  uint64_t* d_tot = reinterpret_cast<uint64_t*>(counters.as<uint8_t>() + sizeof(BatchCounters));
  for (uint32_t p = 0; p < n_parts; ++p) {
    pv.hits[p] = d_hits[p];
    pv.counts[p] = d_counts[p];
    MTSV_TRY(offs[p].reserve(((size_t)nr + 1) * 4));
    MTSV_TRY(exclusive_scan_u32(d_counts[p], offs[p].as<uint32_t>(), nr, scan_tmp, nullptr, st));
    pv.offs[p] = offs[p].as<uint32_t>();
  }
  MTSV_TRY(total.reserve(((size_t)nr + 1) * 4));
  MTSV_TRY(comb_off.reserve(((size_t)nr + 1) * 4));
  MTSV_TRY(cnt_out.reserve(((size_t)nr + 1) * 4));
  MTSV_TRY(off_out32.reserve(((size_t)nr + 1) * 4));
  const unsigned rgrid = (nr + 255) / 256 + 1;
  if (nr) MTSV_LAUNCH(collapse_total_kernel, rgrid, 256, 0, st, pv, nr, total.as<uint32_t>());
  MTSV_TRY(exclusive_scan_u32(total.as<uint32_t>(), comb_off.as<uint32_t>(), nr, scan_tmp, d_tot, st));
  uint64_t h_tot = 0;
  MTSV_CUDA_TRY(cudaMemcpyAsync(&h_tot, d_tot, 8, cudaMemcpyDeviceToHost, st));
  MTSV_CUDA_TRY(cudaStreamSynchronize(st));
  if (h_tot > 0xfffffff0ull) return set_error(MTSVGPU_ELIMIT, "more than 2^32 hits in one collapse call");
  MTSV_TRY(keys.reserve((size_t)(h_tot + 1) * 8));
  if (nr && h_tot) {
    const uint64_t threads = (uint64_t)nr * n_parts;
    MTSV_LAUNCH(collapse_scatter_kernel, (unsigned)((threads + 255) / 256), 256, 0, st, pv, nr,
                comb_off.as<uint32_t>(), keys.as<uint64_t>());
    MTSV_TRY(run_segmented_sort(st, worklist, keys.as<uint64_t>(), comb_off.as<uint32_t>(), total.as<uint32_t>(), nr,
                                1, counters.as<BatchCounters>()));
  }
  if (nr) MTSV_LAUNCH(collapse_count_kernel, rgrid, 256, 0, st, keys.as<uint64_t>(), comb_off.as<uint32_t>(), nr,
                      cnt_out.as<uint32_t>());
  MTSV_TRY(exclusive_scan_u32(cnt_out.as<uint32_t>(), off_out32.as<uint32_t>(), nr, scan_tmp, d_tot, st));
  MTSV_CUDA_TRY(cudaMemcpyAsync(&h_tot, d_tot, 8, cudaMemcpyDeviceToHost, st));
  MTSV_CUDA_TRY(cudaStreamSynchronize(st));
  DevPtr<mtsvgpu_taxhit> out;
  DevPtr<uint64_t> out_off;
  MTSV_TRY(dev_alloc(out, h_tot + 1));
  MTSV_TRY(dev_alloc(out_off, (uint64_t)nr + 1));
  MTSV_LAUNCH(collapse_write_kernel, rgrid, 256, 0, st, keys.as<uint64_t>(), comb_off.as<uint32_t>(),
              off_out32.as<uint32_t>(), nr, out.get(), out_off.get());
  cudaError_t e = cudaStreamSynchronize(st);
  if (e != cudaSuccess) return set_error(MTSVGPU_ECUDA, "collapse: %s", cudaGetErrorString(e));
  // the caller frees the results with mtsvgpu_device_free
  *d_out = out.release();
  *d_out_off = out_off.release();
  *n_out = h_tot;
  return 0;
}

// The same TaxId-mode merge without a host round trip: scratch and outputs are pre-sized by the caller's bound on
// the combined hits (`hit_cap`), the total lands in *d_n_out.  Used as the epilogue of the chunk-sharded exchange
// (chunked.cu); once the scratch has grown to its working size nothing here synchronises.
int collapse_taxid_async(CollapseScratch& w, cudaStream_t st, uint32_t n_parts, const mtsvgpu_hit* const* d_hits,
                         const uint32_t* const* d_counts, uint32_t nr, uint64_t hit_cap, mtsvgpu_taxhit* out,
                         uint64_t* out_off, uint64_t* d_n_out) {
  if (n_parts == 0 || n_parts > 16) return set_error(MTSVGPU_EINVAL, "n_parts must be in [1,16]");
  if (hit_cap > 0xfffffff0ull) return set_error(MTSVGPU_ELIMIT, "more than 2^32 hits in one collapse call");
  PartsView pv{};
  pv.n_parts = n_parts;
  MTSV_TRY(w.counters.reserve(sizeof(BatchCounters) + 16));
  MTSV_CUDA_TRY(cudaMemsetAsync(w.counters.p.get(), 0, sizeof(BatchCounters) + 16, st));
  uint64_t* d_tot = reinterpret_cast<uint64_t*>(w.counters.as<uint8_t>() + sizeof(BatchCounters));
  MTSV_TRY(w.scan_tmp.reserve((((size_t)nr + 1 + 2047) / 2048 + 1) * 8));
  MTSV_TRY(w.worklist.reserve((size_t)3 * (nr + 1) * 4));
  for (uint32_t p = 0; p < n_parts; ++p) {
    pv.hits[p] = d_hits[p];
    pv.counts[p] = d_counts[p];
    MTSV_TRY(w.offs[p].reserve(((size_t)nr + 1) * 4));
    MTSV_TRY(exclusive_scan_u32(d_counts[p], w.offs[p].as<uint32_t>(), nr, w.scan_tmp, nullptr, st));
    pv.offs[p] = w.offs[p].as<uint32_t>();
  }
  MTSV_TRY(w.total.reserve(((size_t)nr + 1) * 4));
  MTSV_TRY(w.comb_off.reserve(((size_t)nr + 1) * 4));
  MTSV_TRY(w.cnt_out.reserve(((size_t)nr + 1) * 4));
  MTSV_TRY(w.off_out32.reserve(((size_t)nr + 1) * 4));
  MTSV_TRY(w.keys.reserve((size_t)(hit_cap + 1) * 8));
  const unsigned rgrid = (nr + 255) / 256 + 1;
  if (nr) MTSV_LAUNCH(collapse_total_kernel, rgrid, 256, 0, st, pv, nr, w.total.as<uint32_t>());
  MTSV_TRY(exclusive_scan_u32(w.total.as<uint32_t>(), w.comb_off.as<uint32_t>(), nr, w.scan_tmp, d_tot, st));
  if (nr) {
    const uint64_t threads = (uint64_t)nr * n_parts;
    MTSV_LAUNCH(collapse_scatter_kernel, (unsigned)((threads + 255) / 256), 256, 0, st, pv, nr,
                w.comb_off.as<uint32_t>(), w.keys.as<uint64_t>());
    MTSV_TRY(run_segmented_sort(st, w.worklist, w.keys.as<uint64_t>(), w.comb_off.as<uint32_t>(), w.total.as<uint32_t>(),
                                nr, 1, w.counters.as<BatchCounters>()));
    MTSV_LAUNCH(collapse_count_kernel, rgrid, 256, 0, st, w.keys.as<uint64_t>(), w.comb_off.as<uint32_t>(), nr,
                w.cnt_out.as<uint32_t>());
  }
  MTSV_TRY(exclusive_scan_u32(w.cnt_out.as<uint32_t>(), w.off_out32.as<uint32_t>(), nr, w.scan_tmp, d_n_out, st));
  MTSV_LAUNCH(collapse_write_kernel, rgrid, 256, 0, st, w.keys.as<uint64_t>(), w.comb_off.as<uint32_t>(),
              w.off_out32.as<uint32_t>(), nr, out, out_off);
  MTSV_CUDA_TRY(cudaGetLastError());
  return 0;
}

int collapse_device_long(int device, cudaStream_t st, uint32_t n_parts, const mtsvgpu_hit* const* d_hits,
                         const uint32_t* const* d_counts, uint64_t n_reads, mtsvgpu_hit** d_out,
                         uint64_t** d_out_off, uint64_t* n_out) {
  if (!d_hits || !d_counts || !d_out || !d_out_off || !n_out) return set_error(MTSVGPU_EINVAL, "null argument");
  if (n_parts == 0 || n_parts > 16) return set_error(MTSVGPU_EINVAL, "n_parts must be in [1,16]");
  if (n_reads > 0x07fffff0ull) return set_error(MTSVGPU_ELIMIT, "too many reads in one collapse call");
  MTSV_TRY(use_device(device));
  const uint32_t nr = (uint32_t)n_reads;
  DevBuf offs[16], total, comb_off, comb, flag, scan_tmp, counters, cnt_out, off_out32;
  PartsView pv{};
  pv.n_parts = n_parts;
  MTSV_TRY(counters.reserve(16));
  MTSV_CUDA_TRY(cudaMemsetAsync(counters.p.get(), 0, 16, st));
  uint64_t* d_tot = counters.as<uint64_t>();
  for (uint32_t p = 0; p < n_parts; ++p) {
    pv.hits[p] = d_hits[p];
    pv.counts[p] = d_counts[p];
    MTSV_TRY(offs[p].reserve(((size_t)nr + 1) * 4));
    MTSV_TRY(exclusive_scan_u32(d_counts[p], offs[p].as<uint32_t>(), nr, scan_tmp, nullptr, st));
    pv.offs[p] = offs[p].as<uint32_t>();
  }
  MTSV_TRY(total.reserve(((size_t)nr + 1) * 4));
  MTSV_TRY(comb_off.reserve(((size_t)nr + 1) * 4));
  MTSV_TRY(cnt_out.reserve(((size_t)nr + 1) * 4));
  MTSV_TRY(off_out32.reserve(((size_t)nr + 1) * 4));
  const unsigned rgrid = (nr + 255) / 256 + 1;
  if (nr) MTSV_LAUNCH(collapse_total_kernel, rgrid, 256, 0, st, pv, nr, total.as<uint32_t>());
  MTSV_TRY(exclusive_scan_u32(total.as<uint32_t>(), comb_off.as<uint32_t>(), nr, scan_tmp, d_tot, st));
  uint64_t h_tot = 0;
  MTSV_CUDA_TRY(cudaMemcpyAsync(&h_tot, d_tot, 8, cudaMemcpyDeviceToHost, st));
  MTSV_CUDA_TRY(cudaStreamSynchronize(st));
  if (h_tot > 0xfffffff0ull) return set_error(MTSVGPU_ELIMIT, "more than 2^32 hits in one collapse call");
  MTSV_TRY(comb.reserve((size_t)(h_tot + 1) * sizeof(mtsvgpu_hit)));
  MTSV_TRY(flag.reserve((size_t)h_tot + 1));
  const unsigned wgrid = (unsigned)(((uint64_t)(nr + 1) * 32 + 127) / 128);
  if (nr) {
    if (h_tot) {
      const uint64_t threads = (uint64_t)nr * n_parts;
      MTSV_LAUNCH(collapse_gather_kernel, (unsigned)((threads + 255) / 256), 256, 0, st, pv, nr,
                  comb_off.as<uint32_t>(), comb.as<mtsvgpu_hit>());
    }
    MTSV_LAUNCH(collapse_long_flag_kernel, wgrid, 128, 0, st, comb.as<mtsvgpu_hit>(), comb_off.as<uint32_t>(), nr,
                flag.as<uint8_t>(), cnt_out.as<uint32_t>());
  }
  MTSV_TRY(exclusive_scan_u32(cnt_out.as<uint32_t>(), off_out32.as<uint32_t>(), nr, scan_tmp, d_tot, st));
  MTSV_CUDA_TRY(cudaMemcpyAsync(&h_tot, d_tot, 8, cudaMemcpyDeviceToHost, st));
  MTSV_CUDA_TRY(cudaStreamSynchronize(st));
  DevPtr<mtsvgpu_hit> out;
  DevPtr<uint64_t> out_off;
  MTSV_TRY(dev_alloc(out, h_tot + 1));
  MTSV_TRY(dev_alloc(out_off, (uint64_t)nr + 1));
  MTSV_LAUNCH(collapse_long_write_kernel, wgrid, 128, 0, st, comb.as<mtsvgpu_hit>(), comb_off.as<uint32_t>(),
              flag.as<uint8_t>(), off_out32.as<uint32_t>(), nr, out.get(), out_off.get());
  cudaError_t e = cudaStreamSynchronize(st);
  if (e != cudaSuccess) return set_error(MTSVGPU_ECUDA, "collapse (taxid-gi): %s", cudaGetErrorString(e));
  *d_out = out.release();
  *d_out_off = out_off.release();
  *n_out = h_tot;
  return 0;
}

}  // namespace mtsv
