// collapse.cu — the library's (TaxID, edit) merge, and the device collapse of chunk-sharded operation.
//
// The merge (taxid_merge_count / taxid_merge_write): per read, a segment of keys tax << 32 | edit becomes each TaxID
// once with its minimum edit, by ascending TaxID (core.cuh::taxid_count / taxid_write).  The binner's assignments
// output (binner.cu) and the TaxId collapse below both go through it.
//
// The collapse (SURVEY §8e): merge the hit lists that several MG-index chunks produced for the SAME reads.  This is
// the reduction mtsv-collapse performs on results files (src/collapse.rs:543-654); mode TaxId: for equal read ids
// keep the minimum edit per TaxID (:597-602), hits listed by ascending TaxID (write_collapsed_taxid, :278-279); mode
// TaxIdGi further down.  Inputs: n_parts device arrays of mtsvgpu_hit, each with a per-read u32 count array for the
// same n_reads reads (after the chunk exchange every rank holds all parts for its own range of reads).
// All kernels are flat over reads / hits; the per-read sort is segsort.cu's.
#include <mutex>

#include "ctx.h"

namespace mtsv {

// records per read, after the segments have been sorted
__global__ void __launch_bounds__(256) taxid_count_kernel(const uint64_t* __restrict__ keys,
                                                          const uint32_t* __restrict__ seg_off, uint32_t n_reads,
                                                          uint32_t* __restrict__ n_out) {
  uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n_reads) return;
  n_out[r] = taxid_count(keys, seg_off[r], seg_off[r + 1]);
}

// appends the sub-batch's records to the batch output at out_base; read offsets go to out_off from read_base on
__global__ void __launch_bounds__(256) taxid_write_kernel(const uint64_t* __restrict__ keys,
                                                          const uint32_t* __restrict__ seg_off,
                                                          const uint32_t* __restrict__ tax_off, uint32_t n_reads,
                                                          mtsvgpu_taxhit* __restrict__ out, uint64_t out_base,
                                                          uint64_t* __restrict__ out_off, uint64_t read_base) {
  uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r > n_reads) return;
  out_off[read_base + r] = out_base + tax_off[r];  // r == n_reads: the end
  if (r == n_reads) return;
  taxid_write(keys, seg_off[r], seg_off[r + 1], out + out_base, tax_off[r]);
}

int taxid_merge_count(cudaStream_t st, SegSortScratch& sort, DevBuf& scan_tmp, uint64_t* keys, const uint32_t* seg_off,
                      const uint32_t* seg_cnt, uint32_t n_reads, uint64_t key_bound, uint32_t* tax_cnt,
                      uint32_t* tax_off, uint64_t* d_total) {
  if (n_reads) {
    if (key_bound) MTSV_TRY(run_segmented_sort(st, sort, keys, seg_off, seg_cnt, n_reads, 1));
    MTSV_LAUNCH(taxid_count_kernel, (n_reads + 255) / 256, 256, 0, st, keys, seg_off, n_reads, tax_cnt);
  }
  return exclusive_scan_u32(tax_cnt, tax_off, n_reads, scan_tmp, d_total, st);
}

void taxid_merge_write(cudaStream_t st, const uint64_t* keys, const uint32_t* seg_off, const uint32_t* tax_off,
                       uint32_t n_reads, mtsvgpu_taxhit* out, uint64_t out_base, uint64_t* out_off, uint64_t read_base) {
  MTSV_LAUNCH(taxid_write_kernel, (n_reads + 1 + 255) / 256, 256, 0, st, keys, seg_off, tax_off, n_reads, out, out_base,
              out_off, read_base);
}

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

// The parts of one collapse call: pv, their per-read offsets, and per read the combined count (w.total) and offset
// (w.comb_off); the combined total goes to *d_tot.
static int prepare_parts(CollapseScratch& w, cudaStream_t st, uint32_t n_parts, const mtsvgpu_hit* const* d_hits,
                         const uint32_t* const* d_counts, uint32_t nr, PartsView* pv, uint64_t** d_tot) {
  *pv = PartsView{};
  pv->n_parts = n_parts;
  MTSV_TRY(w.comb_total.reserve(8));
  *d_tot = w.comb_total.as<uint64_t>();
  for (uint32_t p = 0; p < n_parts; ++p) {
    pv->hits[p] = d_hits[p];
    pv->counts[p] = d_counts[p];
    MTSV_TRY(w.offs[p].reserve(((size_t)nr + 1) * 4));
    MTSV_TRY(exclusive_scan_u32(d_counts[p], w.offs[p].as<uint32_t>(), nr, w.scan_tmp, nullptr, st));
    pv->offs[p] = w.offs[p].as<uint32_t>();
  }
  for (DevBuf* b : {&w.total, &w.comb_off, &w.cnt_out, &w.off_out32}) MTSV_TRY(b->reserve(((size_t)nr + 1) * 4));
  if (nr) MTSV_LAUNCH(collapse_total_kernel, (nr + 255) / 256 + 1, 256, 0, st, *pv, nr, w.total.as<uint32_t>());
  return exclusive_scan_u32(w.total.as<uint32_t>(), w.comb_off.as<uint32_t>(), nr, w.scan_tmp, *d_tot, st);
}

// Mode TaxId after prepare_parts: the parts' hits as keys in read order (at most hit_cap of them), merged; per read
// the record count (w.cnt_out) and offset (w.off_out32), the record total to *d_n_out.
static int merge_parts_count(CollapseScratch& w, cudaStream_t st, const PartsView& pv, uint32_t nr, uint64_t hit_cap,
                             uint64_t* d_n_out) {
  MTSV_TRY(w.keys.reserve((size_t)(hit_cap + 1) * 8));
  if (nr && hit_cap) {
    const uint64_t threads = (uint64_t)nr * pv.n_parts;
    MTSV_LAUNCH(collapse_scatter_kernel, (unsigned)((threads + 255) / 256), 256, 0, st, pv, nr,
                w.comb_off.as<uint32_t>(), w.keys.as<uint64_t>());
  }
  return taxid_merge_count(st, w.sort, w.scan_tmp, w.keys.as<uint64_t>(), w.comb_off.as<uint32_t>(),
                           w.total.as<uint32_t>(), nr, hit_cap, w.cnt_out.as<uint32_t>(), w.off_out32.as<uint32_t>(),
                           d_n_out);
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
  PartsView pv;
  uint64_t* d_tot = nullptr;
  MTSV_TRY(prepare_parts(w, st, n_parts, d_hits, d_counts, nr, &pv, &d_tot));
  uint64_t h_tot = 0;
  MTSV_CUDA_TRY(cudaMemcpyAsync(&h_tot, d_tot, 8, cudaMemcpyDeviceToHost, st));
  MTSV_CUDA_TRY(cudaStreamSynchronize(st));
  if (h_tot > 0xfffffff0ull) return set_error(MTSVGPU_ELIMIT, "more than 2^32 hits in one collapse call");
  MTSV_TRY(merge_parts_count(w, st, pv, nr, h_tot, d_tot));
  MTSV_CUDA_TRY(cudaMemcpyAsync(&h_tot, d_tot, 8, cudaMemcpyDeviceToHost, st));
  MTSV_CUDA_TRY(cudaStreamSynchronize(st));
  DevPtr<mtsvgpu_taxhit> out;
  DevPtr<uint64_t> out_off;
  MTSV_TRY(dev_alloc(out, h_tot + 1));
  MTSV_TRY(dev_alloc(out_off, (uint64_t)nr + 1));
  taxid_merge_write(st, w.keys.as<uint64_t>(), w.comb_off.as<uint32_t>(), w.off_out32.as<uint32_t>(), nr, out.get(), 0,
                    out_off.get(), 0);
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
  // (the scans and the sort synchronise the stream when they have to grow these)
  MTSV_TRY(w.scan_tmp.reserve((((size_t)nr + 1 + 2047) / 2048 + 1) * 8));
  MTSV_TRY(w.sort.reserve(nr + 1));
  PartsView pv;
  uint64_t* d_tot = nullptr;
  MTSV_TRY(prepare_parts(w, st, n_parts, d_hits, d_counts, nr, &pv, &d_tot));
  MTSV_TRY(merge_parts_count(w, st, pv, nr, hit_cap, d_n_out));
  taxid_merge_write(st, w.keys.as<uint64_t>(), w.comb_off.as<uint32_t>(), w.off_out32.as<uint32_t>(), nr, out, 0,
                    out_off, 0);
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
  CollapseScratch w;
  DevBuf comb, flag;
  PartsView pv;
  uint64_t* d_tot = nullptr;
  MTSV_TRY(prepare_parts(w, st, n_parts, d_hits, d_counts, nr, &pv, &d_tot));
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
                  w.comb_off.as<uint32_t>(), comb.as<mtsvgpu_hit>());
    }
    MTSV_LAUNCH(collapse_long_flag_kernel, wgrid, 128, 0, st, comb.as<mtsvgpu_hit>(), w.comb_off.as<uint32_t>(), nr,
                flag.as<uint8_t>(), w.cnt_out.as<uint32_t>());
  }
  MTSV_TRY(exclusive_scan_u32(w.cnt_out.as<uint32_t>(), w.off_out32.as<uint32_t>(), nr, w.scan_tmp, d_tot, st));
  MTSV_CUDA_TRY(cudaMemcpyAsync(&h_tot, d_tot, 8, cudaMemcpyDeviceToHost, st));
  MTSV_CUDA_TRY(cudaStreamSynchronize(st));
  DevPtr<mtsvgpu_hit> out;
  DevPtr<uint64_t> out_off;
  MTSV_TRY(dev_alloc(out, h_tot + 1));
  MTSV_TRY(dev_alloc(out_off, (uint64_t)nr + 1));
  MTSV_LAUNCH(collapse_long_write_kernel, wgrid, 128, 0, st, comb.as<mtsvgpu_hit>(), w.comb_off.as<uint32_t>(),
              flag.as<uint8_t>(), w.off_out32.as<uint32_t>(), nr, out.get(), out_off.get());
  cudaError_t e = cudaStreamSynchronize(st);
  if (e != cudaSuccess) return set_error(MTSVGPU_ECUDA, "collapse (taxid-gi): %s", cudaGetErrorString(e));
  *d_out = out.release();
  *d_out_off = out_off.release();
  *n_out = h_tot;
  return 0;
}

}  // namespace mtsv
