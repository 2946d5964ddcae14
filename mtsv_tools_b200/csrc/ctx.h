// ctx.h — host-side handle, error plumbing and device-buffer helpers shared by index.cu,
// binner.cu and capi.cu.
#pragma once
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdint.h>

#include <algorithm>
#include <atomic>
#include <memory>
#include <string>
#include <vector>

#include "../../include/mtsv_b200.h"
#include "core.cuh"

namespace mtsv {

int set_error(int code, const char* fmt, ...);
unsigned sm_count();  // SMs of the current device (cached)
extern std::atomic<uint64_t> g_launches;

#define MTSV_CUDA_TRY(expr)                                                                  \
  do {                                                                                       \
    cudaError_t e_ = (expr);                                                                 \
    if (e_ != cudaSuccess)                                                                   \
      return ::mtsv::set_error(MTSVGPU_ECUDA, "%s: %s (%s:%d)", #expr, cudaGetErrorString(e_), \
                               __FILE__, __LINE__);                                          \
  } while (0)

#define MTSV_TRY(expr)          \
  do {                          \
    int rc_ = (expr);           \
    if (rc_ != 0) return rc_;   \
  } while (0)

// every kernel launch of the library goes through this so gpu_launches can be reported
#define MTSV_LAUNCH(kernel, grid, block, smem, stream, ...)       \
  do {                                                            \
    kernel<<<(grid), (block), (smem), (stream)>>>(__VA_ARGS__);   \
    ::mtsv::g_launches.fetch_add(1, std::memory_order_relaxed);   \
  } while (0)

// owners of device and page-locked memory
struct CudaFree {
  void operator()(void* p) const;
};
struct CudaFreeHost {
  void operator()(void* p) const;
};
template <typename T>
using DevPtr = std::unique_ptr<T, CudaFree>;
template <typename T>
using PinnedPtr = std::unique_ptr<T, CudaFreeHost>;

// The library's only allocators (cudaMalloc, cudaHostAlloc).  A failure clears the runtime's last error, so that it
// cannot fail a later, unrelated call, and returns MTSVGPU_ENOMEM.
int device_alloc(void** p, size_t bytes);
int pinned_alloc(void** p, size_t bytes, unsigned flags);

// `count ? count : 1` elements of T; the bytes are added to *acc
template <typename T>
int dev_alloc(DevPtr<T>& p, uint64_t count, uint64_t* acc = nullptr) {
  const size_t bytes = (size_t)(count ? count : 1) * sizeof(T);
  void* q = nullptr;
  MTSV_TRY(device_alloc(&q, bytes));
  p.reset(static_cast<T*>(q));
  if (acc) *acc += bytes;
  return 0;
}
template <typename T>
int pinned_alloc(PinnedPtr<T>& p, uint64_t count, unsigned flags = cudaHostAllocDefault) {
  void* q = nullptr;
  MTSV_TRY(pinned_alloc(&q, (size_t)(count ? count : 1) * sizeof(T), flags));
  p.reset(static_cast<T*>(q));
  return 0;
}

// owners of streams and events
struct CudaStreamDestroy {
  void operator()(cudaStream_t s) const;
};
struct CudaEventDestroy {
  void operator()(cudaEvent_t e) const;
};
using Stream = std::unique_ptr<CUstream_st, CudaStreamDestroy>;
using Event = std::unique_ptr<CUevent_st, CudaEventDestroy>;

// The library's only stream and event creation: a non-blocking stream; an event with cudaEventCreateWithFlags's
// flags.  A failure clears the runtime's last error and returns MTSVGPU_ECUDA.
int stream_create(Stream& s);
int event_create(Event& e, unsigned flags);
// grows `pool` to at least n events created with `flags`
int events_reserve(std::vector<Event>& pool, size_t n, unsigned flags);

// MTSVGPU_ENODEVICE without a device, MTSVGPU_EINVAL for a number outside [0, count), else cudaSetDevice
int use_device(int device);

// growable device allocation
struct DevBuf {
  DevPtr<uint8_t> p;
  size_t cap = 0;
  int reserve(size_t bytes);  // contents are NOT preserved
  template <typename T>
  T* as() const {
    return reinterpret_cast<T*>(p.get());
  }
};

// segsort.cu
// Sorts keys[seg_off[q] .. + seg_cnt[q]) ascending for each segment q < nq with more than min_count keys.  The sort
// reserves its scratch, synchronising the stream first when it has to grow; reserve it in advance to avoid that.
struct SegSortScratch {
  DevBuf lists;   // three work lists of nq segments: one warp, one CTA in shared memory, one CTA in global memory
  DevBuf counts;  // their lengths
  int reserve(uint32_t nq);
};
int run_segmented_sort(cudaStream_t st, SegSortScratch& s, uint64_t* keys, const uint32_t* seg_off,
                       const uint32_t* seg_cnt, uint32_t nq, uint32_t min_count);

struct BatchCounters {  // device-side scalars of one sub-batch
  unsigned long long total_slots, total_hits, total_cands, total_out;
  unsigned int max_len, overflow, bad_offsets, n_heavy, heavy_cursor, n_monster;
  unsigned int inv_min_len;  // ~(shortest read) so that a zeroed struct means "no read seen"
  unsigned int n_ssw_full, n_over_len;  // candidates of reads >= 254 bases that needed the full SW matrices; reads over the length limit
  unsigned long long verified[2];  // two-round verification: candidates verified in round 1 / round 2
  unsigned long long rank_steps[32], window_bytes[32];  // profiling only; spread to avoid one hot address
  unsigned long long total_taxhits;  // assignments output: merged (TaxID, edit) records of the sub-batch
};


// device-resident index (one per GPU)
struct DeviceIndex {
  int device = 0;
  uint64_t n = 0;  // rows / text length incl. '$'
  // FM-index
  DevPtr<FmBlock> blocks;
  DevPtr<SuperCounts> super;
  DevPtr<uint32_t> n_before;
  uint64_t n_blocks = 0, n_super = 0;
  uint32_t C[5] = {0, 0, 0, 0, 0};
  DevPtr<uint32_t> d_C;  // device copy of C
  uint32_t dollar_row = 0;
  // suffix array at the device rate
  DevPtr<uint32_t> sa;
  uint32_t sa_rate = 1;
  uint64_t sa_len = 0;
  uint64_t file_sa_rate = 0;
  // k-mer interval table
  DevPtr<uint2> ktab;
  uint32_t ktab_k = 0;
  uint32_t ktab_direct = 0;  // unique k-mers hold (text position, preceding symbols) instead of their SA interval
  // reference text (bytes, as in the file) and bins (SoA)
  DevPtr<uint8_t> text;
  DevPtr<uint64_t> text4;  // the same text as 4-bit match classes (0..3 = A,C,G,T, 4 = anything else), 16 per word
  uint64_t text4_words = 0;
  DevPtr<uint32_t> bin_start, bin_end, bin_tax, bin_gi;
  uint64_t n_bins = 0;
  uint64_t n_taxids = 0;  // distinct TaxIDs among the bins (== n_bins: no TaxID has a second sequence)
  uint64_t device_bytes = 0;
  double load_seconds = 0, relayout_seconds = 0, build_seconds = 0;

  FmView fm_view() const {
    FmView v;
    v.blocks = blocks.get();
    v.super = super.get();
    v.n_before = n_before.get();
    v.C = d_C.get();
    v.n = (uint32_t)n;
    v.dollar_row = dollar_row;
    return v;
  }
  SaView sa_view() const { return SaView{sa.get(), sa_rate}; }
  KtabView ktab_view() const { return KtabView{ktab.get(), ktab_k, ktab_direct, text.get()}; }
  BinsView bins_view() const {
    return BinsView{bin_start.get(), bin_end.get(), bin_tax.get(), bin_gi.get(), (uint32_t)n_bins};
  }
};

enum Stage {
  ST_PREP = 0,    // slot counting + scans
  ST_SEARCH = 1,  // backward search of all seed slots
  ST_SELECT = 2,  // tune/max-hits replay + hit offsets
  ST_LOCATE = 3,  // SA lookup / LF walks
  ST_SORT = 4,    // segmented sort of seed hits
  ST_COALESCE = 5,
  ST_RANK = 6,    // candidate ranking + compaction
  ST_VERIFY = 7,  // bit-vector edit distance
  ST_EMIT = 8,    // selection, compaction of hits
  ST_COPY = 9,    // H2D / D2H inside bin_batch
  ST_N = 10
};
static_assert(ST_N <= MTSVGPU_N_STAGES, "stage table too small");

struct BatchWorkspace {
  // per query (nq+1 where a scan is involved)
  DevBuf slot_off, q_nseeds, q_nhits, hit_off, q_ncand, cand_off, q_nout, out_off;
  // per slot
  DevBuf slot_q, slot_lo, slot_cnt, slot_hoff;
  DevBuf pack_rel;  // packed input with ragged lengths: byte offset of each read's record inside the sub-batch
  // per seed hit
  DevBuf hit_keys, cand_sparse, cand_stage;
  // per candidate (dense)
  DevBuf cand_dense, cand_q, cand_edit, hit_tmp, cand_flag, cand_order, cand_end, ssw_list, ssw_scratch;
  DevBuf cand_lead, cand_order2;  // two-round verification: leader of each candidate, compacted visiting order
  // bit-plane encoded reads of the sub-batch
  DevBuf enc;
  // scan scratch, counters, coalesce's heavy and monster lists, the segmented sort's scratch
  DevBuf scan_tmp, counters, worklist;
  SegSortScratch sort;
  // whole-batch results (device-resident API): mtsvgpu_hit or mtsvgpu_taxhit records
  DevBuf out_hits, out_hit_off;
  // staged inputs for the host API
  DevBuf d_seqs, d_seq_off;
};

// One in-flight device sub-batch.  A batch call alternates its slices between two lanes (own stream, own
// scratch, own host thread): while one lane's host thread waits for the scalars of a stage, the other lane's
// kernels keep the device busy, and the tails of memory-bound and ALU-bound kernels of different slices overlap.
struct Lane {
  cudaStream_t stream = nullptr;   // lane 0: the handle's stream; lane 1: the handle's lane1_stream
  BatchWorkspace* ws = nullptr;    // scratch of the lane (results and staged inputs live in the handle's ws)
  PinnedPtr<BatchCounters> h_ctr;  // mapped: sub-batch scalars published by the device
  BatchCounters* h_ctr_dev = nullptr;
  Event emit_event;                // recorded after each append to the batch output
  std::vector<Event> ev_pool;      // per-stage timing (profiling)
};

// What a batch call returns, CSR by read: the Hit records of every strand (mtsvgpu_hit), or per read each TaxID once
// with its minimum edit over both strands, by ascending TaxID (mtsvgpu_taxhit: the default results format)
enum class BatchOutput { Hits, TaxHits };

// What the host API knows about a batch that bin_batch_device computes from device buffers it is still filling (none
// for device-resident input: a null source).  The uploader writes pack_base[i] before it lets wait_slice(i) return.
struct BatchSource {
  const uint64_t* seq_off = nullptr;  // host copy of the device seq_off
  std::vector<uint64_t> bounds;       // read boundaries of the slices (slice_bounds)
  std::vector<uint64_t> pack_base;    // packed records: byte offset of each slice's first record; empty: raw bytes
  // before slice i is computed: wait until it has landed, ordering `stream` after its upload
  virtual int wait_slice(uint64_t i, cudaStream_t stream) = 0;
  // after a sub-batch's results are enqueued on `stream` (records of the call's BatchOutput)
  virtual int results(uint64_t first_hit, uint64_t n_hits, uint64_t first_read, uint64_t n_reads,
                      cudaStream_t stream) = 0;
};

}  // namespace mtsv

struct mtsvgpu_index {
  mtsv::DeviceIndex ix;
  mtsvgpu_index_opts opts{};
  mtsv::Stream own_stream;
  cudaStream_t stream = nullptr;  // own_stream or the caller's (mtsvgpu_set_stream)
  bool profiling = false;
  mtsv::BatchWorkspace ws;   // lane 0 scratch + the batch results + the staged inputs of the host API
  mtsv::BatchWorkspace ws1;  // lane 1 scratch
  mtsv::Lane lanes[2];
  mtsv::Stream lane1_stream;
  mtsv::Event fork_event, join_event;
  mtsvgpu_batch_stats stats{};  // of the last batch call
  // host API: copy streams, per-sub-batch "input landed" events, pinned result buffers
  mtsv::Stream copy_in_stream;
  std::vector<mtsv::Event> in_events;
  mtsv::Stream copy_out_stream;
  mtsv::Event out_event;
  std::vector<mtsv::Event> trace_events;  // MTSV_B200_TRACE: the slice timeline
  mtsv::PinnedPtr<uint8_t> pin_hits;
  size_t pin_hits_cap = 0;
  mtsv::PinnedPtr<uint8_t> pin_off;
  size_t pin_off_cap = 0;
};

namespace mtsv {
// the fields of an MGIndex (src/index.rs:60-68) as index.cu takes them
struct IndexParts {
  const uint8_t* text = nullptr;  // n bytes incl. the final '$'; host memory unless text_on_device
  bool text_on_device = false;
  uint64_t n = 0;
  const mtsvgpu_bin* bins = nullptr;  // host
  uint64_t n_bins = 0;
  const uint8_t* bwt = nullptr;  // n bytes; when bwt_on_device the allocation must extend 64 bytes past n
  bool bwt_on_device = false;
  const uint64_t* sa_sample = nullptr;  // host: suffix array rows 0, s, 2s, ... (the file's sample)
  uint64_t sa_sample_len = 0;
  uint64_t sa_rate = 0;  // s
  DevPtr<uint32_t> d_sa_full;  // instead of sa_sample: the complete suffix array on the device (adopted)
};
// index.cu
int index_assemble(IndexParts parts, int device, const mtsvgpu_index_opts* opts, mtsvgpu_index** out);
int index_from_host_parts(const uint8_t* text, uint64_t n, const mtsvgpu_bin* bins, uint64_t n_bins,
                          const uint8_t* bwt, const uint64_t* sa_sample, uint64_t sa_sample_len,
                          uint64_t sa_rate, int device, const mtsvgpu_index_opts* opts,
                          mtsvgpu_index** out);
int index_open_file(const char* path, int device, const mtsvgpu_index_opts* opts,
                    mtsvgpu_index** out);
void index_destroy(mtsvgpu_index* h);
// build.cu
int index_build(const uint8_t* seqs, const uint64_t* seq_off, const uint32_t* gi, const uint32_t* tax_id, uint64_t n_seqs,
                int device, const mtsvgpu_index_opts* opts, mtsvgpu_index** out);
int index_write(mtsvgpu_index* h, const char* path, uint32_t sample_interval, uint32_t sa_sample);
int index_export(mtsvgpu_index* h, uint8_t* text_out, uint8_t* bwt_out, uint64_t* sample_out, uint32_t sa_sample);
int suffix_array_host(int device, const uint8_t* text, uint64_t n, uint32_t* sa_out, uint8_t* bwt_out);
// binner.cu
int bin_batch_device(mtsvgpu_index* h, const uint8_t* d_seqs, const uint64_t* d_seq_off,
                     uint64_t n_reads, BatchSource* src, BatchOutput kind,
                     const mtsvgpu_params* params, const void** d_out,
                     const uint64_t** d_out_off, uint64_t* n_out);
int backward_search_batch(mtsvgpu_index* h, const uint8_t* pats, uint32_t pat_len, uint64_t n_pats,
                          uint64_t* lower, uint64_t* upper);
int locate_batch(mtsvgpu_index* h, const uint64_t* rows, uint64_t n_rows, uint64_t* pos);
int edit_distance_batch(int device, const uint8_t* pats, const uint64_t* pat_off,
                        const uint8_t* texts, const uint64_t* text_off, uint64_t n_pairs,
                        uint32_t* edits);
// collapse.cu
// The (TaxID, edit) merge of keys tax << 32 | edit, read r's keys at [seg_off[r], seg_off[r] + seg_cnt[r])
// (seg_off[n_reads] = the end).  taxid_merge_count sorts each segment (none when key_bound, a bound on the keys, is
// 0), counts its records into tax_cnt and scans them into tax_off; the record total goes to *d_total.
// taxid_merge_write then writes read r's records to out[out_base + tax_off[r]] on and out_off[read_base + r] =
// out_base + tax_off[r] for r = 0 .. n_reads.
int taxid_merge_count(cudaStream_t st, SegSortScratch& sort, DevBuf& scan_tmp, uint64_t* keys, const uint32_t* seg_off,
                      const uint32_t* seg_cnt, uint32_t n_reads, uint64_t key_bound, uint32_t* tax_cnt,
                      uint32_t* tax_off, uint64_t* d_total);
void taxid_merge_write(cudaStream_t st, const uint64_t* keys, const uint32_t* seg_off, const uint32_t* tax_off,
                       uint32_t n_reads, mtsvgpu_taxhit* out, uint64_t out_base, uint64_t* out_off, uint64_t read_base);
int collapse_device(int device, cudaStream_t st, uint32_t n_parts, const mtsvgpu_hit* const* d_hits,
                    const uint32_t* const* d_counts, uint64_t n_reads, mtsvgpu_taxhit** d_out,
                    uint64_t** d_out_off, uint64_t* n_out);
int collapse_device_long(int device, cudaStream_t st, uint32_t n_parts, const mtsvgpu_hit* const* d_hits,
                         const uint32_t* const* d_counts, uint64_t n_reads, mtsvgpu_hit** d_out,
                         uint64_t** d_out_off, uint64_t* n_out);
struct CollapseScratch {
  DevBuf offs[16], total, comb_off, comb_total, keys, scan_tmp, cnt_out, off_out32;  // comb_total: one u64
  SegSortScratch sort;
};
int collapse_taxid_async(CollapseScratch& w, cudaStream_t st, uint32_t n_parts, const mtsvgpu_hit* const* d_hits,
                         const uint32_t* const* d_counts, uint32_t nr, uint64_t hit_cap, mtsvgpu_taxhit* out,
                         uint64_t* out_off, uint64_t* d_n_out);
// chunked.cu
int comm_create(int device, uint32_t rank, uint32_t world, uint64_t max_local_reads, uint64_t max_hits_per_source,
                mtsvgpu_comm** out, uint8_t* handle_out);
int comm_connect(mtsvgpu_comm* c, const uint8_t* all_handles);
void comm_destroy(mtsvgpu_comm* c);
int bin_batch_chunked(mtsvgpu_index* h, mtsvgpu_comm* c, const uint8_t* d_seqs, const uint64_t* d_seq_off,
                      uint64_t n_reads, const mtsvgpu_params* params, uint64_t* first_read, uint64_t* n_local_reads,
                      const mtsvgpu_taxhit** d_out, const uint64_t** d_out_off, uint64_t* n_out);
// scan.cuh users
int exclusive_scan_u32(const uint32_t* d_in, uint32_t* d_out, uint64_t n, DevBuf& tmp,
                       uint64_t* d_total, cudaStream_t stream);
}  // namespace mtsv
