// ctx.h — host-side handle, error plumbing and device-buffer helpers shared by index.cu,
// binner.cu and capi.cu.
#pragma once
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdint.h>

#include <algorithm>
#include <atomic>
#include <condition_variable>
#include <mutex>
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

// growable device allocation
struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  int reserve(size_t bytes);  // contents are NOT preserved
  void release();
  template <typename T>
  T* as() const {
    return reinterpret_cast<T*>(p);
  }
};

struct BatchCounters {  // device-side scalars of one sub-batch
  unsigned long long total_slots, total_hits, total_cands, total_out;
  unsigned int max_len, overflow, n_warp, n_medium, n_large, bad_offsets, n_heavy, heavy_cursor, n_monster;
  unsigned int inv_min_len;  // ~(shortest read) so that a zeroed struct means "no read seen"
  unsigned int n_ssw_full, n_over_len;  // candidates of reads >= 254 bases that needed the full SW matrices; reads over the length limit
  unsigned long long verified[2];  // two-round verification: candidates verified in round 1 / round 2
  unsigned long long rank_steps[32], window_bytes[32];  // profiling only; spread to avoid one hot address
};


// device-resident index (one per GPU)
struct DeviceIndex {
  int device = 0;
  uint64_t n = 0;  // rows / text length incl. '$'
  // FM-index
  FmBlock* blocks = nullptr;
  SuperCounts* super = nullptr;
  uint32_t* n_before = nullptr;
  uint64_t n_blocks = 0, n_super = 0;
  uint32_t C[5] = {0, 0, 0, 0, 0};
  uint32_t* d_C = nullptr;  // device copy of C
  uint32_t dollar_row = 0;
  // suffix array at the device rate
  uint32_t* sa = nullptr;
  uint32_t sa_rate = 1;
  uint64_t sa_len = 0;
  uint64_t file_sa_rate = 0;
  // k-mer interval table
  uint2* ktab = nullptr;
  uint32_t ktab_k = 0;
  uint32_t ktab_direct = 0;  // unique k-mers hold (text position, preceding symbols) instead of their SA interval
  // reference text (bytes, as in the file) and bins (SoA)
  uint8_t* text = nullptr;
  uint64_t* text4 = nullptr;  // the same text as 4-bit match classes (0..3 = A,C,G,T, 4 = anything else), 16 per word
  uint64_t text4_words = 0;
  uint32_t *bin_start = nullptr, *bin_end = nullptr, *bin_tax = nullptr, *bin_gi = nullptr;
  uint64_t n_bins = 0;
  uint64_t n_taxids = 0;  // distinct TaxIDs among the bins (== n_bins: no TaxID has a second sequence)
  uint64_t device_bytes = 0;
  double load_seconds = 0, relayout_seconds = 0, build_seconds = 0;

  FmView fm_view() const {
    FmView v;
    v.blocks = blocks;
    v.super = super;
    v.n_before = n_before;
    v.C = d_C;
    v.n = (uint32_t)n;
    v.dollar_row = dollar_row;
    return v;
  }
  SaView sa_view() const { return SaView{sa, sa_rate}; }
  KtabView ktab_view() const { return KtabView{ktab, ktab_k, ktab_direct, text}; }
  BinsView bins_view() const { return BinsView{bin_start, bin_end, bin_tax, bin_gi, (uint32_t)n_bins}; }
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
  // scan scratch, counters, worklists
  DevBuf scan_tmp, counters, worklist;
  // whole-batch results (device-resident API)
  DevBuf out_hits, out_hit_off;
  // staged inputs for the host API
  DevBuf d_seqs, d_seq_off;
  void release_all();
};

// One in-flight device sub-batch.  A batch call alternates its slices between two lanes (own stream, own
// scratch, own host thread): while one lane's host thread waits for the scalars of a stage, the other lane's
// kernels keep the device busy, and the tails of memory-bound and ALU-bound kernels of different slices overlap.
struct Lane {
  cudaStream_t stream = nullptr;     // lane 0: the handle's stream; lane 1: a private non-blocking stream
  BatchWorkspace* ws = nullptr;      // scratch of the lane (results and staged inputs live in the handle's ws)
  BatchCounters* h_ctr = nullptr;    // page-locked, mapped: sub-batch scalars published by the device
  BatchCounters* h_ctr_dev = nullptr;
  cudaEvent_t emit_event = nullptr;  // recorded after each append to the batch output
  bool has_turn = false;             // holds the output turnstile for its current slice
  uint64_t slice = 0;                // index of the slice being processed
  uint64_t chunk_reads = 0;          // reads per launch group; halves when a group overflows the seed-hit cap
  mtsvgpu_batch_stats stats{};
  // event pool for profiling
  std::vector<cudaEvent_t> ev_pool;
  std::vector<std::pair<int, std::pair<cudaEvent_t, cudaEvent_t>>> ev_used;
  size_t ev_next = 0;
};

// What the host API knows about a batch that bin_batch_device computes from device buffers it is still filling (none
// for device-resident input: a null source).  The uploader writes pack_base[i] before it lets wait_slice(i) return.
struct BatchSource {
  const uint64_t* seq_off = nullptr;  // host copy of the device seq_off
  std::vector<uint64_t> bounds;       // read boundaries of the slices (slice_bounds)
  std::vector<uint64_t> pack_base;    // packed records: byte offset of each slice's first record; empty: raw bytes
  // before slice i is computed: wait until it has landed, ordering `stream` after its upload
  virtual int wait_slice(uint64_t i, cudaStream_t stream) = 0;
  // after a sub-batch's results are enqueued on `stream`
  virtual int results(uint64_t first_hit, uint64_t n_hits, uint64_t first_read, uint64_t n_reads,
                      cudaStream_t stream) = 0;
};

}  // namespace mtsv

struct mtsvgpu_index {
  mtsv::DeviceIndex ix;
  mtsvgpu_index_opts opts{};
  cudaStream_t own_stream = nullptr;
  cudaStream_t stream = nullptr;
  bool profiling = false;
  mtsv::BatchWorkspace ws;   // lane 0 scratch + the batch results + the staged inputs of the host API
  mtsv::BatchWorkspace ws1;  // lane 1 scratch
  mtsv::Lane lanes[2];
  cudaStream_t lane1_stream = nullptr;
  cudaEvent_t fork_event = nullptr, join_event = nullptr;
  // slices append to the batch output in order: a turnstile over the slice index
  std::mutex emit_mu;
  std::condition_variable emit_cv;
  uint64_t emit_turn = 0;
  int abort_rc = 0;
  std::string abort_msg;
  mtsvgpu_batch_stats stats{};
  // host API: copy streams, per-sub-batch "input landed" events, pinned result buffers
  cudaStream_t copy_in_stream = nullptr;
  std::vector<cudaEvent_t> in_events;
  cudaStream_t copy_out_stream = nullptr;
  cudaEvent_t out_event = nullptr;
  void* pin_hits = nullptr;
  size_t pin_hits_cap = 0;
  void* pin_off = nullptr;
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
  uint32_t* d_sa_full = nullptr;  // instead of sa_sample: the complete suffix array on the device (adopted)
};
// index.cu
int index_assemble(const IndexParts& parts, int device, const mtsvgpu_index_opts* opts, mtsvgpu_index** out);
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
                     uint64_t n_reads, BatchSource* src,
                     const mtsvgpu_params* params, const mtsvgpu_hit** d_hits,
                     const uint64_t** d_hit_off, uint64_t* n_hits);
int backward_search_batch(mtsvgpu_index* h, const uint8_t* pats, uint32_t pat_len, uint64_t n_pats,
                          uint64_t* lower, uint64_t* upper);
int locate_batch(mtsvgpu_index* h, const uint64_t* rows, uint64_t n_rows, uint64_t* pos);
int edit_distance_batch(int device, const uint8_t* pats, const uint64_t* pat_off,
                        const uint8_t* texts, const uint64_t* text_off, uint64_t n_pairs,
                        uint32_t* edits);
int run_segmented_sort(cudaStream_t st, DevBuf& worklist, uint64_t* keys, const uint32_t* seg_off,
                       const uint32_t* seg_cnt, uint32_t nq, uint32_t min_count, BatchCounters* d_ctr);
int collapse_device(int device, cudaStream_t st, uint32_t n_parts, const mtsvgpu_hit* const* d_hits,
                    const uint32_t* const* d_counts, uint64_t n_reads, mtsvgpu_taxhit** d_out,
                    uint64_t** d_out_off, uint64_t* n_out);
int collapse_device_long(int device, cudaStream_t st, uint32_t n_parts, const mtsvgpu_hit* const* d_hits,
                         const uint32_t* const* d_counts, uint64_t n_reads, mtsvgpu_hit** d_out,
                         uint64_t** d_out_off, uint64_t* n_out);
struct CollapseScratch {
  DevBuf offs[16], total, comb_off, keys, scan_tmp, counters, worklist, cnt_out, off_out32;
  void release_all();
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
