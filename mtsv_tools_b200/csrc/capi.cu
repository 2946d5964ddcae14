// capi.cu — the extern "C" surface declared in include/mtsv_b200.h.
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <chrono>
#include <thread>
#include <stdio.h>

#include "ctx.h"

namespace mtsv {
const char* last_error_cstr();
}

using namespace mtsv;

extern "C" {

const char* mtsvgpu_version(void) { return "mtsv_b200 0.1.0 (sm_100a)"; }
const char* mtsvgpu_last_error(void) { return last_error_cstr(); }
uint64_t mtsvgpu_launch_count(void) { return g_launches.load(); }
void mtsvgpu_free(void* p) { free(p); }

int mtsvgpu_index_open(const char* index_path, int device, const mtsvgpu_index_opts* opts,
                       mtsvgpu_index** out) {
  return index_open_file(index_path, device, opts, out);
}

int mtsvgpu_index_from_parts(const uint8_t* text, uint64_t n, const mtsvgpu_bin* bins, uint64_t n_bins,
                             const uint8_t* bwt, const uint64_t* sa_sample, uint64_t sa_sample_len,
                             uint64_t sa_rate, int device, const mtsvgpu_index_opts* opts,
                             mtsvgpu_index** out) {
  return index_from_host_parts(text, n, bins, n_bins, bwt, sa_sample, sa_sample_len, sa_rate, device, opts,
                               out);
}

int mtsvgpu_index_build(const uint8_t* seqs, const uint64_t* seq_off, const uint32_t* gi, const uint32_t* tax_id,
                        uint64_t n_seqs, int device, const mtsvgpu_index_opts* opts, mtsvgpu_index** out) {
  return index_build(seqs, seq_off, gi, tax_id, n_seqs, device, opts, out);
}

int mtsvgpu_index_write(mtsvgpu_index* ix, const char* path, uint32_t sample_interval, uint32_t sa_sample) {
  return index_write(ix, path, sample_interval, sa_sample);
}

int mtsvgpu_index_export(mtsvgpu_index* ix, uint8_t* text_out, uint8_t* bwt_out, uint64_t* sa_sample_out,
                         uint32_t sa_sample) {
  return index_export(ix, text_out, bwt_out, sa_sample_out, sa_sample);
}

int mtsvgpu_suffix_array(int device, const uint8_t* text, uint64_t n, uint32_t* sa_out, uint8_t* bwt_out) {
  return suffix_array_host(device, text, n, sa_out, bwt_out);
}

void mtsvgpu_index_close(mtsvgpu_index* ix) { index_destroy(ix); }

int mtsvgpu_index_get_info(const mtsvgpu_index* ix, mtsvgpu_index_info* info) {
  if (!ix || !info) return set_error(MTSVGPU_EINVAL, "null argument");
  info->text_len = ix->ix.n;
  info->n_bins = ix->ix.n_bins;
  info->file_sa_rate = ix->ix.file_sa_rate;
  info->device_sa_rate = ix->ix.sa_rate;
  info->ktab_k = ix->ix.ktab_k;
  info->device_bytes = ix->ix.device_bytes;
  info->dollar_row = ix->ix.dollar_row;
  info->load_seconds = ix->ix.load_seconds;
  info->relayout_seconds = ix->ix.relayout_seconds;
  info->build_seconds = ix->ix.build_seconds;
  return 0;
}

int mtsvgpu_set_stream(mtsvgpu_index* ix, void* cuda_stream) {
  if (!ix) return set_error(MTSVGPU_EINVAL, "index is NULL");
  ix->stream = cuda_stream ? (cudaStream_t)cuda_stream : ix->own_stream;
  return 0;
}

int mtsvgpu_set_profiling(mtsvgpu_index* ix, int on) {
  if (!ix) return set_error(MTSVGPU_EINVAL, "index is NULL");
  ix->profiling = on != 0;
  return 0;
}

int mtsvgpu_last_batch_stats(const mtsvgpu_index* ix, mtsvgpu_batch_stats* stats) {
  if (!ix || !stats) return set_error(MTSVGPU_EINVAL, "null argument");
  *stats = ix->stats;
  return 0;
}

int mtsvgpu_bin_batch_device(mtsvgpu_index* ix, const uint8_t* d_seqs, const uint64_t* d_seq_off,
                             uint64_t n_reads, const mtsvgpu_params* params, const mtsvgpu_hit** d_hits,
                             const uint64_t** d_hit_off, uint64_t* n_hits) {
  return bin_batch_device(ix, d_seqs, d_seq_off, n_reads, nullptr, BatchOutput::Hits, params, (const void**)d_hits,
                          d_hit_off, n_hits);
}

int mtsvgpu_assign_batch_device(mtsvgpu_index* ix, const uint8_t* d_seqs, const uint64_t* d_seq_off, uint64_t n_reads,
                                const mtsvgpu_params* params, const mtsvgpu_taxhit** d_out, const uint64_t** d_out_off,
                                uint64_t* n_out) {
  return bin_batch_device(ix, d_seqs, d_seq_off, n_reads, nullptr, BatchOutput::TaxHits, params, (const void**)d_out,
                          d_out_off, n_out);
}

static int ensure_pinned(PinnedPtr<uint8_t>& p, size_t& cap, size_t bytes) {
  if (bytes <= cap && p) return 0;
  p.reset();
  cap = 0;
  const size_t want = bytes + bytes / 2 + 4096;
  MTSV_TRY(pinned_alloc(p, want));
  cap = want;
  return 0;
}

// Per-call state of bin_batch_host, shared by the uploader thread and the compute lanes
struct HostUpload : BatchSource {
  mtsvgpu_index* ix;
  std::atomic<uint64_t> slices_enqueued{0};  // slices whose upload has been enqueued (uploader thread)
  std::atomic<int> upload_rc{0};
  std::string upload_msg;
  uint64_t out_copied_hits = 0, out_copied_reads = 0;  // prefix already on its way to the pinned buffers
  bool out_overlap_ok = false;
  size_t rec_bytes;  // result records: mtsvgpu_hit or mtsvgpu_taxhit
  // MTSV_B200_TRACE: per-slice timeline (when each slice landed, when its compute started), from the handle's pool
  cudaEvent_t trace_t0 = nullptr;
  const cudaEvent_t* trace_landed = nullptr;
  const cudaEvent_t* trace_started = nullptr;
  HostUpload(mtsvgpu_index* h, size_t rec) : ix(h), rec_bytes(rec) {}
  int upload(const uint8_t* seqs, uint64_t base, uint64_t bytes, uint64_t* h2d_bytes);
  int wait_slice(uint64_t i, cudaStream_t st) override;
  int results(uint64_t first_hit, uint64_t n_hits, uint64_t first_read, uint64_t n_reads, cudaStream_t st) override;
};

int HostUpload::wait_slice(uint64_t i, cudaStream_t st) {
  // the uploader thread enqueues slice after slice; wait (on the host) until slice i's event has been recorded
  while (slices_enqueued.load(std::memory_order_acquire) <= i) {
    if (upload_rc.load(std::memory_order_acquire) != 0) return set_error(upload_rc.load(), "%s", upload_msg.c_str());
    std::this_thread::yield();
  }
  if (i < ix->in_events.size()) MTSV_CUDA_TRY(cudaStreamWaitEvent(st, ix->in_events[i], 0));
  if (trace_started) MTSV_CUDA_TRY(cudaEventRecord(trace_started[i], st));
  return 0;
}

// Results of a finished sub-batch go to the pinned result buffers on the copy-out stream while the next
// sub-batch computes.  Only used when the pinned buffers are known to be large enough (they keep the size
// of earlier batches); otherwise everything is copied at the end.
int HostUpload::results(uint64_t first_hit, uint64_t n_hits, uint64_t first_read, uint64_t n_reads, cudaStream_t st) {
  if (!out_overlap_ok) return 0;
  if ((first_hit + n_hits) * rec_bytes > ix->pin_hits_cap ||
      (first_read + n_reads + 1) * sizeof(uint64_t) > ix->pin_off_cap || first_hit != out_copied_hits ||
      first_read != out_copied_reads) {
    out_overlap_ok = false;  // does not fit / unexpected order: the caller copies everything at the end
    return 0;
  }
  MTSV_CUDA_TRY(cudaEventRecord(ix->out_event, st));
  MTSV_CUDA_TRY(cudaStreamWaitEvent(ix->copy_out_stream, ix->out_event, 0));
  const uint8_t* d_recs = ix->ws.out_hits.as<uint8_t>();
  const uint64_t* d_off = ix->ws.out_hit_off.as<uint64_t>();
  if (n_hits)
    MTSV_CUDA_TRY(cudaMemcpyAsync(ix->pin_hits.get() + first_hit * rec_bytes, d_recs + first_hit * rec_bytes,
                                  n_hits * rec_bytes, cudaMemcpyDeviceToHost, ix->copy_out_stream));
  MTSV_CUDA_TRY(cudaMemcpyAsync((uint64_t*)ix->pin_off.get() + first_read, d_off + first_read,
                                (n_reads + 1) * sizeof(uint64_t), cudaMemcpyDeviceToHost, ix->copy_out_stream));
  out_copied_hits = first_hit + n_hits;
  out_copied_reads = first_read + n_reads;
  return 0;
}

// seq_off of a slice whose reads all have the same length is generated on the device instead of uploaded
// (8 bytes per read: 5 % of the upload of 150-base reads, and the upload is what bounds the host API)
__global__ void fill_offsets_kernel(uint64_t* __restrict__ off, uint64_t first, uint64_t len, uint64_t count) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < count) off[i] = first + i * len;
}
static bool uniform_lengths(const uint64_t* o, uint64_t n_reads) {  // o[0 .. n_reads]
  if (n_reads == 0) return false;
  const uint64_t len = o[1] - o[0];
  uint64_t acc = 0;
  for (uint64_t i = 0; i < n_reads; ++i) acc |= (o[i + 1] - o[i]) ^ len;  // (no early exit: vectorises)
  return acc == 0;
}

// The uploader: enqueues the slices one after the other on the copy-in stream (runs on its own host thread so
// that checking a slice's lengths does not hold up the compute lanes; it stays far ahead of the DMA engine).
int HostUpload::upload(const uint8_t* seqs, uint64_t base, uint64_t bytes, uint64_t* h2d_bytes) {
  MTSV_CUDA_TRY(cudaSetDevice(ix->ix.device));
  BatchWorkspace& ws = ix->ws;
  cudaStream_t cin = ix->copy_in_stream;
  const uint64_t* offs = seq_off;
  const bool packed = !pack_base.empty();
  const uint64_t n_sub = bounds.size() - 1;
  uint64_t pack_at = 0;  // packed input: byte offset of the next slice's first record
  for (uint64_t i = 0; i < n_sub; ++i) {
    uint64_t r0 = bounds[i], r1 = bounds[i + 1];
    if (r1 < r0 || offs[r1] < offs[r0]) return set_error(MTSVGPU_EINVAL, "seq_off is not monotone");
    const uint64_t b0 = offs[r0];
    uint64_t c0 = b0, cn = offs[r1] - b0;  // what is copied: the slice's bases, or its packed records
    const bool uniform = uniform_lengths(offs + r0, r1 - r0);
    if (packed) {
      // the slice's records: 3 * ceil(L / 8) bytes per read (core.cuh "packed reads")
      uint64_t pb = 0;
      if (uniform) {
        pb = (r1 - r0) * (uint64_t)packed_record_bytes((uint32_t)(offs[r0 + 1] - offs[r0]));
      } else {
        for (uint64_t r = r0; r < r1; ++r) {
          if (offs[r + 1] < offs[r]) return set_error(MTSVGPU_EINVAL, "seq_off is not monotone");
          pb += 3 * ((offs[r + 1] - offs[r] + 7) >> 3);
        }
      }
      pack_base[i] = pack_at;
      c0 = pack_at;
      cn = pb;
      pack_at += pb;
    }
    if (c0 + cn > bytes) return set_error(MTSVGPU_EINVAL, "seq_off exceeds the reads buffer");
    // offsets of the slice (r0 .. r1 inclusive) first, then its bases: sub-batch i can start as soon as
    // its own slice has landed
    if (uniform) {
      const uint64_t cnt = r1 - r0 + 1;
      MTSV_LAUNCH(fill_offsets_kernel, (unsigned)((cnt + 255) / 256), 256, 0, cin, ws.d_seq_off.as<uint64_t>() + r0, b0,
                  offs[r0 + 1] - offs[r0], cnt);
    } else {
      MTSV_CUDA_TRY(cudaMemcpyAsync(ws.d_seq_off.as<uint64_t>() + r0, offs + r0, (r1 - r0 + 1) * 8,
                                    cudaMemcpyHostToDevice, cin));
      *h2d_bytes += (r1 - r0 + 1) * 8;
    }
    if (cn)
      MTSV_CUDA_TRY(cudaMemcpyAsync(ws.d_seqs.as<uint8_t>() + c0, seqs + base + c0, cn, cudaMemcpyHostToDevice, cin));
    *h2d_bytes += cn;
    MTSV_CUDA_TRY(cudaEventRecord(ix->in_events[i], cin));
    if (trace_landed) MTSV_CUDA_TRY(cudaEventRecord(trace_landed[i], cin));
    slices_enqueued.store(i + 1, std::memory_order_release);
  }
  return 0;
}

// Host-buffer batch: the reads are uploaded sub-batch by sub-batch on a copy stream while earlier
// sub-batches compute (pass page-locked buffers to get the overlap; pageable ones work, serially).
// pinned_result: 0 = results in malloc'ed memory (mtsvgpu_free), 1 = in the handle's page-locked
// buffers, valid until the next batch call on this handle.  kind: Hit records or merged (TaxID, edit) records.
static int bin_batch_host(mtsvgpu_index* ix, const uint8_t* seqs, const uint64_t* seq_off, uint64_t n_reads,
                          const mtsvgpu_params* params, BatchOutput kind, int pinned_result, void** hits,
                          uint64_t** hit_off, uint64_t* n_hits_out, bool packed = false, uint64_t packed_bytes = 0) {
  if (!ix || !seq_off || !hits || !hit_off) return set_error(MTSVGPU_EINVAL, "null argument");
  *hits = nullptr;
  *hit_off = nullptr;
  MTSV_CUDA_TRY(cudaSetDevice(ix->ix.device));
  cudaStream_t st = ix->stream, cin = ix->copy_in_stream;
  static const bool trace = getenv("MTSV_B200_TRACE") != nullptr;  // host-side phase times on stderr
  auto now = [] { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
  const double t_begin = trace ? now() : 0;
  const uint64_t base = seq_off[0];
  if (seq_off[n_reads] < base) return set_error(MTSVGPU_EINVAL, "seq_off is not monotone");
  const uint64_t bytes = packed ? packed_bytes : seq_off[n_reads] - base;
  if (bytes && !seqs) return set_error(MTSVGPU_EINVAL, "seqs is NULL");
  BatchWorkspace& ws = ix->ws;
  MTSV_TRY(ws.d_seqs.reserve(bytes + 16));
  MTSV_TRY(ws.d_seq_off.reserve((n_reads + 1) * 8));
  std::vector<uint64_t> rebased;
  const uint64_t* offs = seq_off;
  if (base != 0) {
    rebased.resize(n_reads + 1);
    for (uint64_t i = 0; i <= n_reads; ++i) rebased[i] = seq_off[i] - base;
    offs = rebased.data();
  }
  // ---- H2D, pipelined per device sub-batch ----
  const size_t rec = kind == BatchOutput::TaxHits ? sizeof(mtsvgpu_taxhit) : sizeof(mtsvgpu_hit);
  HostUpload up(ix, rec);
  up.seq_off = offs;
  up.bounds = slice_bounds(n_reads, ix->opts.batch_reads, true, true);
  const uint64_t n_sub = up.bounds.size() - 1;
  if (packed) up.pack_base.assign(n_sub, 0);
  while (ix->in_events.size() < n_sub) {
    cudaEvent_t e;
    MTSV_CUDA_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    ix->in_events.push_back(e);
  }
  if (trace) {
    while (ix->trace_events.size() < 2 * n_sub + 1) {
      cudaEvent_t e;
      MTSV_CUDA_TRY(cudaEventCreate(&e));
      ix->trace_events.push_back(e);
    }
    up.trace_t0 = ix->trace_events[0];
    up.trace_landed = ix->trace_events.data() + 1;
    up.trace_started = ix->trace_events.data() + 1 + n_sub;
    MTSV_CUDA_TRY(cudaEventRecord(up.trace_t0, cin));
  }
  uint64_t h2d_bytes = 0;
  std::thread uploader;
  if (n_sub) {
    uploader = std::thread([&] {
      int urc = up.upload(seqs, packed ? 0 : base, bytes, &h2d_bytes);
      if (urc != 0) {
        up.upload_msg = last_error_cstr();
        up.upload_rc.store(urc, std::memory_order_release);
      }
    });
  } else {
    MTSV_CUDA_TRY(cudaMemcpyAsync(ws.d_seq_off.p.get(), offs, 8, cudaMemcpyHostToDevice, cin));
  }
  const double t_enq = trace ? now() : 0;
  // ---- compute (each sub-batch waits for its slice) ----
  const void* d_hits = nullptr;
  const uint64_t* d_hit_off = nullptr;
  uint64_t n_hits = 0;
  // overlap the result copy when the pinned buffers from earlier batches are big enough for this one
  up.out_overlap_ok = pinned_result && ix->pin_hits && ix->pin_off &&
                      (n_reads + 1) * sizeof(uint64_t) <= ix->pin_off_cap;
  // a device-side regrowth of the output buffer would invalidate copies in flight: reserve generously
  if (up.out_overlap_ok) (void)ws.out_hits.reserve(ix->pin_hits_cap);
  int rc = bin_batch_device(ix, ws.d_seqs.as<uint8_t>(), ws.d_seq_off.as<uint64_t>(), n_reads, &up, kind, params,
                            &d_hits, &d_hit_off, &n_hits);
  if (uploader.joinable()) uploader.join();
  ix->stats.h2d_bytes = h2d_bytes;
  if (rc != 0) {
    cudaStreamSynchronize(cin);
    cudaStreamSynchronize(ix->copy_out_stream);
    return rc;
  }
  const double t_comp = trace ? now() : 0;
  MTSV_CUDA_TRY(cudaStreamSynchronize(cin));
  // ---- D2H ----
  void* h_hits = nullptr;
  uint64_t* h_off = nullptr;
  const size_t hb = (n_hits ? n_hits : 1) * rec, ob = (n_reads + 1) * sizeof(uint64_t);
  if (pinned_result) {
    // slices may still be on their way into the buffers ensure_pinned is about to replace
    MTSV_CUDA_TRY(cudaStreamSynchronize(ix->copy_out_stream));
    MTSV_TRY(ensure_pinned(ix->pin_hits, ix->pin_hits_cap, hb));
    MTSV_TRY(ensure_pinned(ix->pin_off, ix->pin_off_cap, ob));
    h_hits = ix->pin_hits.get();
    h_off = (uint64_t*)ix->pin_off.get();
  } else {
    h_hits = malloc(hb);
    h_off = (uint64_t*)malloc(ob);
    if (!h_hits || !h_off) {
      free(h_hits);
      free(h_off);
      return set_error(MTSVGPU_ENOMEM, "host allocation of the result failed");
    }
  }
  cudaError_t e = cudaStreamSynchronize(ix->copy_out_stream);
  // (nothing more to copy when everything was copied slice by slice)
  if (!(pinned_result && up.out_overlap_ok && up.out_copied_hits == n_hits && up.out_copied_reads == n_reads)) {
    if (e == cudaSuccess && n_hits)
      e = cudaMemcpyAsync(h_hits, d_hits, n_hits * rec, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(h_off, d_hit_off, ob, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  }
  if (e != cudaSuccess) {
    if (!pinned_result) {
      free(h_hits);
      free(h_off);
    }
    return set_error(MTSVGPU_ECUDA, "result copy failed: %s", cudaGetErrorString(e));
  }
  *hits = h_hits;
  *hit_off = h_off;
  if (n_hits_out) *n_hits_out = n_hits;
  if (trace) {
    // one write per call, so that the tables of calls on other threads do not interleave with it
    std::string out = "[mtsv_b200 trace] slice: reads, landed at ms, compute started at ms\n";
    char line[256];
    for (uint64_t i = 0; i < n_sub; ++i) {
      float a = 0, b = 0;
      cudaEventElapsedTime(&a, up.trace_t0, up.trace_landed[i]);  // (every slice's events have completed)
      cudaEventElapsedTime(&b, up.trace_t0, up.trace_started[i]);
      snprintf(line, sizeof line, "[mtsv_b200 trace]   %2llu: %8llu  %7.2f  %7.2f\n", (unsigned long long)i,
               (unsigned long long)(up.bounds[i + 1] - up.bounds[i]), a, b);
      out += line;
    }
    snprintf(line, sizeof line, "[mtsv_b200 trace] bin_batch_host: enqueue H2D %.2f ms, compute %.2f ms, tail (D2H "
             "rest) %.2f ms, overlapped D2H %s\n", t_enq - t_begin, t_comp - t_enq, now() - t_comp,
             up.out_overlap_ok ? "yes" : "no");
    fputs((out + line).c_str(), stderr);
  }
  return 0;
}

int mtsvgpu_bin_batch(mtsvgpu_index* ix, const uint8_t* seqs, const uint64_t* seq_off, uint64_t n_reads,
                      const mtsvgpu_params* params, mtsvgpu_hit** hits, uint64_t** hit_off) {
  return bin_batch_host(ix, seqs, seq_off, n_reads, params, BatchOutput::Hits, 0, (void**)hits, hit_off, nullptr);
}

// the pinned-result entry points: results in the handle's page-locked buffers
static int batch_pinned(mtsvgpu_index* ix, const uint8_t* seqs, const uint64_t* seq_off, uint64_t n_reads,
                        const mtsvgpu_params* params, BatchOutput kind, const void** out, const uint64_t** out_off,
                        uint64_t* n_out, bool packed, uint64_t packed_bytes) {
  void* h = nullptr;
  uint64_t* o = nullptr;
  int rc = bin_batch_host(ix, seqs, seq_off, n_reads, params, kind, 1, &h, &o, n_out, packed, packed_bytes);
  if (out) *out = h;
  if (out_off) *out_off = o;
  return rc;
}

int mtsvgpu_bin_batch_pinned(mtsvgpu_index* ix, const uint8_t* seqs, const uint64_t* seq_off, uint64_t n_reads,
                             const mtsvgpu_params* params, const mtsvgpu_hit** hits,
                             const uint64_t** hit_off, uint64_t* n_hits) {
  return batch_pinned(ix, seqs, seq_off, n_reads, params, BatchOutput::Hits, (const void**)hits, hit_off, n_hits,
                      false, 0);
}

int mtsvgpu_bin_batch_packed(mtsvgpu_index* ix, const uint8_t* packed, uint64_t packed_bytes, const uint64_t* seq_off,
                             uint64_t n_reads, const mtsvgpu_params* params, const mtsvgpu_hit** hits,
                             const uint64_t** hit_off, uint64_t* n_hits) {
  return batch_pinned(ix, packed, seq_off, n_reads, params, BatchOutput::Hits, (const void**)hits, hit_off, n_hits,
                      true, packed_bytes);
}

int mtsvgpu_assign_batch_pinned(mtsvgpu_index* ix, const uint8_t* seqs, const uint64_t* seq_off, uint64_t n_reads,
                                const mtsvgpu_params* params, const mtsvgpu_taxhit** out, const uint64_t** out_off,
                                uint64_t* n_out) {
  return batch_pinned(ix, seqs, seq_off, n_reads, params, BatchOutput::TaxHits, (const void**)out, out_off, n_out,
                      false, 0);
}

int mtsvgpu_assign_batch_packed(mtsvgpu_index* ix, const uint8_t* packed, uint64_t packed_bytes,
                                const uint64_t* seq_off, uint64_t n_reads, const mtsvgpu_params* params,
                                const mtsvgpu_taxhit** out, const uint64_t** out_off, uint64_t* n_out) {
  return batch_pinned(ix, packed, seq_off, n_reads, params, BatchOutput::TaxHits, (const void**)out, out_off, n_out,
                      true, packed_bytes);
}

int mtsvgpu_collapse_device(int device, void* stream, uint32_t n_parts, const mtsvgpu_hit* const* d_hits,
                            const uint32_t* const* d_counts, uint64_t n_reads, mtsvgpu_taxhit** d_out,
                            uint64_t** d_out_off, uint64_t* n_out) {
  return collapse_device(device, (cudaStream_t)stream, n_parts, d_hits, d_counts, n_reads, d_out, d_out_off, n_out);
}

int mtsvgpu_collapse_device_taxid_gi(int device, void* stream, uint32_t n_parts, const mtsvgpu_hit* const* d_hits,
                                     const uint32_t* const* d_counts, uint64_t n_reads, mtsvgpu_hit** d_out,
                                     uint64_t** d_out_off, uint64_t* n_out) {
  return collapse_device_long(device, (cudaStream_t)stream, n_parts, d_hits, d_counts, n_reads, d_out, d_out_off,
                              n_out);
}

int mtsvgpu_comm_create(int device, uint32_t rank, uint32_t world, uint64_t max_local_reads,
                        uint64_t max_hits_per_source, mtsvgpu_comm** out, uint8_t* handle_out) {
  return comm_create(device, rank, world, max_local_reads, max_hits_per_source, out, handle_out);
}
int mtsvgpu_comm_connect(mtsvgpu_comm* comm, const uint8_t* all_handles) { return comm_connect(comm, all_handles); }
void mtsvgpu_comm_destroy(mtsvgpu_comm* comm) { comm_destroy(comm); }
int mtsvgpu_bin_batch_chunked(mtsvgpu_index* ix, mtsvgpu_comm* comm, const uint8_t* d_seqs, const uint64_t* d_seq_off,
                              uint64_t n_reads, const mtsvgpu_params* params, uint64_t* first_read,
                              uint64_t* n_local_reads, const mtsvgpu_taxhit** d_out, const uint64_t** d_out_off,
                              uint64_t* n_out) {
  return bin_batch_chunked(ix, comm, d_seqs, d_seq_off, n_reads, params, first_read, n_local_reads, d_out, d_out_off,
                           n_out);
}

void* mtsvgpu_host_alloc(uint64_t bytes) {
  void* p = nullptr;
  cudaError_t e = cudaMallocHost(&p, bytes ? bytes : 1);
  if (e != cudaSuccess) {
    (void)cudaGetLastError();
    set_error(e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver ? MTSVGPU_ENODEVICE : MTSVGPU_ENOMEM,
              "cudaMallocHost(%llu) failed: %s", (unsigned long long)bytes, cudaGetErrorString(e));
    return nullptr;
  }
  return p;
}
void mtsvgpu_host_free(void* p) {
  if (p) cudaFreeHost(p);
}

void mtsvgpu_device_free(void* d_ptr) {
  if (d_ptr) cudaFree(d_ptr);
}

int mtsvgpu_backward_search(mtsvgpu_index* ix, const uint8_t* pats, uint32_t pat_len, uint64_t n_pats,
                            uint64_t* lower, uint64_t* upper) {
  return backward_search_batch(ix, pats, pat_len, n_pats, lower, upper);
}

int mtsvgpu_locate(mtsvgpu_index* ix, const uint64_t* rows, uint64_t n_rows, uint64_t* pos) {
  return locate_batch(ix, rows, n_rows, pos);
}

int mtsvgpu_edit_distance(int device, const uint8_t* pats, const uint64_t* pat_off, const uint8_t* texts,
                          const uint64_t* text_off, uint64_t n_pairs, uint32_t* edits) {
  return edit_distance_batch(device, pats, pat_off, texts, text_off, n_pairs, edits);
}

}  // extern "C"
