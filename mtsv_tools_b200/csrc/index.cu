// index.cu — load an mtsv-build `.index` (bincode 1.3.3 dump of MGIndex, src/io.rs:115-132,
// src/index.rs:60-68) and re-lay it out for the B200: 2-bit BWT sectors with interleaved
// occurrence counts, dense(r) suffix array, k-mer interval table.  Nothing is rebuilt from the
// text: the file's BWT and suffix-array samples are the inputs.
#include <errno.h>
#include <fcntl.h>
#include <math.h>
#include <stdlib.h>
#include <string.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>

#include <chrono>

#include "ctx.h"

namespace mtsv {

// ---------------------------------------------------------------------------------------------
// kernel A1: byte BWT -> FmBlock sectors (+ per-superblock totals)
//   one CUDA block of 512 threads = one superblock (512 sectors, 32768 rows)
//   HBM-streaming: reads 1 B/row, writes 0.5 B/row
// ---------------------------------------------------------------------------------------------
struct PackDiag {
  unsigned long long n_dollar;
  unsigned long long dollar_row;
  unsigned long long n_other;
  unsigned long long sa_mismatch;
  unsigned long long rows_seen;
};

constexpr uint32_t kMaxLfWalk = 1u << 22;  // no valid index has an LF walk between samples this long

__device__ __forceinline__ uint64_t warp_incl_u64(uint64_t v) {
  const unsigned lane = threadIdx.x & 31;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    uint64_t o = __shfl_up_sync(0xffffffffu, v, d);
    if (lane >= (unsigned)d) v += o;
  }
  return v;
}

__global__ void __launch_bounds__(kBlocksPerSuper) fm_pack_kernel(
    const uint8_t* __restrict__ bwt, uint64_t n, uint64_t n_blocks, FmBlock* __restrict__ blocks,
    uint32_t* __restrict__ n_before, uint32_t* __restrict__ super_tot /*[n_super][5]*/,
    PackDiag* __restrict__ diag) {
  __shared__ uint64_t w_acgt[16];
  __shared__ uint64_t w_n[16];
  const uint64_t blk = (uint64_t)blockIdx.x * kBlocksPerSuper + threadIdx.x;
  const uint64_t row0 = blk * kRowsPerBlock;
  uint64_t lo = 0, hi = 0, exc = 0;
  uint32_t cnt[5] = {0, 0, 0, 0, 0};
  if (blk < n_blocks && row0 < n) {
    // 64 rows = 4 x 16-byte loads (the staging buffer is padded by 64 bytes, rows >= n are masked)
    uint32_t w[16];
    const uint4* src = reinterpret_cast<const uint4*>(bwt + row0);
#pragma unroll
    for (int v = 0; v < 4; ++v) {
      uint4 x = __ldg(src + v);
      w[4 * v + 0] = x.x;
      w[4 * v + 1] = x.y;
      w[4 * v + 2] = x.z;
      w[4 * v + 3] = x.w;
    }
    const int valid = (int)(n - row0 < 64 ? n - row0 : 64);
#pragma unroll
    for (int j = 0; j < 64; ++j) {
      if (j < valid) {
        uint32_t c = text_code((uint8_t)((w[j >> 2] >> ((j & 3) * 8)) & 0xff));
        if (c < 4) {
          lo |= (uint64_t)(c & 1) << j;
          hi |= (uint64_t)(c >> 1) << j;
          cnt[c]++;
        } else {
          exc |= 1ull << j;
          if (c == SYM_N) {
            cnt[4]++;
          } else if (c == SYM_DOLLAR) {
            atomicAdd(&diag->n_dollar, 1ull);
            atomicExch(&diag->dollar_row, (unsigned long long)(row0 + j));
          } else {
            atomicAdd(&diag->n_other, 1ull);
          }
        }
      }
    }
  }
  // block-wide exclusive scan of the five counters (A,C,G,T packed 16 bits each; N separately)
  uint64_t packed = (uint64_t)cnt[0] | ((uint64_t)cnt[1] << 16) | ((uint64_t)cnt[2] << 32) |
                    ((uint64_t)cnt[3] << 48);
  uint64_t nn = cnt[4];
  const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint64_t inc = warp_incl_u64(packed), ninc = warp_incl_u64(nn);
  if (lane == 31) {
    w_acgt[warp] = inc;
    w_n[warp] = ninc;
  }
  __syncthreads();
  // totals of a full superblock can reach 32768 per symbol: still < 65536, so 16-bit lanes hold
  // every *exclusive* prefix; the inclusive grand total is accumulated in 32 bits below.
  uint64_t base = 0, nbase = 0;
  for (unsigned w = 0; w < warp; ++w) {
    base += w_acgt[w];
    nbase += w_n[w];
  }
  uint64_t ex = base + inc - packed, nex = nbase + ninc - nn;
  if (blk < n_blocks) {
    uint4* dst = reinterpret_cast<uint4*>(blocks + blk);
    dst[0] = make_uint4((uint32_t)ex, (uint32_t)(ex >> 32), (uint32_t)exc, (uint32_t)(exc >> 32));
    dst[1] = make_uint4((uint32_t)lo, (uint32_t)(lo >> 32), (uint32_t)hi, (uint32_t)(hi >> 32));
    n_before[blk] = (uint32_t)nex;  // relative for now; fm_finish_kernel adds the superblock base
  }
  if (threadIdx.x == kBlocksPerSuper - 1) {
    // inclusive totals: exclusive prefix of the last thread + its own counts (no 16-bit overflow
    // because each field is added in 32 bits here)
    uint32_t* t = super_tot + (uint64_t)blockIdx.x * 5;
    t[0] = (uint32_t)(ex & 0xffff) + cnt[0];
    t[1] = (uint32_t)((ex >> 16) & 0xffff) + cnt[1];
    t[2] = (uint32_t)((ex >> 32) & 0xffff) + cnt[2];
    t[3] = (uint32_t)((ex >> 48) & 0xffff) + cnt[3];
    t[4] = (uint32_t)nex + cnt[4];
  }
}

// kernel A2: exclusive scan over superblock totals (tiny: n/32768 entries), C[] table
__global__ void fm_super_scan_kernel(const uint32_t* __restrict__ super_tot, uint64_t n_super,
                                     SuperCounts* __restrict__ super, uint32_t* __restrict__ super_n,
                                     unsigned long long* __restrict__ totals /*[5]*/) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  unsigned long long run[5] = {0, 0, 0, 0, 0};
  for (uint64_t s = 0; s < n_super; ++s) {
    SuperCounts sc;
    for (int a = 0; a < 4; ++a) sc.c[a] = (uint32_t)run[a];
    super[s] = sc;
    super_n[s] = (uint32_t)run[4];
    for (int a = 0; a < 5; ++a) run[a] += super_tot[s * 5 + a];
  }
  for (int a = 0; a < 5; ++a) totals[a] = run[a];
}

__global__ void fm_finish_kernel(uint32_t* __restrict__ n_before, uint64_t n_blocks,
                                 const uint32_t* __restrict__ super_n) {
  uint64_t blk = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (blk < n_blocks) n_before[blk] += super_n[blk / kBlocksPerSuper];
}

// ---------------------------------------------------------------------------------------------
// kernel A3: suffix-array densification.  One thread per sample of the file (row i*s): walk LF
// from the sampled row, assigning SA[LF^j(row)] = sample - j, until the next sampled row.  Every
// row is visited by exactly one walk, so a full SA costs n LF steps in total (not n*s/2).
// Random-access bound: one FmBlock sector + one 4-byte scattered store per step.
// ---------------------------------------------------------------------------------------------
__global__ void sa_densify_kernel(FmView fm, const uint64_t* __restrict__ sample, uint64_t n_sample,
                                  uint32_t s_file, uint32_t rate, uint32_t* __restrict__ sa,
                                  PackDiag* __restrict__ diag) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_sample) return;
  uint32_t row = (uint32_t)(i * s_file);
  uint32_t pos = (uint32_t)sample[i];
  if (row % rate == 0) sa[row / rate] = pos;
  // The walk also runs when rate == s_file: it proves that every row reaches a sample (a corrupt
  // BWT can contain LF cycles that would hang locate), counted in diag->rows_seen.
  unsigned long long seen = 1;
  for (uint32_t step = 0;; ++step) {
    if (step >= kMaxLfWalk) {
      atomicAdd(&diag->sa_mismatch, 1ull);
      break;
    }
    FmBlock b = load_block(fm.blocks + (row >> 6));
    uint32_t c = fm_symbol(fm, b, row);
    if (c == SYM_DOLLAR) {
      if (pos != 0) atomicAdd(&diag->sa_mismatch, 1ull);
      break;
    }
    row = fm_lf(fm, c, b, row);
    pos -= 1;
    if (row % s_file == 0) {
      if ((uint32_t)sample[row / s_file] != pos) atomicAdd(&diag->sa_mismatch, 1ull);
      break;
    }
    ++seen;
    if (row % rate == 0) sa[row / rate] = pos;
  }
  atomicAdd(&diag->rows_seen, seen);
}

// ---------------------------------------------------------------------------------------------
// kernel A4: k-mer interval table, built level by level: interval(c.X) = step(interval(X), c)
// ---------------------------------------------------------------------------------------------
__global__ void ktab_level_kernel(FmView fm, const uint2* __restrict__ cur, uint2* __restrict__ next,
                                  uint32_t t /* length of the k-mers in `next` */) {
  // key of a t-mer = lo | hi << t (base j at bit j).  c.X prepends base c: X's planes shift up by one.
  uint64_t key = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (key >= (1ull << (2 * t))) return;
  uint64_t lo = key & ((1ull << t) - 1), hi = key >> t;
  uint32_t c = (uint32_t)(lo & 1) | ((uint32_t)(hi & 1) << 1);
  uint64_t prev = (lo >> 1) | ((hi >> 1) << (t - 1));
  uint2 e = cur[prev];
  uint32_t l = e.x, u = e.y;
  if (l < u) fm_step(fm, c, l, u);
  if (l >= u) l = u = 0;
  next[key] = make_uint2(l, u);
}

__global__ void ktab_init_kernel(uint2* cur, uint32_t n) { cur[0] = make_uint2(0, n); }

// k-mers that occur exactly once become direct entries (core.cuh): text position + the 8 preceding symbols
__global__ void ktab_direct_kernel(FmView fm, SaView sv, const uint8_t* __restrict__ text, uint2* __restrict__ tab,
                                   uint64_t size) {
  uint64_t key = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (key >= size) return;
  uint2 e = tab[key];
  if (e.y - e.x != 1) return;
  tab[key] = ktab_direct_entry(fm_locate(fm, sv, e.x, nullptr), text);
}

__global__ void sa_thin_kernel(const uint32_t* __restrict__ full, uint64_t len, uint32_t rate, uint32_t* __restrict__ out) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < len) out[i] = full[i * rate];
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
static double now_s() {
  return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

// reference text -> 4-bit match classes, 16 symbols per 64-bit word (symbol i of a word in bits 4i..4i+3)
__global__ void text_pack4_kernel(const uint8_t* __restrict__ text, uint64_t n, uint64_t* __restrict__ text4,
                                  uint64_t n_words) {
  uint64_t w = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= n_words) return;
  uint64_t v = 0;
  for (uint32_t i = 0; i < 16; ++i) {
    uint64_t pos = w * 16 + i;
    uint32_t c = 4;
    if (pos < n) {
      c = upper_acgtn_code(text[pos]);
      if (c > 3) c = 4;  // N, '$' and any other byte match nothing (src/index.rs:272-279: read N became '.')
    }
    v |= (uint64_t)c << (4 * i);
  }
  text4[w] = v;
}

void index_destroy(mtsvgpu_index* h) {
  if (!h) return;
  cudaSetDevice(h->ix.device);  // the members' memory is freed by `delete h`, on this device
  for (Lane& ln : h->lanes) {
    if (ln.emit_event) cudaEventDestroy(ln.emit_event);
    for (cudaEvent_t e : ln.ev_pool) cudaEventDestroy(e);
  }
  if (h->lane1_stream) cudaStreamDestroy(h->lane1_stream);
  if (h->fork_event) cudaEventDestroy(h->fork_event);
  if (h->join_event) cudaEventDestroy(h->join_event);
  for (cudaEvent_t e : h->in_events) cudaEventDestroy(e);
  for (cudaEvent_t e : h->trace_events) cudaEventDestroy(e);
  if (h->copy_in_stream) cudaStreamDestroy(h->copy_in_stream);
  if (h->copy_out_stream) cudaStreamDestroy(h->copy_out_stream);
  if (h->out_event) cudaEventDestroy(h->out_event);
  if (h->own_stream) cudaStreamDestroy(h->own_stream);
  delete h;
}

static uint32_t auto_ktab_k(uint64_t n) {
  // floor(log4 n) + 2, clamped to [1, 16]: with ~n/16 expected chance matches per key most seeds that do
  // not occur in the reference die at the table lookup itself (one DRAM line instead of ~4 rank steps);
  // the caller shrinks k until the table fits a third of the free memory.
  uint32_t k = 0;
  while (k < 16 && (1ull << (2 * (k + 1))) <= n) ++k;
  k += 2;
  if (k > 16) k = 16;
  if (k < 1) k = 1;
  return k;
}

int index_assemble(IndexParts parts, int device, const mtsvgpu_index_opts* opts, mtsvgpu_index** out) {
  double t0 = now_s();
  const uint8_t* text = parts.text;
  const uint64_t n = parts.n;
  const mtsvgpu_bin* bins = parts.bins;
  const uint64_t n_bins = parts.n_bins;
  const uint8_t* bwt = parts.bwt;
  const uint64_t* sa_sample = parts.sa_sample;
  const uint64_t sa_sample_len = parts.sa_sample_len;
  const uint64_t sa_rate = parts.sa_rate;
  if (!text || !bins || !bwt || (!sa_sample && !parts.d_sa_full) || !out)
    return set_error(MTSVGPU_EINVAL, "null argument");
  *out = nullptr;
  // ---- validation of the MGIndex fields (SURVEY §8b "loader must assert") ----
  if (n < 2) return set_error(MTSVGPU_EFORMAT, "index text has %llu symbols", (unsigned long long)n);
  if (n >= (1ull << 32) - 64)
    return set_error(MTSVGPU_ELIMIT,
                     "index has %llu symbols; this build keeps 32-bit rows (limit 2^32-64)",
                     (unsigned long long)n);
  if (!parts.text_on_device && text[n - 1] != '$') return set_error(MTSVGPU_EFORMAT, "sequences do not end with '$'");
  if (sa_rate == 0 || sa_rate > 0xffffffffull)
    return set_error(MTSVGPU_EFORMAT, "bad suffix-array sample rate");
  if (!parts.d_sa_full && sa_sample_len != (n + sa_rate - 1) / sa_rate)
    return set_error(MTSVGPU_EFORMAT, "suffix-array sample has %llu entries, expected %llu",
                     (unsigned long long)sa_sample_len,
                     (unsigned long long)((n + sa_rate - 1) / sa_rate));
  if (n_bins == 0 || n_bins > 0xfffffff0ull) return set_error(MTSVGPU_EFORMAT, "bad bin count");
  {
    uint64_t prev_end = 0;
    for (uint64_t i = 0; i < n_bins; ++i) {
      if (bins[i].start != prev_end || bins[i].end < bins[i].start || bins[i].end > n - 1)
        return set_error(MTSVGPU_EFORMAT, "bin %llu [%llu,%llu) is not contiguous within the text",
                         (unsigned long long)i, (unsigned long long)bins[i].start,
                         (unsigned long long)bins[i].end);
      prev_end = bins[i].end;
    }
    if (prev_end != n - 1)
      return set_error(MTSVGPU_EFORMAT, "bins end at %llu, text (without '$') at %llu",
                       (unsigned long long)prev_end, (unsigned long long)(n - 1));
  }

  MTSV_TRY(use_device(device));

  std::unique_ptr<mtsvgpu_index, void (*)(mtsvgpu_index*)> guard(new mtsvgpu_index, index_destroy);
  mtsvgpu_index* h = guard.get();
  if (opts) h->opts = *opts;
  DeviceIndex& d = h->ix;
  d.device = device;
  d.n = n;
  d.n_bins = n_bins;
  d.file_sa_rate = sa_rate;

  MTSV_CUDA_TRY(cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking));
  h->stream = h->own_stream;
  h->lanes[0].ws = &h->ws;
  h->lanes[1].ws = &h->ws1;
  MTSV_CUDA_TRY(cudaStreamCreateWithFlags(&h->copy_in_stream, cudaStreamNonBlocking));
  MTSV_CUDA_TRY(cudaStreamCreateWithFlags(&h->copy_out_stream, cudaStreamNonBlocking));
  MTSV_CUDA_TRY(cudaEventCreateWithFlags(&h->out_event, cudaEventDisableTiming));
  cudaStream_t st = h->stream;

  // ---- text and bins ----
  MTSV_TRY(dev_alloc(d.text, n + 16, &d.device_bytes));
  MTSV_CUDA_TRY(cudaMemcpyAsync(d.text.get(), text, n, cudaMemcpyDefault, st));
  MTSV_CUDA_TRY(cudaMemsetAsync(d.text.get() + n, 0, 16, st));
  if (parts.text_on_device) {
    uint8_t last = 0;
    MTSV_CUDA_TRY(cudaMemcpyAsync(&last, d.text.get() + n - 1, 1, cudaMemcpyDeviceToHost, st));
    MTSV_CUDA_TRY(cudaStreamSynchronize(st));
    if (last != '$') return set_error(MTSVGPU_EFORMAT, "sequences do not end with '$'");
  }
  // 4-bit match classes for the verifier's fast path (+ 2 words of slack: it reads one word ahead)
  d.text4_words = (n + 15) / 16 + 2;
  MTSV_TRY(dev_alloc(d.text4, d.text4_words, &d.device_bytes));
  MTSV_LAUNCH(text_pack4_kernel, (unsigned)((d.text4_words + 255) / 256), 256, 0, st, d.text.get(), n, d.text4.get(),
              d.text4_words);
  {
    std::vector<uint32_t> bs(n_bins), be(n_bins), bt(n_bins), bg(n_bins);
    for (uint64_t i = 0; i < n_bins; ++i) {
      bs[i] = (uint32_t)bins[i].start;
      be[i] = (uint32_t)bins[i].end;
      bt[i] = bins[i].tax_id;
      bg[i] = bins[i].gi;
    }
    {
      std::vector<uint32_t> t = bt;
      std::sort(t.begin(), t.end());
      d.n_taxids = (uint64_t)(std::unique(t.begin(), t.end()) - t.begin());
    }
    MTSV_TRY(dev_alloc(d.bin_start, n_bins, &d.device_bytes));
    MTSV_TRY(dev_alloc(d.bin_end, n_bins, &d.device_bytes));
    MTSV_TRY(dev_alloc(d.bin_tax, n_bins, &d.device_bytes));
    MTSV_TRY(dev_alloc(d.bin_gi, n_bins, &d.device_bytes));
    MTSV_CUDA_TRY(cudaMemcpy(d.bin_start.get(), bs.data(), n_bins * 4, cudaMemcpyHostToDevice));
    MTSV_CUDA_TRY(cudaMemcpy(d.bin_end.get(), be.data(), n_bins * 4, cudaMemcpyHostToDevice));
    MTSV_CUDA_TRY(cudaMemcpy(d.bin_tax.get(), bt.data(), n_bins * 4, cudaMemcpyHostToDevice));
    MTSV_CUDA_TRY(cudaMemcpy(d.bin_gi.get(), bg.data(), n_bins * 4, cudaMemcpyHostToDevice));
  }

  // ---- BWT re-layout ----
  d.n_blocks = n / kRowsPerBlock + 1;
  d.n_super = (d.n_blocks + kBlocksPerSuper - 1) / kBlocksPerSuper;
  MTSV_TRY(dev_alloc(d.blocks, d.n_super * kBlocksPerSuper, &d.device_bytes));
  MTSV_TRY(dev_alloc(d.super, d.n_super, &d.device_bytes));
  MTSV_TRY(dev_alloc(d.n_before, d.n_super * kBlocksPerSuper, &d.device_bytes));

  DevPtr<uint8_t> d_bwt;
  DevPtr<uint32_t> d_super_tot, d_super_n;
  DevPtr<unsigned long long> d_totals;
  DevPtr<PackDiag> d_diag;
  // (a BWT that is already on the device is used where it lies: the caller pads it by 64 bytes)
  const uint8_t* bwt_dev = bwt;
  if (!parts.bwt_on_device) {
    MTSV_TRY(dev_alloc(d_bwt, n + 64));
    bwt_dev = d_bwt.get();
  }
  MTSV_TRY(dev_alloc(d_super_tot, d.n_super * 5));
  MTSV_TRY(dev_alloc(d_super_n, d.n_super));
  MTSV_TRY(dev_alloc(d_totals, 5));
  MTSV_TRY(dev_alloc(d_diag, 1));
  MTSV_CUDA_TRY(cudaMemsetAsync(d_diag.get(), 0, sizeof(PackDiag), st));
  if (!parts.bwt_on_device) MTSV_CUDA_TRY(cudaMemcpyAsync(d_bwt.get(), bwt, n, cudaMemcpyHostToDevice, st));
  MTSV_CUDA_TRY(cudaStreamSynchronize(st));
  double t_relayout0 = now_s();

  MTSV_LAUNCH(fm_pack_kernel, (unsigned)d.n_super, kBlocksPerSuper, 0, st, bwt_dev, n, d.n_blocks,
              d.blocks.get(), d.n_before.get(), d_super_tot.get(), d_diag.get());
  MTSV_LAUNCH(fm_super_scan_kernel, 1, 32, 0, st, d_super_tot.get(), d.n_super, d.super.get(), d_super_n.get(),
              d_totals.get());
  MTSV_LAUNCH(fm_finish_kernel, (unsigned)((d.n_blocks + 255) / 256), 256, 0, st, d.n_before.get(),
              d.n_blocks, d_super_n.get());
  MTSV_CUDA_TRY(cudaGetLastError());
  unsigned long long totals[5];
  PackDiag diag;
  MTSV_CUDA_TRY(cudaMemcpyAsync(totals, d_totals.get(), sizeof totals, cudaMemcpyDeviceToHost, st));
  MTSV_CUDA_TRY(cudaMemcpyAsync(&diag, d_diag.get(), sizeof diag, cudaMemcpyDeviceToHost, st));
  MTSV_CUDA_TRY(cudaStreamSynchronize(st));
  if (diag.n_dollar != 1)
    return set_error(MTSVGPU_EFORMAT, "BWT holds %llu '$' symbols, expected exactly 1", diag.n_dollar);
  if (diag.n_other != 0)
    return set_error(MTSVGPU_EFORMAT, "BWT holds %llu symbols outside $ACGTN", diag.n_other);
  if (totals[0] + totals[1] + totals[2] + totals[3] + totals[4] + 1 != n)
    return set_error(MTSVGPU_EFORMAT, "BWT symbol counts do not add up to the text length");
  d.dollar_row = (uint32_t)diag.dollar_row;
  // `less` recomputed from the BWT (never trusted from the file): $ < A < C < G < N < T
  d.C[SYM_A] = 1;
  d.C[SYM_C] = (uint32_t)(1 + totals[0]);
  d.C[SYM_G] = (uint32_t)(1 + totals[0] + totals[1]);
  d.C[SYM_N] = (uint32_t)(1 + totals[0] + totals[1] + totals[2]);
  d.C[SYM_T] = (uint32_t)(1 + totals[0] + totals[1] + totals[2] + totals[4]);
  MTSV_TRY(dev_alloc(d.d_C, 8, &d.device_bytes));
  MTSV_CUDA_TRY(cudaMemcpy(d.d_C.get(), d.C, 5 * sizeof(uint32_t), cudaMemcpyHostToDevice));
  d_bwt.reset();

  // ---- suffix array at the device rate ----
  size_t free_b = 0, total_b = 0;
  MTSV_CUDA_TRY(cudaMemGetInfo(&free_b, &total_b));
  uint32_t rate = h->opts.sa_rate;
  if (parts.d_sa_full) {
    // built on this device (sufsort.cu): the complete array is adopted as it is, or thinned to the requested rate
    if (rate <= 1) {
      d.sa = std::move(parts.d_sa_full);
      d.sa_rate = 1;
      d.sa_len = n;
      d.device_bytes += n * 4;
    } else {
      d.sa_rate = rate;
      d.sa_len = (n + rate - 1) / rate;
      MTSV_TRY(dev_alloc(d.sa, d.sa_len, &d.device_bytes));
      MTSV_LAUNCH(sa_thin_kernel, (unsigned)((d.sa_len + 255) / 256), 256, 0, st, parts.d_sa_full.get(), d.sa_len, rate,
                  d.sa.get());
      MTSV_CUDA_TRY(cudaStreamSynchronize(st));
      parts.d_sa_full.reset();
    }
  } else {
  if (rate == 0) {
    rate = 1;
    // keep the dense array under a quarter of what is still free (the rest is for batches)
    while (rate < sa_rate && (n / rate + 1) * 4ull + sa_sample_len * 8ull > free_b / 4) rate *= 2;
    if (rate > sa_rate) rate = (uint32_t)sa_rate;
  }
  if (rate > sa_rate) rate = (uint32_t)sa_rate;
  d.sa_rate = rate;
  d.sa_len = (n + rate - 1) / rate;
  MTSV_TRY(dev_alloc(d.sa, d.sa_len, &d.device_bytes));
  DevPtr<uint64_t> d_sample;
  MTSV_TRY(dev_alloc(d_sample, sa_sample_len));
  MTSV_CUDA_TRY(cudaMemcpyAsync(d_sample.get(), sa_sample, sa_sample_len * 8, cudaMemcpyHostToDevice, st));
  MTSV_CUDA_TRY(cudaMemsetAsync(d.sa.get(), 0xff, d.sa_len * 4, st));
  MTSV_LAUNCH(sa_densify_kernel, (unsigned)((sa_sample_len + 127) / 128), 128, 0, st, d.fm_view(),
              d_sample.get(), sa_sample_len, (uint32_t)sa_rate, rate, d.sa.get(), d_diag.get());
  MTSV_CUDA_TRY(cudaGetLastError());
  MTSV_CUDA_TRY(cudaMemcpyAsync(&diag, d_diag.get(), sizeof diag, cudaMemcpyDeviceToHost, st));
  MTSV_CUDA_TRY(cudaStreamSynchronize(st));
  if (diag.sa_mismatch != 0 || diag.rows_seen != n)
    return set_error(MTSVGPU_EFORMAT,
                     "suffix-array samples are inconsistent with the BWT (%llu LF walks disagree, "
                     "%llu of %llu rows reached)",
                     diag.sa_mismatch, diag.rows_seen, (unsigned long long)n);
  }

  // ---- k-mer interval table ----
  uint32_t kk = h->opts.ktab_k;
  if (kk == 0) kk = auto_ktab_k(n);
  if (kk == 0xffffffffu) kk = 0;
  if (kk > 16) kk = 16;
  if (kk > 0) {
    MTSV_CUDA_TRY(cudaMemGetInfo(&free_b, &total_b));
    while (kk > 1 && (1ull << (2 * kk)) * 8ull * 5 / 4 > free_b / 3) --kk;
    uint64_t size = 1ull << (2 * kk);
    MTSV_TRY(dev_alloc(d.ktab, size, &d.device_bytes));
    if (kk >= 1) {
      DevPtr<uint2> d_ktmp;
      MTSV_TRY(dev_alloc(d_ktmp, kk >= 2 ? (1ull << (2 * (kk - 1))) : 1));
      // levels alternate between the two buffers so that level kk lands in d.ktab
      uint2* bufs[2] = {d.ktab.get(), d_ktmp.get()};
      int cur = (kk % 2 == 0) ? 0 : 1;  // level 0 buffer
      MTSV_LAUNCH(ktab_init_kernel, 1, 1, 0, st, bufs[cur], (uint32_t)n);
      uint64_t cur_size = 1;
      for (uint32_t lev = 1; lev <= kk; ++lev) {
        uint64_t threads = cur_size * 4;
        MTSV_LAUNCH(ktab_level_kernel, (unsigned)((threads + 255) / 256), 256, 0, st, d.fm_view(),
                    bufs[cur], bufs[cur ^ 1], lev);
        cur ^= 1;
        cur_size *= 4;
      }
      // row indexes of ordinary entries must stay below the direct tag; MTSV_B200_KTAB_DIRECT=0 is an A/B knob
      const char* de = getenv("MTSV_B200_KTAB_DIRECT");
      if (n < ((uint64_t)kKtabDirectTag << 24) && !(de && de[0] == '0')) {
        MTSV_LAUNCH(ktab_direct_kernel, (unsigned)((size + 255) / 256), 256, 0, st, d.fm_view(), d.sa_view(),
                    d.text.get(), d.ktab.get(), size);
        d.ktab_direct = 1;
      }
      MTSV_CUDA_TRY(cudaGetLastError());
      MTSV_CUDA_TRY(cudaStreamSynchronize(st));
    }
  }
  d.ktab_k = kk;
  MTSV_CUDA_TRY(cudaStreamSynchronize(st));
  double t1 = now_s();
  d.relayout_seconds = t1 - t_relayout0;
  d.load_seconds = t1 - t0;
  *out = guard.release();
  return 0;
}

int index_from_host_parts(const uint8_t* text, uint64_t n, const mtsvgpu_bin* bins, uint64_t n_bins,
                          const uint8_t* bwt, const uint64_t* sa_sample, uint64_t sa_sample_len,
                          uint64_t sa_rate, int device, const mtsvgpu_index_opts* opts,
                          mtsvgpu_index** out) {
  if (!sa_sample) return set_error(MTSVGPU_EINVAL, "null argument");
  IndexParts parts;
  parts.text = text;
  parts.n = n;
  parts.bins = bins;
  parts.n_bins = n_bins;
  parts.bwt = bwt;
  parts.sa_sample = sa_sample;
  parts.sa_sample_len = sa_sample_len;
  parts.sa_rate = sa_rate;
  return index_assemble(std::move(parts), device, opts, out);
}

// ---------------------------------------------------------------------------------------------
// bincode 1.3.3 reader (legacy `deserialize_from`: fixed-width little-endian integers, usize and
// lengths as u64, structs as their fields in order; SURVEY §8b).  Field order of
// SampledSuffixArray per bio 3.0.0: bwt, less, occ{occ: Vec<Vec<usize>>, k: u32}, sample, s,
// extra_rows (HashMap<usize,usize>), sentinel.  `less` and `occ` are skipped, not trusted.
// ---------------------------------------------------------------------------------------------
namespace {
struct Cursor {
  const uint8_t* p;
  uint64_t size, pos = 0;
  bool ok = true;
  bool need(uint64_t k) {
    if (!ok || k > size - pos) ok = false;
    return ok;
  }
  uint64_t u64() {
    if (!need(8)) return 0;
    uint64_t v;
    memcpy(&v, p + pos, 8);
    pos += 8;
    return v;
  }
  uint32_t u32() {
    if (!need(4)) return 0;
    uint32_t v;
    memcpy(&v, p + pos, 4);
    pos += 4;
    return v;
  }
  uint8_t u8() {
    if (!need(1)) return 0;
    return p[pos++];
  }
  const uint8_t* bytes(uint64_t k) {
    if (!need(k)) return nullptr;
    const uint8_t* r = p + pos;
    pos += k;
    return r;
  }
};
}  // namespace

int index_open_file(const char* path, int device, const mtsvgpu_index_opts* opts,
                    mtsvgpu_index** out) {
  if (!path || !out) return set_error(MTSVGPU_EINVAL, "null argument");
  *out = nullptr;
  int fd = open(path, O_RDONLY);
  if (fd < 0) return set_error(MTSVGPU_EIO, "cannot open %s: %s", path, strerror(errno));
  struct stat sb;
  if (fstat(fd, &sb) != 0 || sb.st_size < 64) {
    close(fd);
    return set_error(MTSVGPU_EFORMAT, "%s is too small to be an MGIndex", path);
  }
  uint64_t size = (uint64_t)sb.st_size;
  void* map = mmap(nullptr, size, PROT_READ, MAP_PRIVATE, fd, 0);
  close(fd);
  if (map == MAP_FAILED) return set_error(MTSVGPU_EIO, "mmap(%s) failed: %s", path, strerror(errno));
  madvise(map, size, MADV_SEQUENTIAL);
  struct Unmap {
    void* m;
    uint64_t s;
    ~Unmap() { munmap(m, s); }
  } um{map, size};

  Cursor c{(const uint8_t*)map, size};
  uint64_t n = c.u64();
  const uint8_t* text = c.bytes(n);
  uint64_t n_bins = c.u64();
  if (!c.ok || n_bins > size / 24) return set_error(MTSVGPU_EFORMAT, "%s: truncated (sequences/bins)", path);
  std::vector<mtsvgpu_bin> bins(n_bins);
  for (uint64_t i = 0; i < n_bins; ++i) {
    bins[i].gi = c.u32();
    bins[i].tax_id = c.u32();
    bins[i].start = c.u64();
    bins[i].end = c.u64();
  }
  uint64_t n_bwt = c.u64();
  const uint8_t* bwt = c.bytes(n_bwt);
  if (!c.ok) return set_error(MTSVGPU_EFORMAT, "%s: truncated (bwt)", path);
  if (n_bwt != n)
    return set_error(MTSVGPU_EFORMAT, "%s: sequences (%llu) and BWT (%llu) lengths differ", path,
                     (unsigned long long)n, (unsigned long long)n_bwt);
  uint64_t n_less = c.u64();
  if (!c.ok || n_less > 65536) return set_error(MTSVGPU_EFORMAT, "%s: bad `less` length", path);
  c.bytes(n_less * 8);
  uint64_t n_occ = c.u64();
  if (!c.ok || n_occ > size / 8) return set_error(MTSVGPU_EFORMAT, "%s: bad occ table", path);
  for (uint64_t i = 0; i < n_occ && c.ok; ++i) {
    uint64_t len = c.u64();
    if (!c.ok || len > size / 8) return set_error(MTSVGPU_EFORMAT, "%s: bad occ row", path);
    c.bytes(len * 8);
  }
  (void)c.u32();  // Occ.k — the device layout has its own checkpoint spacing
  uint64_t n_sample = c.u64();
  if (!c.ok || n_sample > size / 8) return set_error(MTSVGPU_EFORMAT, "%s: bad sample length", path);
  const uint8_t* sample_bytes = c.bytes(n_sample * 8);
  uint64_t s = c.u64();
  uint64_t n_extra = c.u64();
  if (!c.ok || n_extra > size / 16) return set_error(MTSVGPU_EFORMAT, "%s: bad extra_rows", path);
  c.bytes(n_extra * 16);
  uint8_t sentinel = c.u8();
  if (!c.ok) return set_error(MTSVGPU_EFORMAT, "%s: truncated", path);
  if (c.pos != size)
    return set_error(MTSVGPU_EFORMAT, "%s: %llu trailing bytes after MGIndex", path,
                     (unsigned long long)(size - c.pos));
  if (sentinel != '$') return set_error(MTSVGPU_EFORMAT, "%s: sentinel is 0x%02x, expected '$'", path, sentinel);
  // bincode does not align: copy the samples to an aligned buffer
  std::vector<uint64_t> sample(n_sample);
  if (n_sample) memcpy(sample.data(), sample_bytes, n_sample * 8);
  return index_from_host_parts(text, n, bins.data(), n_bins, bwt, sample.data(), n_sample, s, device,
                               opts, out);
}

}  // namespace mtsv
