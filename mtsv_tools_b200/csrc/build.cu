// build.cu — mtsv-build on the device: MGIndex::new (src/index.rs:491-582) and write_to_file (src/io.rs:125-132).
//
//   mtsvgpu_index_build   reference sequences -> bins in TaxID order, text normalised to ACGTN + '$'
//                         (src/index.rs:496-556), suffix array (sufsort.cu), BWT (:566-567), and straight into the
//                         device layout of index.cu: the complete suffix array stays in HBM as the index's own,
//                         nothing travels through the host.
//   mtsvgpu_index_write   any loaded index -> the bincode 1.3.3 `.index` a reference mtsv-binner reads: byte BWT
//                         unpacked from the 2-bit sectors, `less`, Occ checkpoints every `sample_interval` rows and
//                         the row-sampled suffix array are produced by kernels chunk by chunk and streamed to the file.
#include <errno.h>
#include <stdio.h>
#include <string.h>

#include <chrono>
#include <numeric>

#include "ctx.h"

namespace mtsv {

int suffix_array_device(const uint8_t* d_text, uint64_t n, cudaStream_t st, DevPtr<uint32_t>& sa_out, int verbose);
int bwt_from_sa_device(const uint8_t* d_text, const uint32_t* d_sa, uint64_t n, cudaStream_t st, uint8_t* d_bwt);

namespace {

double now_s() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

// "convert whole reference sequence to DNA5 alphabet" (src/index.rs:543-553), 16 bytes per thread
__global__ void __launch_bounds__(256) normalise_text_kernel(uint8_t* __restrict__ text, uint64_t total) {
  const uint64_t i0 = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) * 16;
  if (i0 >= total) return;
  if (i0 + 16 <= total && (reinterpret_cast<uintptr_t>(text + i0) & 15) == 0) {
    uint4 v = *reinterpret_cast<uint4*>(text + i0);
    uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      uint32_t o = 0;
#pragma unroll
      for (int b = 0; b < 4; ++b) {
        const uint32_t c = read_code((uint8_t)(w[k] >> (8 * b)));
        o |= (uint32_t)"ACGTN"[c] << (8 * b);
      }
      w[k] = o;
    }
    *reinterpret_cast<uint4*>(text + i0) = make_uint4(w[0], w[1], w[2], w[3]);
  } else {
    for (uint64_t i = i0; i < total && i < i0 + 16; ++i) text[i] = (uint8_t)"ACGTN"[read_code(text[i])];
  }
}

// byte BWT of rows [row0, row0 + count) from the 2-bit sectors
__global__ void __launch_bounds__(256) bwt_unpack_kernel(FmView fm, uint64_t row0, uint64_t count, uint8_t* __restrict__ out) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  const uint32_t row = (uint32_t)(row0 + i);
  const FmBlock b = load_block(fm.blocks + (row >> 6));
  const uint32_t c = fm_symbol(fm, b, row);
  out[i] = (uint8_t)"ACGTN$"[c];
}

// Occ checkpoints (bio Occ::new): entry j of symbol a = occurrences of a in bwt[0 ..= j*K]
__global__ void __launch_bounds__(256) occ_checkpoint_kernel(FmView fm, uint32_t sym, uint64_t K, uint64_t j0, uint64_t count,
                                                             uint64_t* __restrict__ out) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  const uint64_t row = (j0 + i) * K;  // <= n - 1
  uint64_t v;
  if (sym == SYM_DOLLAR) v = fm.dollar_row <= row ? 1 : 0;
  else v = fm_occ(fm, sym, (uint32_t)(row + 1));
  out[i] = v;
}

// row-sampled suffix array (bio SuffixArray::sample): entry i = SA[i * s]
__global__ void __launch_bounds__(256) sa_sample_kernel(FmView fm, SaView sv, uint64_t s, uint64_t i0, uint64_t count,
                                                        uint64_t* __restrict__ out) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  out[i] = fm_locate(fm, sv, (uint32_t)((i0 + i) * s), nullptr);
}

struct FileWriter {
  FILE* f = nullptr;
  bool ok = true;
  ~FileWriter() {
    if (f) fclose(f);
  }
  void raw(const void* p, size_t n) {
    if (ok && n && fwrite(p, 1, n, f) != n) ok = false;
  }
  void u64(uint64_t v) { raw(&v, 8); }
  void u32(uint32_t v) { raw(&v, 4); }
  void u8(uint8_t v) { raw(&v, 1); }
};

}  // namespace

int index_build(const uint8_t* seqs, const uint64_t* seq_off, const uint32_t* gi, const uint32_t* tax_id, uint64_t n_seqs,
                int device, const mtsvgpu_index_opts* opts, mtsvgpu_index** out) {
  if (!seq_off || !gi || !tax_id || !out) return set_error(MTSVGPU_EINVAL, "null argument");
  *out = nullptr;
  if (n_seqs == 0 || n_seqs > 0xfffffff0ull) return set_error(MTSVGPU_EINVAL, "bad sequence count");
  for (uint64_t i = 0; i < n_seqs; ++i)
    if (seq_off[i + 1] < seq_off[i]) return set_error(MTSVGPU_EINVAL, "seq_off is not monotone");
  const uint64_t total = seq_off[n_seqs] - seq_off[0];
  const uint64_t n = total + 1;
  if (n >= (1ull << 32) - 64)
    return set_error(MTSVGPU_ELIMIT, "reference has %llu symbols; this build keeps 32-bit rows (limit 2^32-64)",
                     (unsigned long long)n);
  if (total && !seqs) return set_error(MTSVGPU_EINVAL, "seqs is NULL");
  MTSV_TRY(use_device(device));
  const double t0 = now_s();
  const int verbose = getenv("MTSV_B200_VERBOSE") != nullptr;

  // bins in TaxID order, file order within a TaxID: the BTreeMap<TaxId, Vec<(Gi, Sequence)>> of parse_fasta_db
  // (src/io.rs:135-150) walked by MGIndex::new (src/index.rs:497-511)
  std::vector<uint64_t> order(n_seqs);
  std::iota(order.begin(), order.end(), 0ull);
  std::stable_sort(order.begin(), order.end(), [&](uint64_t a, uint64_t b) { return tax_id[a] < tax_id[b]; });
  std::vector<mtsvgpu_bin> bins(n_seqs);
  bool in_place = true;
  {
    uint64_t at = 0;
    for (uint64_t k = 0; k < n_seqs; ++k) {
      const uint64_t o = order[k], len = seq_off[o + 1] - seq_off[o];
      bins[k] = mtsvgpu_bin{gi[o], tax_id[o], at, at + len};
      if (seq_off[o] - seq_off[0] != at) in_place = false;
      at += len;
    }
  }

  cudaStream_t st = nullptr;
  MTSV_CUDA_TRY(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
  struct StreamGuard {
    cudaStream_t s;
    ~StreamGuard() { cudaStreamDestroy(s); }
  } sg{st};
  DevPtr<uint8_t> text_g, bwt_g;
  MTSV_TRY(dev_alloc(text_g, n + 16));
  uint8_t* d_text = text_g.get();
  if (in_place) {
    if (total) MTSV_CUDA_TRY(cudaMemcpyAsync(d_text, seqs + seq_off[0], total, cudaMemcpyDefault, st));
  } else {
    for (uint64_t k = 0; k < n_seqs; ++k) {
      const uint64_t o = order[k], len = seq_off[o + 1] - seq_off[o];
      if (len) MTSV_CUDA_TRY(cudaMemcpyAsync(d_text + bins[k].start, seqs + seq_off[o], len, cudaMemcpyDefault, st));
    }
  }
  if (total) MTSV_LAUNCH(normalise_text_kernel, (unsigned)(((total + 15) / 16 + 255) / 256), 256, 0, st, d_text, total);
  MTSV_CUDA_TRY(cudaMemsetAsync(d_text + total, '$', 1, st));
  MTSV_CUDA_TRY(cudaMemsetAsync(d_text + n, 0, 16, st));
  MTSV_CUDA_TRY(cudaGetLastError());

  DevPtr<uint32_t> d_sa;
  MTSV_TRY(suffix_array_device(d_text, n, st, d_sa, verbose));
  const double t_sa = now_s();
  MTSV_TRY(dev_alloc(bwt_g, n + 64));
  uint8_t* d_bwt = bwt_g.get();
  MTSV_CUDA_TRY(cudaMemsetAsync(d_bwt + n, 0, 64, st));
  MTSV_TRY(bwt_from_sa_device(d_text, d_sa.get(), n, st, d_bwt));
  if (cudaStreamSynchronize(st) != cudaSuccess)
    return set_error(MTSVGPU_ECUDA, "BWT construction failed: %s", cudaGetErrorString(cudaGetLastError()));
  const double t_bwt = now_s();
  if (verbose)
    fprintf(stderr, "[mtsv_b200 build] %llu symbols, %llu bins: suffix array %.2f s, BWT %.3f s\n", (unsigned long long)n,
            (unsigned long long)n_seqs, t_sa - t0, t_bwt - t_sa);

  IndexParts parts;
  parts.text = d_text;
  parts.text_on_device = true;
  parts.n = n;
  parts.bins = bins.data();
  parts.n_bins = n_seqs;
  parts.bwt = d_bwt;
  parts.bwt_on_device = true;
  parts.sa_rate = 32;  // what mtsv-build samples by default (src/bin/mtsv-build.rs); only recorded
  parts.d_sa_full = std::move(d_sa);
  MTSV_TRY(index_assemble(std::move(parts), device, opts, out));
  (*out)->ix.build_seconds = t_bwt - t0;
  return 0;
}

int index_write(mtsvgpu_index* h, const char* path, uint32_t sample_interval, uint32_t sa_sample) {
  if (!h || !path) return set_error(MTSVGPU_EINVAL, "null argument");
  if (sample_interval == 0 || sa_sample == 0) return set_error(MTSVGPU_EINVAL, "sample intervals must be > 0");
  DeviceIndex& d = h->ix;
  MTSV_CUDA_TRY(cudaSetDevice(d.device));
  cudaStream_t st = h->stream;
  const uint64_t n = d.n, K = sample_interval, s = sa_sample;
  FileWriter w;
  w.f = fopen(path, "wb");
  if (!w.f) return set_error(MTSVGPU_EIO, "cannot create %s: %s", path, strerror(errno));
  const uint64_t chunk = 1ull << 25;  // 32 Mi items per step
  DevPtr<uint64_t> dev;
  PinnedPtr<uint64_t> host;
  MTSV_TRY(dev_alloc(dev, chunk));
  MTSV_TRY(pinned_alloc(host, chunk));
  uint8_t* d8 = (uint8_t*)dev.get();
  uint64_t* d64 = dev.get();
  const FmView fm = d.fm_view();

  // sequences: Vec<u8>
  w.u64(n);
  for (uint64_t o = 0; o < n && w.ok; o += chunk * 8) {
    const uint64_t c = std::min<uint64_t>(chunk * 8, n - o);
    MTSV_CUDA_TRY(cudaMemcpyAsync(host.get(), d.text.get() + o, c, cudaMemcpyDeviceToHost, st));
    MTSV_CUDA_TRY(cudaStreamSynchronize(st));
    w.raw(host.get(), c);
  }
  // bins: Vec<Bin{gi, tax_id, start, end}>
  {
    const uint64_t nb = d.n_bins;
    std::vector<uint32_t> bs(nb), be(nb), bt(nb), bg(nb);
    MTSV_CUDA_TRY(cudaMemcpy(bs.data(), d.bin_start.get(), nb * 4, cudaMemcpyDeviceToHost));
    MTSV_CUDA_TRY(cudaMemcpy(be.data(), d.bin_end.get(), nb * 4, cudaMemcpyDeviceToHost));
    MTSV_CUDA_TRY(cudaMemcpy(bt.data(), d.bin_tax.get(), nb * 4, cudaMemcpyDeviceToHost));
    MTSV_CUDA_TRY(cudaMemcpy(bg.data(), d.bin_gi.get(), nb * 4, cudaMemcpyDeviceToHost));
    w.u64(nb);
    for (uint64_t i = 0; i < nb; ++i) {
      w.u32(bg[i]);
      w.u32(bt[i]);
      w.u64(bs[i]);
      w.u64(be[i]);
    }
  }
  // suffix_array.bwt: Vec<u8>
  w.u64(n);
  for (uint64_t o = 0; o < n && w.ok; o += chunk * 8) {
    const uint64_t c = std::min<uint64_t>(chunk * 8, n - o);
    MTSV_LAUNCH(bwt_unpack_kernel, (unsigned)((c + 255) / 256), 256, 0, st, fm, o, c, d8);
    MTSV_CUDA_TRY(cudaMemcpyAsync(host.get(), d8, c, cudaMemcpyDeviceToHost, st));
    MTSV_CUDA_TRY(cudaStreamSynchronize(st));
    w.raw(host.get(), c);
  }
  // less: counts of smaller bytes, over the symbols 0 ..= 't'+1 of n_alphabet() "ACGTNacgtn" (bio::bwt::less)
  {
    uint64_t cnt[256] = {0};
    cnt['$'] = 1;
    cnt['A'] = d.C[SYM_C] - d.C[SYM_A];
    cnt['C'] = d.C[SYM_G] - d.C[SYM_C];
    cnt['G'] = d.C[SYM_N] - d.C[SYM_G];
    cnt['N'] = d.C[SYM_T] - d.C[SYM_N];
    cnt['T'] = n - d.C[SYM_T];
    const uint64_t m_less = 118;
    w.u64(m_less);
    uint64_t sum = 0;
    for (uint64_t c = 0; c < m_less; ++c) {
      w.u64(sum);
      sum += cnt[c];
    }
  }
  // occ: Vec<Vec<usize>> indexed by byte (117 rows, filled for the alphabet symbols and the sentinel), then k
  {
    const uint64_t m_occ = 117, len = (n - 1) / K + 1;
    w.u64(m_occ);
    for (uint64_t byte = 0; byte < m_occ && w.ok; ++byte) {
      uint32_t sym = SYM_OTHER;
      bool zero_row = false;
      switch (byte) {
        case 'A': sym = SYM_A; break;
        case 'C': sym = SYM_C; break;
        case 'G': sym = SYM_G; break;
        case 'T': sym = SYM_T; break;
        case 'N': sym = SYM_N; break;
        case '$': sym = SYM_DOLLAR; break;
        case 'a': case 'c': case 'g': case 't': case 'n': zero_row = true; break;
        default: break;
      }
      if (sym == SYM_OTHER && !zero_row) {
        w.u64(0);
        continue;
      }
      w.u64(len);
      for (uint64_t o = 0; o < len && w.ok; o += chunk) {
        const uint64_t c = std::min<uint64_t>(chunk, len - o);
        if (zero_row) {
          memset(host.get(), 0, c * 8);
        } else {
          MTSV_LAUNCH(occ_checkpoint_kernel, (unsigned)((c + 255) / 256), 256, 0, st, fm, sym, K, o, c, d64);
          MTSV_CUDA_TRY(cudaMemcpyAsync(host.get(), d64, c * 8, cudaMemcpyDeviceToHost, st));
          MTSV_CUDA_TRY(cudaStreamSynchronize(st));
        }
        w.raw(host.get(), c * 8);
      }
    }
    w.u32(sample_interval);
  }
  // sample: Vec<usize>, s, extra_rows: HashMap<usize, usize>, sentinel
  {
    const uint64_t len = (n + s - 1) / s;
    w.u64(len);
    for (uint64_t o = 0; o < len && w.ok; o += chunk) {
      const uint64_t c = std::min<uint64_t>(chunk, len - o);
      MTSV_LAUNCH(sa_sample_kernel, (unsigned)((c + 255) / 256), 256, 0, st, fm, d.sa_view(), s, o, c, d64);
      MTSV_CUDA_TRY(cudaMemcpyAsync(host.get(), d64, c * 8, cudaMemcpyDeviceToHost, st));
      MTSV_CUDA_TRY(cudaStreamSynchronize(st));
      w.raw(host.get(), c * 8);
    }
    w.u64(s);
    if (d.dollar_row % s != 0) {  // the row holding the sentinel is kept when it is not sampled (bio SuffixArray::sample)
      w.u64(1);
      w.u64(d.dollar_row);
      w.u64(0);
    } else {
      w.u64(0);
    }
    w.u8('$');
  }
  MTSV_CUDA_TRY(cudaGetLastError());
  const bool ok = w.ok;
  const int crc = fclose(w.f);
  w.f = nullptr;
  if (!ok || crc != 0) return set_error(MTSVGPU_EIO, "writing %s failed: %s", path, strerror(errno));
  return 0;
}

// The MGIndex fields of a loaded index back in host memory (each output optional): sequences, the byte BWT and the
// suffix array sampled every sa_sample rows — what an oracle / a reference-side consumer needs, without a file.
int index_export(mtsvgpu_index* h, uint8_t* text_out, uint8_t* bwt_out, uint64_t* sample_out, uint32_t sa_sample) {
  if (!h) return set_error(MTSVGPU_EINVAL, "index is NULL");
  if (sample_out && sa_sample == 0) return set_error(MTSVGPU_EINVAL, "sa_sample must be > 0");
  DeviceIndex& d = h->ix;
  MTSV_CUDA_TRY(cudaSetDevice(d.device));
  cudaStream_t st = h->stream;
  const uint64_t n = d.n;
  const FmView fm = d.fm_view();
  if (text_out) MTSV_CUDA_TRY(cudaMemcpyAsync(text_out, d.text.get(), n, cudaMemcpyDeviceToHost, st));
  const uint64_t chunk = 1ull << 28;
  DevPtr<uint8_t> dev;
  if (bwt_out || sample_out) MTSV_TRY(dev_alloc(dev, chunk));
  if (bwt_out) {
    for (uint64_t o = 0; o < n; o += chunk) {
      const uint64_t c = std::min<uint64_t>(chunk, n - o);
      MTSV_LAUNCH(bwt_unpack_kernel, (unsigned)((c + 255) / 256), 256, 0, st, fm, o, c, dev.get());
      MTSV_CUDA_TRY(cudaMemcpyAsync(bwt_out + o, dev.get(), c, cudaMemcpyDeviceToHost, st));
      MTSV_CUDA_TRY(cudaStreamSynchronize(st));
    }
  }
  if (sample_out) {
    const uint64_t len = (n + sa_sample - 1) / sa_sample, step = chunk / 8;
    for (uint64_t o = 0; o < len; o += step) {
      const uint64_t c = std::min<uint64_t>(step, len - o);
      MTSV_LAUNCH(sa_sample_kernel, (unsigned)((c + 255) / 256), 256, 0, st, fm, d.sa_view(), (uint64_t)sa_sample, o, c,
                  (uint64_t*)dev.get());
      MTSV_CUDA_TRY(cudaMemcpyAsync(sample_out + o, dev.get(), c * 8, cudaMemcpyDeviceToHost, st));
      MTSV_CUDA_TRY(cudaStreamSynchronize(st));
    }
  }
  MTSV_CUDA_TRY(cudaStreamSynchronize(st));
  MTSV_CUDA_TRY(cudaGetLastError());
  return 0;
}

// stage-level entry point: suffix array (and BWT) of a '$'-terminated text held in host memory
int suffix_array_host(int device, const uint8_t* text, uint64_t n, uint32_t* sa_out, uint8_t* bwt_out) {
  if (!text || !sa_out || n == 0) return set_error(MTSVGPU_EINVAL, "null argument");
  if (text[n - 1] != '$') return set_error(MTSVGPU_EINVAL, "the text must end with '$'");
  MTSV_TRY(use_device(device));
  DevPtr<uint8_t> t, b;
  DevPtr<uint32_t> sa;
  MTSV_TRY(dev_alloc(t, n + 16));
  MTSV_CUDA_TRY(cudaMemcpy(t.get(), text, n, cudaMemcpyHostToDevice));
  MTSV_TRY(suffix_array_device(t.get(), n, cudaStreamPerThread, sa, getenv("MTSV_B200_VERBOSE") != nullptr));
  MTSV_CUDA_TRY(cudaStreamSynchronize(cudaStreamPerThread));
  MTSV_CUDA_TRY(cudaMemcpy(sa_out, sa.get(), n * 4, cudaMemcpyDeviceToHost));
  if (bwt_out) {
    MTSV_TRY(dev_alloc(b, n));
    MTSV_TRY(bwt_from_sa_device(t.get(), sa.get(), n, cudaStreamPerThread, b.get()));
    MTSV_CUDA_TRY(cudaStreamSynchronize(cudaStreamPerThread));
    MTSV_CUDA_TRY(cudaMemcpy(bwt_out, b.get(), n, cudaMemcpyDeviceToHost));
  }
  return 0;
}

}  // namespace mtsv
