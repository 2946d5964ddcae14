// chunked.cu — chunk-sharded operation behind the C ABI (SURVEY §8e, BASELINE config 3).
//
// GPU g holds MG-index chunk g; every rank bins the SAME batch of reads against its own chunk (exactly a
// single-index run), then the per-read hit lists are brought together the way mtsv-collapse merges the per-chunk
// results files (src/collapse.rs:543-654; TaxId mode: minimum edit per TaxID, :597-602).  Rank r ends up with the
// merged lists of its contiguous range of the reads.
//
// The exchange is this library's own kernel over NVLink peer memory, not a library collective: every rank exposes
// one device buffer to its peers (CUDA IPC), a source stores the hits and per-read counts of each read range
// straight into the owning rank's buffer, in a slot reserved for that source (no count exchange first), raises a
// flag there, and the owner starts the merge (collapse.cu) as soon as all its flags are up.  Buffers are double
// buffered by batch parity, so the one flag barrier per batch is the only inter-GPU synchronisation, and the
// host synchronises once, at the end, to read the result size.
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "ctx.h"

namespace mtsv {
namespace {

constexpr uint32_t kMaxRanks = 16;
constexpr uint32_t kCommMagic = 0x4d545356u;  // "MTSV"

struct CommHeader {  // first bytes of every rank's buffer; slot s of each array is written by rank s only
  uint32_t flags[kMaxRanks];          // last batch (epoch) whose data from rank s has landed here
  uint32_t error[kMaxRanks];          // epoch in which rank s could not fit a range into its slot
  uint64_t slot_hits[2][kMaxRanks];   // [parity][s]: hits rank s stored for this batch
};

struct CommLayout {
  uint64_t max_local_reads, cap_hits;  // per source slot
  uint32_t world;
  __host__ __device__ uint64_t counts_off(uint32_t parity, uint32_t src) const {
    return 512 + ((uint64_t)parity * world + src) * max_local_reads * 4;
  }
  __host__ __device__ uint64_t hits_base() const {
    return (512 + 2ull * world * max_local_reads * 4 + 255) & ~255ull;
  }
  __host__ __device__ uint64_t hits_off(uint32_t parity, uint32_t src) const {
    return hits_base() + ((uint64_t)parity * world + src) * cap_hits * sizeof(mtsvgpu_hit);
  }
  __host__ __device__ uint64_t total_bytes() const { return hits_off(2, 0); }
};

struct PeerTable {
  uint8_t* base[kMaxRanks];
};

struct HandleBlob {  // what the ranks hand to each other (MTSVGPU_COMM_HANDLE_BYTES)
  uint32_t magic, rank, world, reserved;
  uint64_t max_local_reads, cap_hits;
  cudaIpcMemHandle_t mem;
  uint8_t pad[MTSVGPU_COMM_HANDLE_BYTES - 32 - sizeof(cudaIpcMemHandle_t)];
};
static_assert(sizeof(HandleBlob) == MTSVGPU_COMM_HANDLE_BYTES, "handle blob size");

__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

__host__ __device__ inline uint64_t range_bound(uint64_t n_reads, uint64_t step, uint32_t d) {
  const uint64_t b = (uint64_t)d * step;
  return b < n_reads ? b : n_reads;
}

// does every range fit its slot?  If not, tell everybody (all ranks must fail the batch together).
__global__ void chunk_check_kernel(PeerTable pt, CommLayout lay, const uint64_t* __restrict__ hit_off, uint64_t n_reads,
                                   uint64_t step, uint32_t rank, uint32_t epoch, uint32_t* __restrict__ overflow) {
  const uint32_t d = threadIdx.x;
  if (d >= lay.world) return;
  const uint64_t lo = range_bound(n_reads, step, d), hi = range_bound(n_reads, step, d + 1);
  if (hit_off[hi] - hit_off[lo] > lay.cap_hits || hi - lo > lay.max_local_reads) {
    *overflow = 1;
    for (uint32_t p = 0; p < lay.world; ++p)
      st_release_sys(&reinterpret_cast<CommHeader*>(pt.base[p])->error[rank], epoch);
  }
}

// blockIdx.y = destination rank: its range's hits (contiguous in the CSR output) and per-read counts go into my
// slot of its buffer, 8-byte stores over NVLink
__global__ void __launch_bounds__(256) chunk_push_kernel(PeerTable pt, CommLayout lay, const mtsvgpu_hit* __restrict__ hits,
                                                         const uint64_t* __restrict__ hit_off, uint64_t n_reads,
                                                         uint64_t step, uint32_t rank, uint32_t parity,
                                                         const uint32_t* __restrict__ overflow) {
  if (*overflow) return;
  const uint32_t d = blockIdx.y;
  const uint64_t lo = range_bound(n_reads, step, d), hi = range_bound(n_reads, step, d + 1);
  const uint64_t h0 = hit_off[lo], cnt = hit_off[hi] - h0;
  uint8_t* peer = pt.base[d];
  const uint64_t tid = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x, nthr = (uint64_t)gridDim.x * blockDim.x;
  const uint64_t* src = reinterpret_cast<const uint64_t*>(hits + h0);
  uint64_t* dst = reinterpret_cast<uint64_t*>(peer + lay.hits_off(parity, rank));
  const uint64_t words = cnt * 3;
  // the slot is 16-byte aligned, the span starts on an 8-byte boundary: 16-byte stores when both agree, four in
  // flight per thread (the NVLink round trip is what has to be covered)
  if ((reinterpret_cast<uintptr_t>(src) & 15) == 0) {
    const uint64_t pairs = words >> 1;
    const ulonglong2* s2 = reinterpret_cast<const ulonglong2*>(src);
    ulonglong2* d2 = reinterpret_cast<ulonglong2*>(dst);
    uint64_t i = tid;
    for (; i + 3 * nthr < pairs; i += 4 * nthr) {
      const ulonglong2 a = s2[i], b = s2[i + nthr], c2 = s2[i + 2 * nthr], e = s2[i + 3 * nthr];
      d2[i] = a;
      d2[i + nthr] = b;
      d2[i + 2 * nthr] = c2;
      d2[i + 3 * nthr] = e;
    }
    for (; i < pairs; i += nthr) d2[i] = s2[i];
    if (tid == 0 && (words & 1)) dst[words - 1] = src[words - 1];
  } else {
    for (uint64_t i = tid; i < words; i += nthr) dst[i] = src[i];
  }
  uint32_t* cdst = reinterpret_cast<uint32_t*>(peer + lay.counts_off(parity, rank));
  for (uint64_t i = tid; i < hi - lo; i += nthr) cdst[i] = (uint32_t)(hit_off[lo + i + 1] - hit_off[lo + i]);
  if (tid == 0) reinterpret_cast<CommHeader*>(peer)->slot_hits[parity][rank] = cnt;
  __threadfence_system();
}

// every pushing thread fenced its own stores at system scope before the push kernel ended, and this kernel starts
// after that one has completed; the flag itself is a system-scope release store
__global__ void chunk_signal_kernel(PeerTable pt, uint32_t world, uint32_t rank, uint32_t epoch) {
  const uint32_t d = threadIdx.x;
  if (d >= world) return;
  st_release_sys(&reinterpret_cast<CommHeader*>(pt.base[d])->flags[rank], epoch);
}

// status: 0 ok, 1 a rank overflowed its slot, 2 timed out waiting for a peer
__global__ void chunk_wait_kernel(uint8_t* my_base, uint32_t world, uint32_t epoch, long long timeout_cycles,
                                  uint32_t* __restrict__ status, volatile uint32_t* __restrict__ host_status) {
  const uint32_t s = threadIdx.x;
  __shared__ uint32_t st;
  if (s == 0) st = 0;
  __syncthreads();
  if (s < world) {
    const CommHeader* h = reinterpret_cast<const CommHeader*>(my_base);
    const long long t0 = clock64();
    while ((int32_t)(ld_acquire_sys(&h->flags[s]) - epoch) < 0) {
      if (clock64() - t0 > timeout_cycles) {
        atomicMax(&st, 2u);
        break;
      }
      __nanosleep(200);
    }
    if (ld_acquire_sys(&h->error[s]) == epoch) atomicMax(&st, 1u);
  }
  __syncthreads();
  if (s == 0) {
    *status = st;
    *host_status = st;
    __threadfence_system();
  }
}

}  // namespace
}  // namespace mtsv

using namespace mtsv;

struct mtsvgpu_comm {
  int device = 0;
  uint32_t rank = 0, world = 0;
  CommLayout lay{};
  DevPtr<uint8_t> base;     // my buffer
  PeerTable peers{};        // peers' buffers as mapped into this process (base[rank] = base)
  bool connected = false;
  uint32_t epoch = 0;
  long long timeout_cycles = 60000000000ll;  // set from the SM clock at creation (the attribute query is a slow driver call)
  DevPtr<uint32_t> d_status;        // [0] wait status, [1] overflow flag
  PinnedPtr<uint32_t> h_status;     // mapped copy of the wait status
  uint32_t* h_status_dev = nullptr;
  DevPtr<uint64_t> d_n_out;
  DevPtr<mtsvgpu_taxhit> out;       // merged result of the last batch (capacity world * cap_hits)
  DevPtr<uint64_t> out_off;
  CollapseScratch scratch;
};

namespace mtsv {

void comm_destroy(mtsvgpu_comm* c) {
  if (!c) return;
  cudaSetDevice(c->device);
  cudaDeviceSynchronize();
  for (uint32_t p = 0; p < c->world; ++p)
    if (p != c->rank && c->peers.base[p]) cudaIpcCloseMemHandle(c->peers.base[p]);
  delete c;
}

int comm_create(int device, uint32_t rank, uint32_t world, uint64_t max_local_reads, uint64_t max_hits_per_source,
                mtsvgpu_comm** out, uint8_t* handle_out) {
  if (!out || !handle_out) return set_error(MTSVGPU_EINVAL, "null argument");
  *out = nullptr;
  if (world == 0 || world > kMaxRanks || rank >= world)
    return set_error(MTSVGPU_EINVAL, "bad rank / world (at most %u ranks)", kMaxRanks);
  if (max_local_reads == 0 || max_hits_per_source == 0) return set_error(MTSVGPU_EINVAL, "capacities must be > 0");
  if (max_local_reads > 0x7ffffff0ull || max_hits_per_source * world > 0xfffffff0ull)
    return set_error(MTSVGPU_ELIMIT, "comm capacities exceed 32-bit merge offsets");
  MTSV_TRY(use_device(device));
  std::unique_ptr<mtsvgpu_comm, void (*)(mtsvgpu_comm*)> guard(new mtsvgpu_comm, comm_destroy);
  mtsvgpu_comm* c = guard.get();
  c->device = device;
  c->rank = rank;
  c->world = world;
  c->lay.world = world;
  c->lay.max_local_reads = max_local_reads;
  c->lay.cap_hits = max_hits_per_source;
  MTSV_TRY(dev_alloc(c->base, c->lay.total_bytes()));
  // header and per-read counts start at zero: a slot that was never (or not this batch) written reads as "no hits"
  MTSV_CUDA_TRY(cudaMemset(c->base.get(), 0, c->lay.hits_base()));
  MTSV_TRY(dev_alloc(c->d_status, 4));
  MTSV_CUDA_TRY(cudaMemset(c->d_status.get(), 0, 16));
  MTSV_TRY(dev_alloc(c->d_n_out, 1));
  MTSV_TRY(pinned_alloc(c->h_status, 4, cudaHostAllocMapped));
  MTSV_CUDA_TRY(cudaHostGetDevicePointer((void**)&c->h_status_dev, c->h_status.get(), 0));
  MTSV_TRY(dev_alloc(c->out, (uint64_t)world * max_hits_per_source + 1));
  MTSV_TRY(dev_alloc(c->out_off, max_local_reads + 1));
  MTSV_CUDA_TRY(cudaDeviceSynchronize());
  {
    int clock_khz = 2000000;
    if (cudaDeviceGetAttribute(&clock_khz, cudaDevAttrClockRate, device) != cudaSuccess) (void)cudaGetLastError();
    c->timeout_cycles = (long long)clock_khz * 1000ll * 30ll;
  }
  HandleBlob blob;
  memset(&blob, 0, sizeof blob);
  blob.magic = kCommMagic;
  blob.rank = rank;
  blob.world = world;
  blob.max_local_reads = max_local_reads;
  blob.cap_hits = max_hits_per_source;
  MTSV_CUDA_TRY(cudaIpcGetMemHandle(&blob.mem, c->base.get()));
  memcpy(handle_out, &blob, sizeof blob);
  c->peers.base[rank] = c->base.get();
  *out = guard.release();
  return 0;
}

// all_handles: world blobs in rank order (every rank's own included), however the host moved them around
int comm_connect(mtsvgpu_comm* c, const uint8_t* all_handles) {
  if (!c || !all_handles) return set_error(MTSVGPU_EINVAL, "null argument");
  if (c->connected) return set_error(MTSVGPU_EINVAL, "communicator is already connected");
  MTSV_CUDA_TRY(cudaSetDevice(c->device));
  for (uint32_t p = 0; p < c->world; ++p) {
    HandleBlob blob;
    memcpy(&blob, all_handles + (size_t)p * MTSVGPU_COMM_HANDLE_BYTES, sizeof blob);
    if (blob.magic != kCommMagic || blob.rank != p || blob.world != c->world ||
        blob.max_local_reads != c->lay.max_local_reads || blob.cap_hits != c->lay.cap_hits)
      return set_error(MTSVGPU_EINVAL, "handle %u does not belong to this communicator (rank, world or capacities differ)", p);
    if (p == c->rank) continue;
    void* ptr = nullptr;
    cudaError_t e = cudaIpcOpenMemHandle(&ptr, blob.mem, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) {
      (void)cudaGetLastError();
      return set_error(MTSVGPU_ECUDA, "cudaIpcOpenMemHandle of rank %u's buffer failed: %s (peer access over NVLink is required)",
                       p, cudaGetErrorString(e));
    }
    c->peers.base[p] = (uint8_t*)ptr;
  }
  c->connected = true;
  return 0;
}

// One batch.  Every rank passes the same reads (device memory) and its own chunk's index.
int bin_batch_chunked(mtsvgpu_index* h, mtsvgpu_comm* c, const uint8_t* d_seqs, const uint64_t* d_seq_off,
                      uint64_t n_reads, const mtsvgpu_params* params, uint64_t* first_read, uint64_t* n_local_reads,
                      const mtsvgpu_taxhit** d_out, const uint64_t** d_out_off, uint64_t* n_out) {
  if (!h || !c) return set_error(MTSVGPU_EINVAL, "null argument");
  if (!c->connected && c->world > 1) return set_error(MTSVGPU_EINVAL, "communicator is not connected");
  if (h->ix.device != c->device) return set_error(MTSVGPU_EINVAL, "index and communicator live on different devices");
  const uint64_t step = (n_reads + c->world - 1) / c->world;
  const uint64_t lo = range_bound(n_reads, step, c->rank), hi = range_bound(n_reads, step, c->rank + 1);
  if (step > c->lay.max_local_reads)
    return set_error(MTSVGPU_ELIMIT, "%llu reads per rank exceed the communicator's max_local_reads %llu",
                     (unsigned long long)step, (unsigned long long)c->lay.max_local_reads);
  // ---- this chunk's hits for all reads (a plain single-index run) ----
  const void* d_recs = nullptr;
  const uint64_t* d_hit_off = nullptr;
  uint64_t n_hits = 0;
  MTSV_TRY(bin_batch_device(h, d_seqs, d_seq_off, n_reads, nullptr, BatchOutput::Hits, params, &d_recs, &d_hit_off,
                            &n_hits));
  const mtsvgpu_hit* d_hits = static_cast<const mtsvgpu_hit*>(d_recs);
  cudaStream_t st = h->stream;
  static const bool trace = getenv("MTSV_B200_TRACE") != nullptr;  // phase times on stderr
  cudaEvent_t ev[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
  if (trace) {
    for (auto& e : ev) cudaEventCreate(&e);
    cudaEventRecord(ev[0], st);
  }
  // ---- exchange: my hits of range d into rank d's buffer, flag, wait for everybody's flags here ----
  const uint32_t epoch = ++c->epoch, parity = epoch & 1u;
  uint32_t* d_overflow = c->d_status.get() + 1;
  MTSV_CUDA_TRY(cudaMemsetAsync(d_overflow, 0, 4, st));
  MTSV_LAUNCH(chunk_check_kernel, 1, 32, 0, st, c->peers, c->lay, d_hit_off, n_reads, step, c->rank, epoch, d_overflow);
  {
    const uint64_t per_dest = std::max<uint64_t>(step, (n_hits / c->world + 1) * 3);
    unsigned gx = (unsigned)std::min<uint64_t>(sm_count() * 2, (per_dest + 2047) / 2048);
    if (gx == 0) gx = 1;
    MTSV_LAUNCH(chunk_push_kernel, dim3(gx, c->world), 256, 0, st, c->peers, c->lay, d_hits, d_hit_off, n_reads, step,
                c->rank, parity, d_overflow);
  }
  if (trace) cudaEventRecord(ev[1], st);
  MTSV_LAUNCH(chunk_signal_kernel, 1, 32, 0, st, c->peers, c->world, c->rank, epoch);
  const long long timeout_cycles = c->timeout_cycles;  // 30 s: a peer that never arrives is an error
  if (trace) cudaEventRecord(ev[4], st);
  MTSV_LAUNCH(chunk_wait_kernel, 1, 32, 0, st, c->base.get(), c->world, epoch, timeout_cycles, c->d_status.get(),
              c->h_status_dev);
  if (trace) cudaEventRecord(ev[2], st);
  // ---- merge epilogue over the world slots of my range (src/collapse.rs:597-602) ----
  const mtsvgpu_hit* part_hits[kMaxRanks];
  const uint32_t* part_counts[kMaxRanks];
  for (uint32_t s = 0; s < c->world; ++s) {
    part_hits[s] = reinterpret_cast<const mtsvgpu_hit*>(c->base.get() + c->lay.hits_off(parity, s));
    part_counts[s] = reinterpret_cast<const uint32_t*>(c->base.get() + c->lay.counts_off(parity, s));
  }
  // (a failed exchange leaves slots untouched: they hold the whole, in-range lists of an earlier batch or the
  // zeros they were created with, so the merge below stays in bounds; its result is discarded)
  MTSV_TRY(collapse_taxid_async(c->scratch, st, c->world, part_hits, part_counts, (uint32_t)(hi - lo),
                                (uint64_t)c->world * c->lay.cap_hits, c->out.get(), c->out_off.get(), c->d_n_out.get()));
  if (trace) cudaEventRecord(ev[3], st);
  uint64_t total = 0;
  MTSV_CUDA_TRY(cudaMemcpyAsync(&total, c->d_n_out.get(), 8, cudaMemcpyDeviceToHost, st));
  MTSV_CUDA_TRY(cudaStreamSynchronize(st));  // the batch's one host synchronisation after the local binning
  if (trace) {
    float a = 0, b = 0, d = 0, sg = 0;
    cudaEventElapsedTime(&a, ev[0], ev[1]);
    cudaEventElapsedTime(&sg, ev[1], ev[4]);
    cudaEventElapsedTime(&b, ev[4], ev[2]);
    cudaEventElapsedTime(&d, ev[2], ev[3]);
    fprintf(stderr, "[mtsv_b200 trace] rank %u chunked batch: %llu hits, push %.3f ms, signal %.3f ms, wait %.3f ms, merge %.3f ms\n",
            c->rank, (unsigned long long)n_hits, a, sg, b, d);
    for (auto& e : ev) cudaEventDestroy(e);
  }
  const uint32_t status = *c->h_status;
  if (status == 1)
    return set_error(MTSVGPU_ELIMIT, "chunk exchange: a rank produced more hits for one read range than max_hits_per_source "
                                     "(%llu); recreate the communicator with a larger capacity", (unsigned long long)c->lay.cap_hits);
  if (status == 2) return set_error(MTSVGPU_ECUDA, "chunk exchange: timed out waiting for a peer rank's data");
  if (first_read) *first_read = lo;
  if (n_local_reads) *n_local_reads = hi - lo;
  if (d_out) *d_out = c->out.get();
  if (d_out_off) *d_out_off = c->out_off.get();
  if (n_out) *n_out = total;
  return 0;
}

}  // namespace mtsv
