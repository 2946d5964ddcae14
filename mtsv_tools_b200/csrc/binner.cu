// binner.cu — the read-assignment hot path as a chain of sm_100a kernels.
//
// Replaces the worker closure of run_fastx_pipeline (src/binner.rs:77-131) and
// MGIndex::matching_tax_ids (src/index.rs:258-432) for a whole batch of reads:
//
//   count/scan      seed slots per read-strand ("query")
//   seed_search     one thread per seed slot: k-mer table lookup + rank steps     [HBM random sectors]
//   seed_select     one thread per query: replay the max-hits / tune-max-hits rule
//   locate          SA lookups (or LF walks when the SA is kept sampled)           [HBM random sectors]
//   sort            segmented sort of (ref_pos, q_off) keys per query
//   coalesce        one thread per query: windows + merge                          (src/index.rs:435-487)
//   rank            segmented sort by num_seeds, compaction to a dense candidate list
//   verify          one thread per candidate: Myers bit-vector edit distance       [SM integer issue]
//   select/emit     one thread per query: per-TaxID first pass, limits, CSR output
//
// All per-item arithmetic lives in core.cuh (shared with the CPU emulation tests).
#include <algorithm>
#include <thread>

#include "ctx.h"

#ifndef MTSV_COALESCE_UNROLL
#define MTSV_COALESCE_UNROLL 4
#endif
#ifndef MTSV_COALESCE_TILES
#define MTSV_COALESCE_TILES 4
#endif
constexpr int kCoalesceTiles = MTSV_COALESCE_TILES;    // tiles of 32 hits fetched together by coalesce_warp
constexpr int kCoalesceUnroll = MTSV_COALESCE_UNROLL;  // replay loop of coalesce_warp (code size vs shuffle look-ahead)

namespace mtsv {

// ------------------------------------------------------------------------------------------
// small kernels
// ------------------------------------------------------------------------------------------
constexpr uint32_t kMaxReadLenDev = MTSVGPU_MAX_READ_LEN;  // longer reads get no seeds, hence no hits; they are counted

// adds `v` of every thread of the CTA into one of 32 counters with a single global atomic per CTA
__device__ __forceinline__ void cta_accumulate(unsigned long long* counters32, unsigned int v) {
  __shared__ unsigned int cta_sum;
  if (threadIdx.x == 0) cta_sum = 0;
  __syncthreads();
  unsigned int w = __reduce_add_sync(0xffffffffu, v);
  if ((threadIdx.x & 31) == 0 && w) atomicAdd(&cta_sum, w);
  __syncthreads();
  if (threadIdx.x == 0 && cta_sum) atomicAdd(&counters32[blockIdx.x & 31], (unsigned long long)cta_sum);
}

__global__ void count_slots_kernel(ReadsView rv, Params p, uint32_t nq, uint32_t* __restrict__ q_nslots,
                                   BatchCounters* __restrict__ ctr) {
  uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t L = 0;
  if (q < nq) {
    uint64_t r = rv.read0 + q / p.ns;
    uint64_t a = rv.seq_off[r], b = rv.seq_off[r + 1];
    if (b < a || b - a > 0xffffffffull) {  // not monotone: treat as empty and flag the batch
      atomicExch(&ctr->bad_offsets, 1u);
    } else {
      L = (uint32_t)(b - a);
    }
    if (L > kMaxReadLenDev) {  // over the documented limit: this read is left out (stats.n_reads_over_limit)
      if (q % p.ns == 0) atomicAdd(&ctr->n_over_len, 1u);
      L = 0;
    }
    q_nslots[q] = seed_slots(L, p.S, p.G);
  }
  // block max of L -> one atomic per block
  __shared__ unsigned int smax, simin;
  if (threadIdx.x == 0) smax = simin = 0;
  __syncthreads();
  unsigned int wmax = __reduce_max_sync(0xffffffffu, L);
  unsigned int wimin = __reduce_max_sync(0xffffffffu, q < nq ? ~L : 0u);  // ~(shortest read)
  if ((threadIdx.x & 31) == 0) {
    atomicMax(&smax, wmax);
    atomicMax(&simin, wimin);
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    atomicMax(&ctr->max_len, smax);
    atomicMax(&ctr->inv_min_len, simin);
  }
}

__global__ void expand_slots_kernel(const uint32_t* __restrict__ slot_off, uint32_t nq,
                                    uint32_t* __restrict__ slot_q) {
  uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= nq) return;
  uint32_t b = slot_off[q], e = slot_off[q + 1];
  for (uint32_t s = b; s < e; ++s) slot_q[s] = q;
}

// read encoding: one thread per (read, 64-base word).  Streaming: reads the batch's bytes once, writes
// 24 B per 64 bases and strand.
__global__ void __launch_bounds__(256) encode_fwd_kernel(ReadsView rv, ReadWord* __restrict__ words,
                                                         uint32_t w_max, int raw) {
  // one warp per (read, word): two coalesced 32-byte loads, the planes come out of warp ballots
  uint64_t t = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const unsigned lane = threadIdx.x & 31;
  uint32_t r = (uint32_t)(t / w_max), w = (uint32_t)(t % w_max);
  if (r >= rv.n_reads) return;
  uint64_t a = rv.seq_off[rv.read0 + r], b = rv.seq_off[rv.read0 + r + 1];
  uint32_t L = (uint32_t)(b - a);
  if (w * 64 >= L) return;
  const uint8_t* seq = rv.seqs + a;
  ReadWord out{0, 0, 0};
#pragma unroll
  for (int half = 0; half < 2; ++half) {
    uint32_t pos = w * 64 + half * 32 + lane;
    bool in = pos < L;
    uint8_t byte = in ? __ldg(seq + pos) : (uint8_t)'A';
    uint32_t c = raw ? text_code(byte) : read_code(byte);
    bool is_base = c < 4;
    uint32_t lo = __ballot_sync(0xffffffffu, in && ((is_base && (c & 1)) || (raw && c > 4)));
    uint32_t hi = __ballot_sync(0xffffffffu, in && is_base && (c & 2));
    uint32_t nn = __ballot_sync(0xffffffffu, in && !is_base);
    out.lo |= (uint64_t)lo << (32 * half);
    out.hi |= (uint64_t)hi << (32 * half);
    out.nn |= (uint64_t)nn << (32 * half);
  }
  if (lane == 0) {
    uint32_t woff = (uint32_t)((a - rv.seq_off[rv.read0]) >> 6) + r;
    words[woff + w] = out;
  }
}

__global__ void __launch_bounds__(256) encode_rc_kernel(ReadsView rv, ReadWord* __restrict__ words,
                                                        uint32_t total_words, uint32_t w_max) {
  uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t r = (uint32_t)(t / w_max), w = (uint32_t)(t % w_max);
  if (r >= rv.n_reads) return;
  uint64_t a = rv.seq_off[rv.read0 + r], b = rv.seq_off[rv.read0 + r + 1];
  uint32_t L = (uint32_t)(b - a);
  if (w * 64 >= L) return;
  uint32_t woff = (uint32_t)((a - rv.seq_off[rv.read0]) >> 6) + r;
  words[total_words + woff + w] = encode_rc_word(words + woff, L, w);
}

// forward strand of the binner's reads: one thread per read, eight bases per step with SWAR
// (core.cuh::encode8) on 8-byte aligned loads; ~30x fewer instructions than a byte-per-lane encoder.
__global__ void __launch_bounds__(128) encode_reads_kernel(ReadsView rv, ReadWord* __restrict__ words) {
  const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= rv.n_reads) return;
  const uint64_t a = rv.seq_off[rv.read0 + r], b = rv.seq_off[rv.read0 + r + 1];
  const uint32_t L = (uint32_t)(b - a);
  const uint32_t W = (L + 63) >> 6;
  const uint32_t woff = (uint32_t)((a - rv.seq_off[rv.read0]) >> 6) + r;
  const uint64_t addr = (uint64_t)(rv.seqs + a);
  const uint64_t* wp = reinterpret_cast<const uint64_t*>(addr & ~7ull);
  const uint32_t boff = (uint32_t)(addr & 7ull);
  for (uint32_t w = 0; w < W; ++w) {
    ReadWord out{0, 0, 0};
#pragma unroll
    for (uint32_t c = 0; c < 8; ++c) {
      uint32_t pos = w * 64 + c * 8;
      if (pos < L) {
        uint32_t nvalid = L - pos < 8 ? L - pos : 8;
        uint32_t first = boff + pos, last = first + nvalid - 1;
        uint64_t x = __ldg(wp + (first >> 3)) >> ((first & 7) * 8);
        if ((last >> 3) != (first >> 3)) x |= __ldg(wp + (last >> 3)) << (64 - (first & 7) * 8);
        uint32_t lo, hi, nn;
        encode8(x, &lo, &hi, &nn);
        uint32_t m = (1u << nvalid) - 1;
        out.lo |= (uint64_t)(lo & m) << (c * 8);
        out.hi |= (uint64_t)(hi & m) << (c * 8);
        out.nn |= (uint64_t)(nn & m) << (c * 8);
      }
    }
    words[woff + w] = out;
  }
}

// packed input: the planes come from the host parser (core.cuh "packed reads"); one thread per read lays its
// record out as ReadWords.  rel == nullptr: every read has the same length, records are `uni_rec` bytes apart.
__global__ void __launch_bounds__(128) packed_sizes_kernel(ReadsView rv, uint32_t* __restrict__ rel) {
  const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= rv.n_reads) return;
  rel[r] = packed_record_bytes((uint32_t)(rv.seq_off[rv.read0 + r + 1] - rv.seq_off[rv.read0 + r]));
}
__global__ void __launch_bounds__(128) unpack_reads_kernel(ReadsView rv, const uint8_t* __restrict__ packed,
                                                           uint32_t uni_rec, const uint32_t* __restrict__ rel,
                                                           ReadWord* __restrict__ words) {
  const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= rv.n_reads) return;
  const uint64_t a = rv.seq_off[rv.read0 + r], b = rv.seq_off[rv.read0 + r + 1];
  const uint32_t L = (uint32_t)(b - a);
  const uint32_t W = (L + 63) >> 6;
  const uint32_t woff = (uint32_t)((a - rv.seq_off[rv.read0]) >> 6) + r;
  const uint8_t* rec = packed + (rel ? (uint64_t)rel[r] : (uint64_t)r * uni_rec);
  for (uint32_t w = 0; w < W; ++w) words[woff + w] = unpack_word(rec, L, w);
}

// seed search: one thread per slot.  Each thread owns one dependent chain of sector fetches;
// ~2048 chains per SM keep the HBM random-access pipeline full.
__global__ void __launch_bounds__(256) seed_search_kernel(FmView fm, KtabView kt, ReadsView rv, EncView ev, Params p,
                                                          const uint32_t* __restrict__ slot_off,
                                                          const uint32_t* __restrict__ slot_q,
                                                          uint32_t n_slots,
                                                          uint32_t* __restrict__ slot_lo,
                                                          uint32_t* __restrict__ slot_cnt,
                                                          BatchCounters* __restrict__ ctr, int count_ranks,
                                                          uint32_t uni_len, uint32_t uni_spq) {
  // uni_spq != 0: every read of the sub-batch has uni_len bases, so a slot's query, seed offset and plane words
  // follow from its index alone (no slot_q / slot_off / seq_off loads in front of the index accesses)
  uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t steps = 0;
  if (s < n_slots) {
    uint32_t q, j, L, woff;
    if (uni_spq) {
      q = s / uni_spq;
      j = s - q * uni_spq;
      L = uni_len;
      const uint32_t r = q / p.ns;
      woff = (uint32_t)(((uint64_t)r * L) >> 6) + r + (q % p.ns) * ev.total_words;
    } else {
      q = slot_q[s];
      j = s - slot_off[q];
      L = query_len(rv, p.ns, q);
      woff = query_word_off(rv, ev, p.ns, q);
    }
    uint32_t lo, cnt;
    seed_search_item(fm, kt, ev.words + woff, L, p.S, j * p.G, &lo, &cnt, &steps);
    slot_lo[s] = lo;
    slot_cnt[s] = cnt;
  }
  if (count_ranks) cta_accumulate(ctr->rank_steps, steps);
}

__global__ void seed_select_kernel(ReadsView rv, EncView ev, Params p, const uint32_t* __restrict__ slot_off,
                                   uint32_t nq, const uint32_t* __restrict__ slot_cnt,
                                   uint32_t* __restrict__ slot_hoff, uint32_t* __restrict__ q_nseeds,
                                   uint32_t* __restrict__ q_nhits, BatchCounters* __restrict__ ctr) {
  uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= nq) return;
  uint32_t b = slot_off[q], e = slot_off[q + 1];
  uint32_t ns = 0, nh = 0, ovf = 0;
  seed_select_item(p, e - b, slot_cnt + b, slot_hoff + b, &ns, &nh, &ovf);
  if (nh != 0) {  // (only strands with hits need the look at their bases)
    const uint32_t L = query_len(rv, p.ns, q);
    if (query_hopeless(ev.words + query_word_off(rv, ev, p.ns, q), L, edit_budget(L, p.edit_rate))) {
      for (uint32_t j = b; j < e; ++j) slot_hoff[j] = kUnused;
      ns = nh = ovf = 0;
    }
  }
  if (ovf) {  // more seed hits than a strand may hold: the strand is left out (stats.n_strands_over_hits)
    for (uint32_t j = b; j < e; ++j) slot_hoff[j] = kUnused;
    ns = nh = 0;
    atomicAdd(&ctr->overflow, 1u);
  }
  q_nseeds[q] = ns;
  q_nhits[q] = nh;
}

// locate: one lane per query, walking its seed slots (most slots carry no hit, and with the k-mer table's
// direct entries most hits already are text positions: a lane per slot would spend its time finding that
// out).  Intervals with more than a few rows are spread over the warp so that consecutive SA entries are read
// coalesced and long LF walks are shared.
__global__ void __launch_bounds__(256) locate_kernel(FmView fm, SaView sv, Params p,
                                                     const uint32_t* __restrict__ slot_off, uint32_t nq,
                                                     const uint32_t* __restrict__ slot_lo,
                                                     const uint32_t* __restrict__ slot_cnt,
                                                     const uint32_t* __restrict__ slot_hoff,
                                                     const uint32_t* __restrict__ hit_off,
                                                     const uint32_t* __restrict__ q_nhits,
                                                     uint64_t* __restrict__ hit_keys) {
  const uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
  const unsigned lane = threadIdx.x & 31;
  uint32_t b = 0, n_slots = 0, base = 0;
  if (q < nq && q_nhits[q] != 0) {
    b = slot_off[q];
    n_slots = slot_off[q + 1] - b;
    base = hit_off[q];
  }
  const uint32_t n_max = __reduce_max_sync(0xffffffffu, n_slots);
  constexpr uint32_t kSolo = 4;
  // (handling several slots of a lane together so that their SA reads overlap was measured slower: 2.7 vs 1.7 ms)
  for (uint32_t j = 0; j < n_max; ++j) {
    uint32_t cnt = 0, lo = 0, dst = 0;
    const uint32_t qoff = j * p.G;
    if (j < n_slots) {
      const uint32_t ho = slot_hoff[b + j];
      if (ho != kUnused) {
        cnt = slot_cnt[b + j];
        lo = slot_lo[b + j];
        dst = base + ho;
      }
    }
    if (cnt & kDirectHit) {  // the k-mer table already gave the text position (core.cuh, direct entries)
      hit_keys[dst] = make_hit_key(lo, qoff);
      cnt = 0;
    }
    if (cnt <= kSolo) {
      for (uint32_t r = 0; r < cnt; ++r)
        hit_keys[dst + r] = make_hit_key(fm_locate(fm, sv, lo + r, nullptr), qoff);
    }
    unsigned big = __ballot_sync(0xffffffffu, cnt > kSolo);
    while (big) {
      int src = __ffs(big) - 1;
      big &= big - 1;
      uint32_t c = __shfl_sync(0xffffffffu, cnt, src);
      uint32_t l = __shfl_sync(0xffffffffu, lo, src);
      uint32_t d = __shfl_sync(0xffffffffu, dst, src);
      for (uint32_t r = lane; r < c; r += 32)
        hit_keys[d + r] = make_hit_key(fm_locate(fm, sv, l + r, nullptr), qoff);
    }
  }
}

// ------------------------------------------------------------------------------------------
// segmented sort of u64 keys: bitonic network in its "all ascending" form (first step of each
// merge compares i with its mirror i ^ (k-1)), which tolerates virtual +inf padding, so segment
// lengths need not be powers of two.  Segment q = keys[seg_off[q] .. + seg_cnt[q]).
//   <= 32 keys : one warp, registers + shuffles
//   <= 4096    : one CTA, shared memory
//   larger     : one CTA, in place in global memory (rare: > 4096 seed hits for one read-strand)
// ------------------------------------------------------------------------------------------
constexpr uint32_t kSortMedium = 4096;
constexpr uint32_t kLightItems = 16;  // segments this small are ordered by their consumer's own lane
constexpr uint32_t kMonsterHits = 1024;  // strands with more seed hits than this get a whole CTA in coalesce

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
                                                            BatchCounters* __restrict__ ctr) {
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
                                                        const BatchCounters* __restrict__ ctr) {
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
                                                          const BatchCounters* __restrict__ ctr) {
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
                                                          const BatchCounters* __restrict__ ctr) {
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

// ------------------------------------------------------------------------------------------
// coalesce / rank
// ------------------------------------------------------------------------------------------
// Queries with few items are handled by their own lane; a query with many items (a read whose seeds
// hit thousands of loci) is handled by the whole warp so that one heavy read does not serialise 31
// idle lanes behind it.  Heavy queries are taken one after the other (ballot loop).

// Batcher's odd-even merge sort as a register sorting network (written out: 63 compare-exchanges for 16 keys, verified with the 0-1 principle), the same for every lane, so a warp whose lanes hold
// differently ordered lists does not diverge (an insertion sort here cost 60 % of coalesce_kernel).
__device__ __forceinline__ void sort_network16(uint64_t (&v)[16]) {
#define CE(a, b)                      \
  {                                   \
    uint64_t x_ = v[a], y_ = v[b];    \
    v[a] = x_ < y_ ? x_ : y_;         \
    v[b] = x_ < y_ ? y_ : x_;         \
  }
  CE(0, 1) CE(2, 3) CE(4, 5) CE(6, 7) CE(8, 9) CE(10, 11) CE(12, 13) CE(14, 15)
  CE(0, 2) CE(1, 3) CE(4, 6) CE(5, 7) CE(8, 10) CE(9, 11) CE(12, 14) CE(13, 15)
  CE(1, 2) CE(5, 6) CE(9, 10) CE(13, 14) CE(0, 4) CE(1, 5) CE(2, 6) CE(3, 7)
  CE(8, 12) CE(9, 13) CE(10, 14) CE(11, 15) CE(2, 4) CE(3, 5) CE(10, 12) CE(11, 13)
  CE(1, 2) CE(3, 4) CE(5, 6) CE(9, 10) CE(11, 12) CE(13, 14) CE(0, 8) CE(1, 9)
  CE(2, 10) CE(3, 11) CE(4, 12) CE(5, 13) CE(6, 14) CE(7, 15) CE(4, 8) CE(5, 9)
  CE(6, 10) CE(7, 11) CE(2, 4) CE(3, 5) CE(6, 8) CE(7, 9) CE(10, 12) CE(11, 13)
  CE(1, 2) CE(3, 4) CE(5, 6) CE(7, 8) CE(9, 10) CE(11, 12) CE(13, 14)
#undef CE
}

__device__ __forceinline__ bool carry_valid_or_lane(unsigned lane, bool carry_valid) {
  return lane > 0 || carry_valid;  // lane 0 compares with the previous tile's last hit, if there is one
}

// coalesce_seed_sites (src/index.rs:435-487) with the warp: lanes compute bins and windows of 32
// hits at a time, then every lane replays the (cheap, inherently sequential) merge automaton on the
// shuffled windows so that control flow stays uniform; lane 0 writes.
__device__ uint32_t coalesce_warp(const BinsView& bv, const uint64_t* __restrict__ keys, uint32_t n_hits,
                                  uint32_t min_seeds, uint32_t L, uint32_t k, CandRec* __restrict__ cand) {
  const unsigned lane = threadIdx.x & 31;
  uint32_t nc = 0;
  bool have = false;
  CandRec cur{0, 0, 0, 0};
  uint32_t carry_site = 0, carry_bin = 0;  // last hit of the previous tile
  bool carry_valid = false;
  // The automaton itself is cheap; what a long strand waits for is memory (keys, bins).  Four tiles of
  // 32 hits are therefore fetched together — the four key loads and the four branch-free binary searches
  // over the bin ends proceed in lock step, i.e. with four loads in flight — and then replayed in order.
  constexpr int U = kCoalesceTiles;
  uint32_t top = 1;
  while (top < bv.n) top <<= 1;
  for (uint32_t g0 = 0; g0 < n_hits; g0 += 32 * U) {
    uint32_t site[U], qoff[U], b[U], ws[U], we[U];
    bool some[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      uint32_t h = g0 + u * 32 + lane;
      uint64_t key = h < n_hits ? keys[h] : 0;
      site[u] = (uint32_t)(key >> 16);
      qoff[u] = (uint32_t)(key & 0xffff);
      b[u] = 0;
    }
    // first bin with end > site == number of bins with end <= site (src/index.rs:455-458)
    for (uint32_t step = top; step >= 1; step >>= 1) {
#pragma unroll
      for (int u = 0; u < U; ++u) {
        uint32_t idx = b[u] + step;
        if (idx <= bv.n && ldg(&bv.end[idx - 1]) <= site[u]) b[u] = idx;
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      uint32_t h = g0 + u * 32 + lane;
      ws[u] = we[u] = 0;
      some[u] = false;
      if (h < n_hits) {
        if (b[u] >= bv.n) b[u] = bv.n - 1;  // cannot happen for a seed hit (it lies before the '$')
        some[u] = candidate_window(site[u], qoff[u], ldg(&bv.start[b[u]]), ldg(&bv.end[b[u]]), L, k, &ws[u], &we[u]);
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const uint32_t t0 = g0 + u * 32;
      if (t0 >= n_hits) break;
      const uint32_t h = t0 + lane;
      const uint32_t cnt = n_hits - t0 < 32 ? n_hits - t0 : 32;
      // Fast path.  A hit whose site lies >= 2(L+k) after its predecessor (or in another bin) cannot
      // overlap any window accumulated so far (windows reach at most L+k either side of their site and
      // hits are sorted by site), so it certainly starts a new candidate.  If that holds for every hit
      // of the tile the automaton degenerates: flush the incoming candidate, emit every hit but the last
      // as a single-seed candidate, carry the last.  Typical for reads whose seeds hit hundreds of
      // unrelated loci.
      uint32_t prev_site = __shfl_up_sync(0xffffffffu, site[u], 1);
      uint32_t prev_b = __shfl_up_sync(0xffffffffu, b[u], 1);
      if (lane == 0) {
        prev_site = carry_site;
        prev_b = carry_bin;
      }
      bool brk = h >= n_hits || !carry_valid_or_lane(lane, carry_valid) || b[u] != prev_b ||
                 (uint64_t)site[u] >= (uint64_t)prev_site + 2ull * ((uint64_t)L + k);
      bool all_break = __all_sync(0xffffffffu, brk);
      const uint32_t last_b = __shfl_sync(0xffffffffu, b[u], cnt - 1);
      carry_site = __shfl_sync(0xffffffffu, site[u], cnt - 1);
      carry_bin = last_b;
      carry_valid = true;
      if (all_break) {
        if (have && cur.num_seeds >= min_seeds) {
          if (lane == 0) {
            cand[nc] = cur;
          }
          ++nc;
        }
        bool emit = h + 1 < t0 + cnt && some[u] && 1u >= min_seeds;  // every hit of the tile except the last
        unsigned em = __ballot_sync(0xffffffffu, emit);
        if (emit) {
          uint32_t pos = nc + __popc(em & ((1u << lane) - 1));
          cand[pos] = CandRec{ws[u], we[u], b[u], 1};
        }
        nc += __popc(em);
        have = __shfl_sync(0xffffffffu, (int)some[u], cnt - 1) != 0;
        cur = CandRec{__shfl_sync(0xffffffffu, ws[u], cnt - 1), __shfl_sync(0xffffffffu, we[u], cnt - 1), last_b, 1};
        continue;
      }
      // (unrolled by 8 so that the shuffles, which do not depend on the automaton's state, are issued ahead of
      //  the short dependent chain through cur / have; the full 32-way unroll of round 1 made four copies of a
      //  2 700-instruction body — ncu: warps stalled on instruction fetch, `no_instruction` 10.8 per issue)
      const uint32_t sb = (b[u] << 1) | (some[u] ? 1u : 0u);
#pragma unroll(kCoalesceUnroll)
      for (uint32_t i = 0; i < 32; ++i) {
        uint32_t ws_i = __shfl_sync(0xffffffffu, ws[u], i), we_i = __shfl_sync(0xffffffffu, we[u], i);
        uint32_t sb_i = __shfl_sync(0xffffffffu, sb, i);
        if (i >= cnt) continue;
        uint32_t b_i = sb_i >> 1;
        bool some_i = (sb_i & 1) != 0;
        bool merged = false;
        if (have && some_i && b_i == cur.bin &&
            ((cur.start <= ws_i && ws_i < cur.end) || (cur.start < we_i && we_i <= cur.end))) {
          cur.start = ws_i < cur.start ? ws_i : cur.start;
          cur.end = we_i > cur.end ? we_i : cur.end;
          cur.num_seeds += 1;
          merged = true;
        }
        if (!merged) {
          if (have && cur.num_seeds >= min_seeds) {
            if (lane == 0) {
              cand[nc] = cur;
            }
            ++nc;
          }
          have = some_i;
          if (some_i) cur = CandRec{ws_i, we_i, b_i, 1};
        }
      }
    }
  }
  if (have && cur.num_seeds >= min_seeds) {
    if (lane == 0) {
      cand[nc] = cur;
    }
    ++nc;
  }
  return nc;
}

__global__ void __launch_bounds__(128) coalesce_kernel(BinsView bv, ReadsView rv, Params p, uint32_t nq,
                                                       const uint32_t* __restrict__ hit_off,
                                                       const uint32_t* __restrict__ q_nhits,
                                                       const uint32_t* __restrict__ q_nseeds,
                                                       uint64_t* __restrict__ hit_keys,
                                                       CandRec* __restrict__ cand_sparse,
                                                       uint32_t* __restrict__ q_ncand,
                                                       uint32_t* __restrict__ heavy_list,
                                                       uint32_t* __restrict__ monster_list,
                                                       BatchCounters* __restrict__ ctr) {
  // one lane per read: its strands are taken one after the other (usually exactly one of them has
  // hits, so lanes carry similar loads); a strand with many hits is handed to the whole warp
  const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
  const unsigned lane = threadIdx.x & 31;
  // first pass: every lane takes the strand of its read that has more hits (nearly always the only one with
  // any), so that the lanes of a warp are busy together; second pass: the other strand
  uint32_t first = 0;
  if (p.ns == 2 && r * 2 + 1 < nq && q_nhits[r * 2 + 1] > q_nhits[r * 2]) first = 1;
  for (uint32_t pass = 0; pass < p.ns; ++pass) {
    const uint32_t s = p.ns == 2 ? (pass ^ first) : 0;
    const uint32_t q = r * p.ns + s;
    uint32_t nh = q < nq ? q_nhits[q] : 0;
    if (pass == 1 && !__any_sync(0xffffffffu, nh != 0)) {  // nothing left for this warp
      if (q < nq) q_ncand[q] = 0;
      continue;
    }
    uint32_t nc = 0, L = 0, k = 0, ms = 0, base = 0;
    if (nh) {
      L = query_len(rv, p.ns, q);
      k = edit_budget(L, p.edit_rate);
      ms = min_seeds_of(q_nseeds[q], p.min_seed);
      base = hit_off[q];
      if (nh <= kLightItems) {
        // few hits: this lane orders them itself with a register sorting network
        uint64_t* kq = hit_keys + base;
        if (nh > 1) {
          uint64_t v[kLightItems];
#pragma unroll
          for (uint32_t i = 0; i < kLightItems; ++i) v[i] = i < nh ? kq[i] : ~0ull;
          static_assert(kLightItems == 16, "sort_network16 sorts exactly 16 keys");
          sort_network16(v);
#pragma unroll
          for (uint32_t i = 0; i < kLightItems; ++i)
            if (i < nh) kq[i] = v[i];
        }
        nc = coalesce_item(bv, kq, nh, ms, L, k, cand_sparse + base);
      }
    }
    // strands with many hits go to a work list: coalesce_heavy_kernel gives each of them a warp of its
    // own, so one warp never has to work through several heavy strands one after the other
    unsigned heavy = __ballot_sync(0xffffffffu, nh > kLightItems && nh <= kMonsterHits);
    if (heavy) {
      uint32_t slot = 0;
      if (lane == (unsigned)(__ffs(heavy) - 1)) slot = atomicAdd(&ctr->n_heavy, (unsigned)__popc(heavy));
      slot = __shfl_sync(0xffffffffu, slot, __ffs(heavy) - 1);
      if (nh > kLightItems && nh <= kMonsterHits) heavy_list[slot + __popc(heavy & ((1u << lane) - 1))] = q;
    }
    if (nh > kMonsterHits) monster_list[atomicAdd(&ctr->n_monster, 1u)] = q;  // a handful per batch
    if (q < nq && nh <= kLightItems) q_ncand[q] = nc;
  }
}

__global__ void __launch_bounds__(128) coalesce_heavy_kernel(BinsView bv, ReadsView rv, Params p,
                                                             const uint32_t* __restrict__ hit_off,
                                                             const uint32_t* __restrict__ q_nhits,
                                                             const uint32_t* __restrict__ q_nseeds,
                                                             const uint64_t* __restrict__ hit_keys,
                                                             CandRec* __restrict__ cand_sparse,
                                                             uint32_t* __restrict__ q_ncand,
                                                             const uint32_t* __restrict__ heavy_list,
                                                             BatchCounters* __restrict__ ctr) {
  const unsigned lane = threadIdx.x & 31;
  const uint32_t n_list = ctr->n_heavy;
  // strands differ by orders of magnitude (17 .. tens of thousands of hits): warps take the next strand
  // from a shared cursor instead of a fixed stride
  for (;;) {
    uint32_t it = 0;
    if (lane == 0) it = atomicAdd(&ctr->heavy_cursor, 1u);
    it = __shfl_sync(0xffffffffu, it, 0);
    if (it >= n_list) break;
    const uint32_t q = heavy_list[it];
    const uint32_t L = query_len(rv, p.ns, q);
    const uint32_t k = edit_budget(L, p.edit_rate);
    const uint32_t ms = min_seeds_of(q_nseeds[q], p.min_seed);
    const uint32_t base = hit_off[q];
    uint32_t nc = coalesce_warp(bv, hit_keys + base, q_nhits[q], ms, L, k, cand_sparse + base);
    if (lane == 0) q_ncand[q] = nc;
  }
}

// A strand with thousands of hits (several seeds at max-hits) would keep one warp busy long after the
// rest of the grid has drained.  It gets a CTA of 32 warps instead: the hit list is cut into 32 chunks
// at positions where a hit provably starts a new candidate (site gap >= 2(L+k), see coalesce_warp), so the
// chunks are independent sub-problems; every warp runs the ordinary warp automaton on its chunk into a
// staging buffer, and the chunks' candidates are then packed together in order.
__global__ void __launch_bounds__(1024) coalesce_monster_kernel(BinsView bv, ReadsView rv, Params p,
                                                                const uint32_t* __restrict__ hit_off,
                                                                const uint32_t* __restrict__ q_nhits,
                                                                const uint32_t* __restrict__ q_nseeds,
                                                                const uint64_t* __restrict__ hit_keys,
                                                                CandRec* __restrict__ cand_sparse,
                                                                CandRec* __restrict__ cand_stage,
                                                                uint32_t* __restrict__ q_ncand,
                                                                const uint32_t* __restrict__ monster_list,
                                                                const BatchCounters* __restrict__ ctr) {
  __shared__ uint32_t s_start[33], s_cnt[32], s_pre[33];
  const unsigned lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const uint32_t n_list = ctr->n_monster;
  for (uint32_t it = blockIdx.x; it < n_list; it += gridDim.x) {
    const uint32_t q = monster_list[it];
    const uint32_t n = q_nhits[q], base = hit_off[q];
    const uint32_t L = query_len(rv, p.ns, q);
    const uint32_t k = edit_budget(L, p.edit_rate);
    const uint32_t ms = min_seeds_of(q_nseeds[q], p.min_seed);
    const uint64_t* keys = hit_keys + base;
    // chunk start of warp w: the first guaranteed-break position at or after w * n / 32
    uint32_t start = (uint32_t)(((uint64_t)n * w) / 32);
    if (w > 0) {
      const uint64_t gap = 2ull * ((uint64_t)L + k);
      for (;;) {
        uint32_t h = start + lane;
        bool brk = false;
        if (h < n && h > 0) brk = (keys[h] >> 16) >= (keys[h - 1] >> 16) + gap;
        unsigned m = __ballot_sync(0xffffffffu, brk);
        if (m) {
          start += __ffs(m) - 1;
          break;
        }
        start += 32;
        if (start >= n) {
          start = n;
          break;
        }
      }
    }
    if (lane == 0) s_start[w] = start;
    if (threadIdx.x == 0) s_start[32] = n;
    __syncthreads();
    const uint32_t my_start = s_start[w], my_end = s_start[w + 1];
    uint32_t cnt = 0;
    if (my_end > my_start)
      cnt = coalesce_warp(bv, keys + my_start, my_end - my_start, ms, L, k, cand_stage + base + my_start);
    if (lane == 0) s_cnt[w] = cnt;
    __syncthreads();
    if (threadIdx.x == 0) {
      uint32_t run = 0;
      for (int i = 0; i < 32; ++i) {
        s_pre[i] = run;
        run += s_cnt[i];
      }
      s_pre[32] = run;
      q_ncand[q] = run;
    }
    __syncthreads();
    for (uint32_t i = lane; i < cnt; i += 32) cand_sparse[base + s_pre[w] + i] = cand_stage[base + my_start + i];
    __syncthreads();
  }
}

// Candidate ranking (src/index.rs:369: stable sort by num_seeds descending) + compaction into the dense
// candidate list.  No sort is needed: a lane with a handful of candidates selects them in order; for a
// strand with many candidates the warp emits, for each distinct num_seeds value from the largest down,
// the candidates holding it in discovery order (ballot compaction) — the values are few (a chance hit
// has num_seeds 1) even when the candidates are thousands.
__global__ void __launch_bounds__(256) rank_emit_kernel(uint32_t nq, const uint32_t* __restrict__ hit_off,
                                                        const uint32_t* __restrict__ q_ncand,
                                                        const uint32_t* __restrict__ cand_off,
                                                        const CandRec* __restrict__ cand_sparse,
                                                        CandRec* __restrict__ cand_dense,
                                                        uint32_t* __restrict__ cand_q) {
  uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
  const unsigned lane = threadIdx.x & 31;
  uint32_t nc = q < nq ? q_ncand[q] : 0;
  uint32_t src = 0, dst = 0;
  if (nc) {
    src = hit_off[q];
    dst = cand_off[q];
    if (nc <= kLightItems) {
      uint64_t prev = 0;
      for (uint32_t i = 0; i < nc; ++i) {
        uint64_t best = ~0ull;
        for (uint32_t j = 0; j < nc; ++j) {
          uint64_t kj = make_rank_key(cand_sparse[src + j].num_seeds, j);
          if ((i == 0 || kj > prev) && kj < best) best = kj;
        }
        prev = best;
        cand_dense[dst + i] = cand_sparse[src + (uint32_t)(best & 0xffffffffu)];
        cand_q[dst + i] = q;
      }
    }
  }
  unsigned heavy = __ballot_sync(0xffffffffu, nc > kLightItems);
  while (heavy) {
    int sl = __ffs(heavy) - 1;
    heavy &= heavy - 1;
    const uint32_t nc_s = __shfl_sync(0xffffffffu, nc, sl), src_s = __shfl_sync(0xffffffffu, src, sl);
    const uint32_t dst_s = __shfl_sync(0xffffffffu, dst, sl), q_s = __shfl_sync(0xffffffffu, q, sl);
    uint32_t out = 0;
    uint32_t bound = 0xffffffffu;  // emit values strictly below `bound`, largest first
    while (out < nc_s) {
      // next value = the largest num_seeds below bound
      uint32_t v = 0;
      for (uint32_t i = lane; i < nc_s; i += 32) {
        uint32_t ns = cand_sparse[src_s + i].num_seeds;
        if (ns < bound && ns > v) v = ns;
      }
      v = __reduce_max_sync(0xffffffffu, v);
      for (uint32_t t0 = 0; t0 < nc_s; t0 += 32) {
        uint32_t i = t0 + lane;
        CandRec c{0, 0, 0, 0};
        bool take = false;
        if (i < nc_s) {
          c = cand_sparse[src_s + i];
          take = c.num_seeds == v;
        }
        unsigned m = __ballot_sync(0xffffffffu, take);
        if (take) {
          uint32_t pos = dst_s + out + __popc(m & ((1u << lane) - 1));
          cand_dense[pos] = c;
          cand_q[pos] = q_s;
        }
        out += __popc(m);
      }
      bound = v;
      if (v == 0) break;  // cannot happen (num_seeds >= 1); guards against an endless loop
    }
  }
}

// ------------------------------------------------------------------------------------------
// verification: one thread per (pattern, text window) job, Myers/Hyyrö bit-vector recurrence with
// the pattern-match masks of the thread staged in shared memory ([class][word][thread], conflict
// free).  W = 64-bit words per pattern (compile time), NCLS = match classes (4: A,C,G,T for the
// binner where any N is a mismatch, src/index.rs:272-279; 5: N equals N, the raw
// Aligner::min_edit_distance semantics used by the stage-level entry point).
// ------------------------------------------------------------------------------------------
constexpr int kVerifyThreads = 128;

struct VerifyJob {
  const ReadWord* enc;  // pattern as bit planes (one strand)
  uint32_t L;           // pattern length
  const uint8_t* txt;   // text window
  uint32_t T;           // window length
  uint32_t limit;       // edit budget k; result > limit is reported as kNoEdit
  uint32_t skip;        // 1 = do not verify (result kNoEdit)
  uint32_t out;         // where the result goes
};

// binner jobs: dense candidate list, visited through `order` so that a warp gets candidates of similar
// cost (single-seed candidates — mostly chance hits that the Ukkonen cut-off rejects within one block —
// are grouped after the multi-seed ones)
struct BinnerJobs {
  ReadsView rv;
  EncView ev;
  Params p;
  const CandRec* cand;
  const uint32_t* cand_q;
  const uint32_t* cand_off;
  const uint32_t* order;
  const uint8_t* text;
  uint32_t n;
  __device__ __forceinline__ uint32_t count() const { return n; }
  __device__ __forceinline__ VerifyJob get(uint32_t i) const {
    VerifyJob j;
    uint32_t ci = order[i];
    CandRec c = cand[ci];
    uint32_t q = cand_q[ci];
    j.enc = ev.words + query_word_off(rv, ev, p.ns, q);
    j.L = query_len(rv, p.ns, q);
    j.txt = text + c.start;
    j.T = c.end - c.start;
    j.limit = edit_budget(j.L, p.edit_rate);
    j.out = ci;
    uint32_t rank = ci - cand_off[q];
    // src/index.rs:385-389 (prefix of the ranked list) and :406 (L - 2k wraps when 2k > L)
    j.skip = (p.max_candidates >= 0 && (uint64_t)rank >= (uint64_t)p.max_candidates) ||
             (2ull * j.limit > (uint64_t)j.L) || j.L == 0;
    return j;
  }
};

// stage-level jobs: explicit pairs; patterns were encoded (raw mode) like a one-strand read batch
struct PairJobs {
  ReadsView pv;  // the patterns as "reads"
  EncView ev;
  const uint8_t* texts;
  const uint64_t* text_off;
  uint32_t n;
  __device__ __forceinline__ uint32_t count() const { return n; }
  __device__ __forceinline__ VerifyJob get(uint32_t i) const {
    VerifyJob j;
    j.enc = ev.words + query_word_off(pv, ev, 1, i);
    j.L = query_len(pv, 1, i);
    j.txt = texts + text_off[i];
    j.T = (uint32_t)(text_off[i + 1] - text_off[i]);
    j.limit = 0xfffffffeu;
    j.skip = 0;
    j.out = i;
    return j;
  }
};

template <int W, int NCLS, bool SMEM_PEQ, typename Jobs>
__global__ void __launch_bounds__(kVerifyThreads) verify_kernel(Jobs jobs, uint32_t* __restrict__ out,
                                                                uint32_t* __restrict__ end_out,
                                                                BatchCounters* __restrict__ ctr) {
  extern __shared__ uint64_t peq[];  // [NCLS][W][kVerifyThreads] when SMEM_PEQ
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= jobs.count()) return;
  VerifyJob job = jobs.get(i);
  if (job.skip) {
    out[job.out] = kNoEdit;
    return;
  }
  const uint32_t L = job.L;
  if (L == 0) {  // empty needle aligns anywhere with 0 edits (src/align.rs test_empty)
    out[job.out] = 0;
    return;
  }
  const int last = (int)((L - 1) >> 6);
  // pattern-match masks straight from the read's bit planes; for reads beyond 1024 bases (W > 16) they do
  // not fit shared memory and are recomputed from the planes (L1-resident) at every use
  if (SMEM_PEQ) {
#pragma unroll
    for (int w = 0; w < W; ++w) {
      ReadWord rw{0, 0, ~0ull};
      if (w <= last) rw = job.enc[w];
#pragma unroll
      for (int c = 0; c < NCLS; ++c) peq[(c * W + w) * kVerifyThreads + threadIdx.x] = word_peq(rw, c);
    }
  }
  // text is read through 8-byte aligned words (the device text has 16 bytes of slack at the end)
  struct TextReader {
    const uint64_t* wp;
    uint32_t sh;
    mutable uint64_t word;
    __device__ __forceinline__ uint32_t operator()(uint32_t j) const {
      uint32_t bi = (j + sh) & 7;
      if (j == 0 || bi == 0) word = __ldg(wp + ((j + sh) >> 3));
      uint32_t c = text_code((uint8_t)(word >> (bi * 8)));
      return c < (uint32_t)NCLS ? c : 7u;
    }
  };
  const uint64_t addr = (uint64_t)job.txt;
  TextReader text{reinterpret_cast<const uint64_t*>(addr & ~7ull), (uint32_t)(addr & 7ull), 0};
  const uint32_t T = job.T;
  const ReadWord* enc = job.enc;
  auto peq_f = [&](uint32_t c, int w) -> uint64_t {
    if (SMEM_PEQ) return peq[(c * W + w) * kVerifyThreads + threadIdx.x];
    ReadWord rw = enc[w];
    uint64_t base = ~rw.nn;
    uint64_t lo = (c & 1) ? rw.lo : ~rw.lo, hi = (c & 2) ? rw.hi : ~rw.hi;
    return c < 4 ? (base & lo & hi) : (rw.nn & ~rw.lo & ~rw.hi);
  };
  uint32_t end_col = 0;
  const uint32_t best = myers_bounded<W>(L, T, job.limit, peq_f, text, end_out ? &end_col : nullptr);
  out[job.out] = best <= job.limit ? best : kNoEdit;
  if (end_out) end_out[job.out] = end_col;  // text columns consumed by the best alignment (for the SW check)
}

template <int NCLS, typename Jobs>
static int launch_verify(const Jobs& jobs, uint32_t max_len, uint32_t* out, uint32_t* end_out, BatchCounters* ctr,
                         cudaStream_t st) {
  if (jobs.n == 0) return 0;
  uint32_t words = (max_len + 63) / 64;
  unsigned grid = (jobs.n + kVerifyThreads - 1) / kVerifyThreads;
#define MTSV_VERIFY_CASE(WW)                                                                      \
  {                                                                                               \
    constexpr bool kSmem = (WW) <= 16;                                                            \
    size_t smem = kSmem ? (size_t)NCLS * WW * kVerifyThreads * sizeof(uint64_t) : 0;              \
    auto kfn = verify_kernel<WW, NCLS, kSmem, Jobs>;                                              \
    if (smem > 48 * 1024)                                                                         \
      MTSV_CUDA_TRY(cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
    MTSV_LAUNCH(kfn, grid, kVerifyThreads, smem, st, jobs, out, end_out, ctr);                    \
  }
  if (words <= 1) MTSV_VERIFY_CASE(1)
  else if (words <= 2) MTSV_VERIFY_CASE(2)
  else if (words <= 3) MTSV_VERIFY_CASE(3)
  else if (words <= 4) MTSV_VERIFY_CASE(4)
  else if (words <= 8) MTSV_VERIFY_CASE(8)
  else if (words <= 16) MTSV_VERIFY_CASE(16)
  else if (words <= 32) MTSV_VERIFY_CASE(32)
  else if (words <= 64) MTSV_VERIFY_CASE(64)
  else return set_error(MTSVGPU_ELIMIT, "pattern of %u bases exceeds the verifier limit of 4096", max_len);
#undef MTSV_VERIFY_CASE
  MTSV_CUDA_TRY(cudaGetLastError());
  return 0;
}

// ------------------------------------------------------------------------------------------
// The binner's fast path: reads of at most 256 bases (W <= 4 words).  Same jobs, same results as
// verify_kernel, but the block range of the recurrence is kept per warp (core.cuh::myers_warp), the
// text comes as 4-bit match classes, 16 columns per load, and with all reads of one length (UNIFORM)
// block scores follow the carries.  Shared memory: [5 classes][W][thread] masks, class 4 = zero.
// ------------------------------------------------------------------------------------------
struct WarpVote {
  __device__ __forceinline__ bool any(bool x) const { return __any_sync(0xffffffffu, x); }
  __device__ __forceinline__ bool all(bool x) const { return __all_sync(0xffffffffu, x); }
  __device__ __forceinline__ uint32_t umax(uint32_t x) const { return __reduce_max_sync(0xffffffffu, x); }
};

template <int W, bool UNIFORM>
__global__ void __launch_bounds__(kVerifyThreads) verify_warp_kernel(BinnerJobs jobs, const uint64_t* __restrict__ text4,
                                                                     uint64_t text4_last_word,
                                                                     uint32_t* __restrict__ out) {
  extern __shared__ uint64_t peq[];  // [5][W][kVerifyThreads]
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  VerifyJob job;
  job.skip = 1;
  job.L = 0;
  job.T = 0;
  job.limit = 0;
  job.out = 0;
  job.enc = nullptr;
  uint32_t start = 0;
  const uint32_t n_jobs = jobs.count();
  if (i < n_jobs) {
    job = jobs.get(i);
    start = (uint32_t)(job.txt - jobs.text);
  }
  bool live = i < n_jobs && !job.skip && job.L != 0;
  if (i < n_jobs && !live) out[job.out] = job.skip ? kNoEdit : 0u;  // L == 0: src/align.rs test_empty
  const uint32_t L = job.L;
  const int nb = live ? (int)((L - 1) >> 6) : -1;
#pragma unroll
  for (int w = 0; w < W; ++w) {
    ReadWord rw{0, 0, ~0ull};
    if (w <= nb) rw = job.enc[w];
#pragma unroll
    for (int c = 0; c < 4; ++c) peq[(c * W + w) * kVerifyThreads + threadIdx.x] = word_peq(rw, c);
    peq[(4 * W + w) * kVerifyThreads + threadIdx.x] = 0;
  }
  // (each thread reads back only what it wrote: no barrier needed)
  const uint64_t* my_peq = peq + threadIdx.x;
  auto peq_f = [&](uint32_t c, int w) -> uint64_t { return my_peq[(c * W + w) * kVerifyThreads]; };
  // 16 columns of text per call, realigned to the window start; one word of look-ahead is carried over
  struct Text16 {
    const uint64_t* t4;
    uint64_t wi, last_word;
    uint32_t sh;
    mutable uint64_t cur;
    __device__ __forceinline__ uint64_t operator()(uint32_t j0) const {
      uint64_t idx = wi + (j0 >> 4) + 1;
      uint64_t nxt = __ldg(t4 + (idx < last_word ? idx : last_word));
      uint64_t v = sh ? (cur >> sh) | (nxt << (64 - sh)) : cur;
      cur = nxt;
      return v;
    }
  };
  Text16 text16{text4, start >> 4, text4_last_word, (start & 15u) * 4u, 0};
  text16.cur = __ldg(text4 + text16.wi);
  const uint32_t best = myers_warp<W, UNIFORM>(L, job.T, job.limit, live, peq_f, text16, WarpVote());
  if (live) out[job.out] = best <= job.limit ? best : kNoEdit;
}

// ------------------------------------------------------------------------------------------
// Reads of 254 bases and more: the SW pre-filter of src/index.rs:402-406 is no longer implied by the edit
// distance (core.cuh, "The SW pre-filter ... for reads of 254 bases and more").  Candidates that passed the
// edit-distance test are re-checked against an exact emulation of ssw_align's 16-bit kernel:
//   ssw_band_kernel  thread per passing candidate: lower bound from the cells within edit+1 of the diagonal
//                    on which the edit alignment ends; settles nearly every candidate;
//   ssw_full_kernel  the few that stay below the threshold (or whose band would not fit its 256-row ring): both full
//                    matrices (textbook SW decides whether the 8-bit kernel overflowed), thread per candidate,
//                    scratch rows in global memory.
// A rejected candidate gets kNoEdit, exactly as if it had failed :406.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) ssw_band_kernel(BinnerJobs jobs, const uint32_t* __restrict__ cand_end,
                                                       const uint32_t* __restrict__ cand_edit,
                                                       uint32_t* __restrict__ list, unsigned int* __restrict__ n_list) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= jobs.count()) return;
  VerifyJob job = jobs.get(i);
  if (job.skip || job.L < 254) return;
  const uint32_t edit = cand_edit[job.out];
  if (edit == kNoEdit) return;
  const uint32_t L = job.L, thr = L - 2 * job.limit;  // 2k <= L here (job.skip otherwise)
  if (thr == 0) return;
  const uint32_t w = edit + 1;
  bool ok = false;
  if (w <= kSswBandMaxW) {
    uint16_t H[kSswBandCap], E[kSswBandCap];
    const ReadWord* enc = job.enc;
    const uint8_t* txt = job.txt;
    auto rcode = [&](uint32_t q) { return plane_code(enc, q); };
    auto tcode = [&](uint32_t c) { return dna5_code(__ldg(txt + c)); };
    ok = ssw_word_band(L, job.T, rcode, tcode, (int64_t)cand_end[job.out] - (int64_t)L, w, thr, H, E) >= thr;
  }
  if (!ok) list[atomicAdd(n_list, 1u)] = i;
}

__global__ void __launch_bounds__(128) ssw_full_kernel(BinnerJobs jobs, const uint32_t* __restrict__ list,
                                                       const unsigned int* __restrict__ n_list,
                                                       uint32_t* __restrict__ cand_edit, uint16_t* __restrict__ scratch,
                                                       uint32_t max_len) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x, nt = gridDim.x * blockDim.x;
  uint16_t* H = scratch + (size_t)t * 4 * max_len;
  const uint32_t n = *n_list;
  for (uint32_t x = t; x < n; x += nt) {
    VerifyJob job = jobs.get(list[x]);
    const uint32_t L = job.L;
    const ReadWord* enc = job.enc;
    const uint8_t* txt = job.txt;
    auto rcode = [&](uint32_t q) { return plane_code(enc, q); };
    auto tcode = [&](uint32_t c) { return dna5_code(__ldg(txt + c)); };
    if (!ssw_accepts_full(L, job.T, rcode, tcode, L - 2 * job.limit, H, H + max_len, H + 2 * (size_t)max_len,
                          H + 3 * (size_t)max_len))
      cand_edit[job.out] = kNoEdit;
  }
}

// ------------------------------------------------------------------------------------------
// select / emit
// ------------------------------------------------------------------------------------------
// The verification loop control of src/index.rs:375-431 with the warp, for queries with many
// candidates: 32 candidates per step, the (rare) passing ones are taken in rank order; the
// "TaxID already matched" test scans the accepted list with all lanes.
constexpr uint32_t kSelectTaxCache = 1024;  // accepted TaxIDs of a heavy strand kept in shared memory

// Strands with up to kSelectTaxCache / 2 candidates: the accepted TaxIDs live in a warp-private hash set in shared
// memory (open addressing, TaxID + 1 as the key), and the passing candidates of a 32-candidate step are taken
// together: a lane drops out when its TaxID is in the set or when a lower lane of the step carries the same TaxID
// (rank order: the lower lane is the earlier candidate), the others are accepted at once.
__device__ uint32_t select_warp_hashed(const BinsView& bv, const Params& p, const CandRec* __restrict__ cand,
                                       const uint32_t* __restrict__ edits, uint32_t n_cand, uint32_t k,
                                       HitRec* __restrict__ out, uint32_t* __restrict__ s_set) {
  const unsigned lane = threadIdx.x & 31;
  uint32_t n_out = 0;
  if (p.max_candidates >= 0 && (uint64_t)n_cand > (uint64_t)p.max_candidates) n_cand = (uint32_t)p.max_candidates;
  for (uint32_t j = lane; j < kSelectTaxCache; j += 32) s_set[j] = 0;
  __syncwarp();
  for (uint32_t t0 = 0; t0 < n_cand; t0 += 32) {
    const uint32_t c = t0 + lane;
    const uint32_t e = c < n_cand ? edits[c] : kNoEdit;
    bool pass = e != kNoEdit && e <= k;
    CandRec cr{0, 0, 0, 0};
    uint32_t tax = 0;
    if (pass) {
      cr = cand[c];
      tax = ldg(&bv.tax[cr.bin]);
      // already accepted?  (the set only changes between steps)
      const uint32_t key = tax + 1u;  // 0 marks an empty slot; TaxID 0xffffffff wraps to 0 and is handled below
      if (key != 0) {
        uint32_t h = (tax * 2654435761u) >> 22;  // 10 bits
        for (;;) {
          const uint32_t v = s_set[h];
          if (v == key) {
            pass = false;
            break;
          }
          if (v == 0) break;
          h = (h + 1) & (kSelectTaxCache - 1);
        }
      }
    }
    const unsigned pm = __ballot_sync(0xffffffffu, pass);
    if (pm == 0) continue;
    // one candidate per TaxID within the step: the lowest lane
    const unsigned peers = __match_any_sync(0xffffffffu, pass ? tax : (0x80000000u | lane) ^ 0x5a5a5a5au) & pm;
    bool win = pass && (unsigned)(__ffs(peers) - 1) == lane;
    if (tax == 0xffffffffu && pass) {  // the one key the set cannot hold: fall back to scanning the output
      bool seen = false;
      for (uint32_t j = 0; j < n_out; ++j) seen |= out[j].tax_id == tax;
      win = win && !seen;
    }
    unsigned wm = __ballot_sync(0xffffffffu, win);
    if (p.max_assignments >= 0) {  // :421-425: stop once max_assignments hits are in (tested after a push: >= 1)
      const uint64_t lim = p.max_assignments > 0 ? (uint64_t)p.max_assignments : 1;
      const uint64_t room = lim > n_out ? lim - n_out : 0;
      while ((uint64_t)__popc(wm) > room) wm &= ~(0x80000000u >> __clz(wm));  // drop the highest lanes
      win = (wm >> lane) & 1u;
    }
    if (win) {
      HitRec hrec;
      hrec.tax_id = tax;
      hrec.gi = ldg(&bv.gi[cr.bin]);
      const uint32_t bs = ldg(&bv.start[cr.bin]);
      hrec.offset = cr.start >= bs ? cr.start - bs : 0;
      hrec.edit = e;
      hrec.reserved = 0;
      out[n_out + __popc(wm & ((1u << lane) - 1u))] = hrec;
      const uint32_t key = tax + 1u;
      if (key != 0) {
        uint32_t h = (tax * 2654435761u) >> 22;
        while (atomicCAS(&s_set[h], 0u, key) != 0u) h = (h + 1) & (kSelectTaxCache - 1);
      }
    }
    __syncwarp();
    n_out += (uint32_t)__popc(wm);
    if (p.max_assignments >= 0 && (uint64_t)n_out >= (uint64_t)p.max_assignments) return n_out;
  }
  return n_out;
}

__device__ uint32_t select_warp(const BinsView& bv, const Params& p, const CandRec* __restrict__ cand,
                                const uint32_t* __restrict__ edits, uint32_t n_cand, uint32_t k,
                                HitRec* __restrict__ out, uint32_t* __restrict__ s_tax) {
  if (n_cand <= kSelectTaxCache / 2) return select_warp_hashed(bv, p, cand, edits, n_cand, k, out, s_tax);
  const unsigned lane = threadIdx.x & 31;
  uint32_t n_out = 0;
  if (p.max_candidates >= 0 && (uint64_t)n_cand > (uint64_t)p.max_candidates) n_cand = (uint32_t)p.max_candidates;
  for (uint32_t t0 = 0; t0 < n_cand; t0 += 32) {
    uint32_t c = t0 + lane;
    uint32_t e = c < n_cand ? edits[c] : kNoEdit;
    bool pass = e != kNoEdit && e <= k;
    CandRec cr{0, 0, 0, 0};
    uint32_t tax = 0;
    if (pass) {
      cr = cand[c];
      tax = ldg(&bv.tax[cr.bin]);
    }
    unsigned m = __ballot_sync(0xffffffffu, pass);
    while (m) {
      int i = __ffs(m) - 1;
      m &= m - 1;
      uint32_t tax_i = __shfl_sync(0xffffffffu, tax, i);
      // "TaxID already matched" (src/index.rs:393-396): the first kSelectTaxCache accepted TaxIDs are
      // scanned in shared memory, any beyond that in the output records
      bool seen = false;
      const uint32_t n_cached = n_out < kSelectTaxCache ? n_out : kSelectTaxCache;
      for (uint32_t j = lane; j < n_cached; j += 32) seen |= s_tax[j] == tax_i;
      for (uint32_t j = kSelectTaxCache + lane; j < n_out; j += 32) seen |= out[j].tax_id == tax_i;
      if (__any_sync(0xffffffffu, seen)) continue;
      if ((int)lane == i) {
        HitRec h;
        h.tax_id = tax;
        h.gi = ldg(&bv.gi[cr.bin]);
        uint32_t bs = ldg(&bv.start[cr.bin]);
        h.offset = cr.start >= bs ? cr.start - bs : 0;
        h.edit = e;
        h.reserved = 0;
        out[n_out] = h;
        if (n_out < kSelectTaxCache) s_tax[n_out] = tax;
      }
      __syncwarp();
      ++n_out;
      if (p.max_assignments >= 0 && (uint64_t)n_out >= (uint64_t)p.max_assignments) return n_out;
    }
  }
  return n_out;
}

__global__ void __launch_bounds__(128) select_kernel(BinsView bv, ReadsView rv, Params p, uint32_t nq,
                                                     const uint32_t* __restrict__ cand_off,
                                                     const CandRec* __restrict__ cand_dense,
                                                     const uint32_t* __restrict__ cand_edit,
                                                     HitRec* __restrict__ hit_tmp,
                                                     uint32_t* __restrict__ q_nout) {
  __shared__ uint32_t s_tax[4][kSelectTaxCache];
  uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
  const unsigned lane = threadIdx.x & 31;
  uint32_t b = 0, nc = 0, k = 0, n = 0;
  if (q < nq) {
    b = cand_off[q];
    nc = cand_off[q + 1] - b;
  }
  if (nc) {
    uint32_t L = query_len(rv, p.ns, q);
    k = edit_budget(L, p.edit_rate);
    if (nc <= kLightItems) n = select_item(bv, p, cand_dense + b, cand_edit + b, nc, k, hit_tmp + b);
  }
  unsigned heavy = __ballot_sync(0xffffffffu, nc > kLightItems);
  while (heavy) {
    int sl = __ffs(heavy) - 1;
    heavy &= heavy - 1;
    uint32_t nc_s = __shfl_sync(0xffffffffu, nc, sl), b_s = __shfl_sync(0xffffffffu, b, sl);
    uint32_t k_s = __shfl_sync(0xffffffffu, k, sl);
    uint32_t r = select_warp(bv, p, cand_dense + b_s, cand_edit + b_s, nc_s, k_s, hit_tmp + b_s,
                             s_tax[threadIdx.x >> 5]);
    if ((int)lane == sl) n = r;
  }
  if (q < nq) q_nout[q] = n;
}

__global__ void __launch_bounds__(256) gather_hits_kernel(uint32_t nq, uint32_t ns,
                                                          const uint32_t* __restrict__ cand_off,
                                                          const uint32_t* __restrict__ out_off,
                                                          const HitRec* __restrict__ hit_tmp,
                                                          HitRec* __restrict__ out_hits, uint64_t out_base,
                                                          uint64_t* __restrict__ out_hit_off, uint64_t read_base) {
  uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
  const unsigned lane = threadIdx.x & 31;
  if (q <= nq && q % ns == 0) out_hit_off[read_base + q / ns] = out_base + out_off[q];  // q == nq: the end
  uint32_t n = 0, src = 0;
  uint64_t dst = 0;
  if (q < nq) {
    n = out_off[q + 1] - out_off[q];
    src = cand_off[q];
    dst = out_base + out_off[q];
    if (n <= kLightItems)
      for (uint32_t i = 0; i < n; ++i) out_hits[dst + i] = hit_tmp[src + i];
  }
  unsigned heavy = __ballot_sync(0xffffffffu, n > kLightItems);
  while (heavy) {
    int sl = __ffs(heavy) - 1;
    heavy &= heavy - 1;
    uint32_t n_s = __shfl_sync(0xffffffffu, n, sl), src_s = __shfl_sync(0xffffffffu, src, sl);
    uint64_t dst_s = __shfl_sync(0xffffffffu, dst, sl);
    for (uint32_t i = lane; i < n_s; i += 32) out_hits[dst_s + i] = hit_tmp[src_s + i];
  }
}

// verification order: multi-seed candidates first, single-seed ones after (stable within each class)
__global__ void cand_class_kernel(const CandRec* __restrict__ cand, uint32_t n, uint32_t* __restrict__ flag,
                                  BatchCounters* __restrict__ ctr, int write_flags) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t wbytes = 0;
  if (i < n) {
    CandRec c = cand[i];
    if (write_flags) flag[i] = c.num_seeds > 1 ? 1u : 0u;
    wbytes = c.end - c.start;
  }
  if (ctr) cta_accumulate(ctr->window_bytes, wbytes);  // profiling: reference bytes the verifier reads
}

__global__ void cand_order_kernel(const CandRec* __restrict__ cand, const uint32_t* __restrict__ multi_before,
                                  uint32_t n, uint32_t* __restrict__ order) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint32_t mb = multi_before[i], n_multi = multi_before[n];
  uint32_t pos = cand[i].num_seeds > 1 ? mb : n_multi + (i - mb);
  order[pos] = i;
}

// ------------------------------------------------------------------------------------------
// Verification in two rounds (strands with several candidates per TaxID).  The reference walks a strand's ranked
// candidates and skips every candidate whose TaxID has already matched (src/index.rs:393-396): the later windows
// of a TaxID are only ever aligned when the earlier ones fail.  Here: the first candidate of every
// (strand, TaxID) group — its leader — is verified in round one; the other members only in round two, and only
// when their leader did not pass.  A member that is never verified keeps "no edit distance", which is what the
// selection does with it anyway (its TaxID has matched).  lead[c] = index of c's leader (c itself for leaders).
// ------------------------------------------------------------------------------------------
constexpr uint32_t kLeaderSlots = 1024;  // per-warp hash map TaxID -> leader, for strands of up to 512 candidates

__global__ void __launch_bounds__(128) cand_leader_kernel(BinsView bv, uint32_t nq, const uint32_t* __restrict__ cand_off,
                                                          const CandRec* __restrict__ cand, uint32_t* __restrict__ lead) {
  __shared__ uint32_t s_key[4][kLeaderSlots];
  __shared__ uint32_t s_val[4][kLeaderSlots];
  const uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
  const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint32_t b = 0, nc = 0;
  if (q < nq) {
    b = cand_off[q];
    nc = cand_off[q + 1] - b;
  }
  if (nc && nc <= kLightItems) {
    for (uint32_t i = 0; i < nc; ++i) {
      const uint32_t tax = ldg(&bv.tax[cand[b + i].bin]);
      uint32_t l = b + i;
      for (uint32_t j = 0; j < i; ++j)
        if (ldg(&bv.tax[cand[b + j].bin]) == tax) {
          l = b + j;
          break;
        }
      lead[b + i] = l;
    }
  }
  unsigned heavy = __ballot_sync(0xffffffffu, nc > kLightItems);
  while (heavy) {
    const int sl = __ffs(heavy) - 1;
    heavy &= heavy - 1;
    const uint32_t nc_s = __shfl_sync(0xffffffffu, nc, sl), b_s = __shfl_sync(0xffffffffu, b, sl);
    if (nc_s > kLeaderSlots / 2) {  // too many for the map: every candidate is its own leader (all are verified)
      for (uint32_t i = lane; i < nc_s; i += 32) lead[b_s + i] = b_s + i;
      continue;
    }
    uint32_t* key = s_key[warp];
    uint32_t* val = s_val[warp];
    for (uint32_t j = lane; j < kLeaderSlots; j += 32) key[j] = 0;
    __syncwarp();
    for (uint32_t t0 = 0; t0 < nc_s; t0 += 32) {
      const uint32_t c = t0 + lane;
      const bool in = c < nc_s;
      uint32_t tax = 0, l = b_s + c;
      bool fresh = in;
      if (in) {
        tax = ldg(&bv.tax[cand[b_s + c].bin]);
        const uint32_t k2 = tax + 1u;
        if (k2 != 0) {
          uint32_t h = (tax * 2654435761u) >> 22;
          for (;;) {
            const uint32_t v = key[h];
            if (v == k2) {
              l = val[h];
              fresh = false;
              break;
            }
            if (v == 0) break;
            h = (h + 1) & (kLeaderSlots - 1);
          }
        }
      }
      const unsigned fm = __ballot_sync(0xffffffffu, fresh);
      const unsigned peers = __match_any_sync(0xffffffffu, fresh ? tax : ~lane) & fm;
      if (fresh) {
        const unsigned first = (unsigned)(__ffs(peers) - 1);
        if (first != lane) {
          l = b_s + t0 + first;  // an earlier candidate of this step carries the TaxID
        } else if (tax + 1u != 0) {
          uint32_t h = (tax * 2654435761u) >> 22;
          while (atomicCAS(&key[h], 0u, tax + 1u) != 0u) h = (h + 1) & (kLeaderSlots - 1);
          val[h] = l;
        }
      }
      if (in) lead[b_s + c] = l;
      __syncwarp();
    }
  }
}

// round 1: positions of `order` whose candidate is a leader; round 2: members whose leader did not pass
__global__ void cand_round_flags_kernel(const uint32_t* __restrict__ order, const uint32_t* __restrict__ lead,
                                        const uint32_t* __restrict__ edit, uint32_t n, int round,
                                        uint32_t* __restrict__ flag) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint32_t c = order[i], l = lead[c];
  flag[i] = round == 1 ? (l == c ? 1u : 0u) : ((l != c && edit[l] == kNoEdit) ? 1u : 0u);
}

__global__ void cand_compact_order_kernel(const uint32_t* __restrict__ order, const uint32_t* __restrict__ idx, uint32_t n,
                                          const CandRec* __restrict__ cand, uint32_t* __restrict__ out,
                                          BatchCounters* __restrict__ ctr) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t wbytes = 0;
  if (i < n && idx[i + 1] != idx[i]) {
    const uint32_t c = order[i];
    out[idx[i]] = c;
    wbytes = cand[c].end - cand[c].start;
  }
  if (ctr) cta_accumulate(ctr->window_bytes, wbytes);  // profiling: reference columns of the candidates verified
}

// ------------------------------------------------------------------------------------------
// host orchestration
// ------------------------------------------------------------------------------------------
static int validate_params(const mtsvgpu_params* in, Params* p) {
  if (!in) return set_error(MTSVGPU_EINVAL, "params is NULL");
  if (!(in->edit_rate >= 0.0 && in->edit_rate <= 1.0))  // src/bin/mtsv-binner.rs:151
    return set_error(MTSVGPU_EINVAL, "edit_rate must be in [0,1]");
  if (!(in->min_seed > 0.0 && in->min_seed <= 1.0))  // src/bin/mtsv-binner.rs:195
    return set_error(MTSVGPU_EINVAL, "min_seed must be in (0,1]");
  if (in->seed_size == 0 || in->seed_size > 4096)
    return set_error(MTSVGPU_EINVAL, "seed_size must be in [1,4096]");
  if (in->seed_gap == 0)  // itertools .step(0) panics in the reference (src/index.rs:285)
    return set_error(MTSVGPU_EINVAL, "seed_gap must be > 0");
  p->edit_rate = in->edit_rate;
  p->min_seed = in->min_seed;
  p->S = in->seed_size;
  p->G = in->seed_gap;
  p->max_hits = in->max_hits;
  p->tune_max_hits = in->tune_max_hits;
  p->max_candidates = in->max_candidates < 0 ? -1 : in->max_candidates;
  p->max_assignments = in->max_assignments < 0 ? -1 : in->max_assignments;
  p->ns = in->strands == 1 ? 1 : 2;
  return 0;
}

int run_segmented_sort(cudaStream_t st, DevBuf& worklist, uint64_t* keys, const uint32_t* seg_off,
                              const uint32_t* seg_cnt, uint32_t nq, uint32_t min_count, BatchCounters* d_ctr) {
  if (worklist.cap < (size_t)3 * nq * 4) {
    MTSV_CUDA_TRY(cudaStreamSynchronize(st));
    MTSV_TRY(worklist.reserve((size_t)3 * nq * 4));
  }
  uint32_t* lists = worklist.as<uint32_t>();
  MTSV_CUDA_TRY(cudaMemsetAsync(&d_ctr->n_warp, 0, 3 * sizeof(unsigned int), st));
  MTSV_LAUNCH(sort_classify_kernel, (nq + 255) / 256, 256, 0, st, seg_cnt, nq, min_count, lists, lists + nq,
              lists + 2 * (size_t)nq, d_ctr);
  MTSV_LAUNCH(sort_warp_kernel, sm_count() * 8, 256, 0, st, keys, seg_off, seg_cnt, lists, d_ctr);
  MTSV_LAUNCH(sort_medium_kernel, sm_count() * 4, 512, 0, st, keys, seg_off, seg_cnt, lists + nq, d_ctr);
  MTSV_LAUNCH(sort_large_kernel, sm_count(), 1024, 0, st, keys, seg_off, seg_cnt, lists + 2 * (size_t)nq, d_ctr);
  MTSV_CUDA_TRY(cudaGetLastError());
  return 0;
}

// grow-with-preserve for the whole-batch output
static int grow_preserve(DevBuf& buf, size_t used_bytes, size_t need_bytes, cudaStream_t st) {
  if (need_bytes <= buf.cap && buf.p) return 0;
  size_t want = std::max(need_bytes + need_bytes / 2, (size_t)1 << 20);
  void* np = nullptr;
  cudaError_t e = cudaMalloc(&np, want);
  if (e != cudaSuccess) {
    (void)cudaGetLastError();
    return set_error(MTSVGPU_ENOMEM, "cudaMalloc(%zu) failed: %s", want, cudaGetErrorString(e));
  }
  if (buf.p && used_bytes) {
    MTSV_CUDA_TRY(cudaMemcpyAsync(np, buf.p, used_bytes, cudaMemcpyDeviceToDevice, st));
    MTSV_CUDA_TRY(cudaStreamSynchronize(st));
  }
  if (buf.p) cudaFree(buf.p);
  buf.p = np;
  buf.cap = want;
  return 0;
}

// The host reads the sub-batch scalars between stages.  They are pushed into page-locked mapped host memory
// by a tiny kernel instead of a cudaMemcpy: a D2H copy would queue on the copy engine behind the result
// slices of the previous sub-batch that the host API streams out concurrently.
__global__ void publish_counters_kernel(const BatchCounters* __restrict__ d, BatchCounters* __restrict__ h) {
  const uint32_t* src = reinterpret_cast<const uint32_t*>(d);
  volatile uint32_t* dst = reinterpret_cast<volatile uint32_t*>(h);
  for (uint32_t i = threadIdx.x; i < sizeof(BatchCounters) / 4; i += blockDim.x) dst[i] = src[i];
  __threadfence_system();
}

static int fetch_counters(Lane& ln, const BatchCounters* d_ctr, BatchCounters* out, cudaStream_t st) {
  if (!ln.h_ctr) {
    MTSV_CUDA_TRY(cudaHostAlloc((void**)&ln.h_ctr, sizeof(BatchCounters), cudaHostAllocMapped));
    MTSV_CUDA_TRY(cudaHostGetDevicePointer((void**)&ln.h_ctr_dev, ln.h_ctr, 0));
  }
  MTSV_LAUNCH(publish_counters_kernel, 1, 160, 0, st, d_ctr, ln.h_ctr_dev);
  MTSV_CUDA_TRY(cudaStreamSynchronize(st));
  memcpy(out, ln.h_ctr, sizeof(BatchCounters));
  return 0;
}

// ---- ordered output: slices append to the batch result in slice order ----
static int emit_acquire(mtsvgpu_index* h, Lane& ln) {
  if (ln.has_turn) return 0;
  std::unique_lock<std::mutex> lk(h->emit_mu);
  h->emit_cv.wait(lk, [&] { return h->abort_rc != 0 || h->emit_turn == ln.slice; });
  if (h->abort_rc != 0) return set_error(h->abort_rc, "%s", h->abort_msg.c_str());
  ln.has_turn = true;
  return 0;
}
static void emit_release(mtsvgpu_index* h, Lane& ln) {  // the slice is complete
  std::lock_guard<std::mutex> lk(h->emit_mu);
  if (ln.has_turn) h->emit_turn = ln.slice + 1;
  ln.has_turn = false;
  h->emit_cv.notify_all();
}
const char* last_error_cstr();
static void emit_abort(mtsvgpu_index* h, int rc) {
  std::lock_guard<std::mutex> lk(h->emit_mu);
  if (h->abort_rc == 0) {
    h->abort_rc = rc;
    h->abort_msg = last_error_cstr();
  }
  h->emit_cv.notify_all();
}

// What stays fixed over one bin_batch_device call
struct BatchCall {
  mtsvgpu_index* h;
  Params p;
  const uint8_t* d_seqs;
  const uint64_t* d_seq_off;
  BatchSource* src;  // null: device-resident input
  const char* group_verify;  // MTSV_B200_GROUP_VERIFY: unset = where it pays, "0" = never, anything else = always
};

// One device sub-batch, reads [rv.read0, rv.read0 + rv.n_reads), as it passes through the stages below.  A stage
// reserves the workspace buffers it is the first to use; 1 from a stage: too large, the caller splits the range.
struct SubBatch : BatchCall {
  Lane& ln;
  BatchWorkspace& ws;  // scratch of the lane
  cudaStream_t st;
  ReadsView rv;
  EncView ev{};
  uint32_t nq;  // strands
  size_t qn;    // nq + 1
  BatchCounters* d_ctr = nullptr;
  BatchCounters hc;      // the device counters as last fetched
  bool uniform = false;  // every read has the same length (never when a read was left out)
  uint32_t uni_spq = 0;  // seed slots per strand when they are addressed arithmetically, else 0
  uint32_t n_slots = 0, n_hits = 0, n_cand = 0;
  uint64_t n_verified = 0;

  SubBatch(const BatchCall& c, Lane& l, uint64_t read0, uint32_t n_reads)
      : BatchCall(c), ln(l), ws(*l.ws), st(l.stream),
        rv{c.d_seqs, c.d_seq_off, read0, n_reads}, nq(n_reads * c.p.ns), qn((size_t)nq + 1) {}
  unsigned qgrid() const { return (nq + 255) / 256; }
  int fetch() { return fetch_counters(ln, d_ctr, &hc, st); }
  // per-stage timing (profiling only)
  cudaEvent_t next_event() {
    if (ln.ev_next == ln.ev_pool.size()) {
      cudaEvent_t e;
      cudaEventCreate(&e);
      ln.ev_pool.push_back(e);
    }
    return ln.ev_pool[ln.ev_next++];
  }
  void begin(int stage) {
    if (!h->profiling) return;
    cudaEvent_t a = next_event(), b = next_event();
    cudaEventRecord(a, ln.stream);
    ln.ev_used.push_back({stage, {a, b}});
  }
  void end() {
    if (!h->profiling) return;
    cudaEventRecord(ln.ev_used.back().second.second, ln.stream);
  }
  void resolve() {
    if (!h->profiling) return;
    cudaStreamSynchronize(ln.stream);
    for (auto& e : ln.ev_used) {
      float ms = 0;
      cudaEventElapsedTime(&ms, e.second.first, e.second.second);
      ln.stats.ms[e.first] += ms;
    }
    ln.ev_used.clear();
    ln.ev_next = 0;
  }

  int slots_encode(uint64_t slot_bound, uint64_t sub_bytes, uint64_t pack_base);
  int search();
  int candidates();
  int verify();
  int launch_verify_warp(const BinnerJobs& jobs);
  template <int W>
  int launch_verify_warp(const BinnerJobs& jobs);
  int verify_ssw(const BinnerJobs& jobs);
  int verify_grouped(const BinnerJobs& jobs, bool* done);
  int select_append(uint64_t* out_total);
};

// ---- seed slots, then the reads' bit planes ----
int SubBatch::slots_encode(uint64_t slot_bound, uint64_t sub_bytes, uint64_t pack_base) {
  const uint32_t n_reads = rv.n_reads;
  MTSV_TRY(ws.counters.reserve(sizeof(BatchCounters)));
  d_ctr = ws.counters.as<BatchCounters>();
  MTSV_CUDA_TRY(cudaMemsetAsync(d_ctr, 0, sizeof(BatchCounters), st));
  MTSV_TRY(ws.slot_off.reserve(qn * 4));
  for (DevBuf* b : {&ws.slot_q, &ws.slot_lo, &ws.slot_cnt, &ws.slot_hoff}) MTSV_TRY(b->reserve((slot_bound + 1) * 4));
  MTSV_TRY(ws.scan_tmp.reserve(((qn + 2047) / 2048 + 1) * 8));
  const uint64_t total_words64 = (sub_bytes >> 6) + n_reads;  // words of one strand (closed-form layout)
  if (total_words64 * p.ns > 0x7fffffffull) return 1;
  const uint32_t total_words = (uint32_t)total_words64;
  MTSV_TRY(ws.enc.reserve(((size_t)total_words * p.ns + 1) * sizeof(ReadWord)));
  ev = EncView{ws.enc.as<ReadWord>(), total_words};

  begin(ST_PREP);
  uint32_t* slot_off = ws.slot_off.as<uint32_t>();
  MTSV_LAUNCH(count_slots_kernel, qgrid(), 256, 0, st, rv, p, nq, slot_off, d_ctr);
  MTSV_TRY(exclusive_scan_u32(slot_off, slot_off, nq, ws.scan_tmp, (uint64_t*)&d_ctr->total_slots, st));
  end();
  MTSV_TRY(fetch());
  if (hc.bad_offsets) return set_error(MTSVGPU_EINVAL, "seq_off is not monotone");
  ln.stats.n_reads_over_limit += hc.n_over_len;
  if (hc.total_slots > slot_bound)
    return set_error(MTSVGPU_ECUDA, "internal: seed slots %llu exceed bound %llu (reads [%llu,+%u), %llu bytes)",
                     hc.total_slots, (unsigned long long)slot_bound, (unsigned long long)rv.read0, n_reads,
                     (unsigned long long)sub_bytes);
  n_slots = (uint32_t)hc.total_slots;
  // min_len == max_len: every read of the sub-batch has the same length (never when a read was left out)
  const uint32_t min_len = hc.n_over_len ? 0u : ~hc.inv_min_len;
  uniform = min_len == hc.max_len;
  ln.stats.n_seed_slots += n_slots;
  // (only now that the slot count is known to fit the buffers)
  begin(ST_PREP);
  // all reads of one length: slots are addressed arithmetically, no slot -> query map needed
  uni_spq = (uniform && nq && n_slots % nq == 0) ? n_slots / nq : 0;
  if (!uni_spq) MTSV_LAUNCH(expand_slots_kernel, qgrid(), 256, 0, st, slot_off, nq, ws.slot_q.as<uint32_t>());
  if (!src || src->pack_base.empty()) {
    MTSV_LAUNCH(encode_reads_kernel, (n_reads + 127) / 128, 128, 0, st, rv, ws.enc.as<ReadWord>());
  } else {
    // d_seqs holds packed records: the sub-batch's first one at pack_base
    const uint32_t* rel = nullptr;
    if (!uniform) {
      MTSV_TRY(ws.pack_rel.reserve(((size_t)n_reads + 1) * 4));
      MTSV_LAUNCH(packed_sizes_kernel, (n_reads + 127) / 128, 128, 0, st, rv, ws.pack_rel.as<uint32_t>());
      MTSV_TRY(exclusive_scan_u32(ws.pack_rel.as<uint32_t>(), ws.pack_rel.as<uint32_t>(), n_reads, ws.scan_tmp, nullptr, st));
      rel = ws.pack_rel.as<uint32_t>();
    }
    MTSV_LAUNCH(unpack_reads_kernel, (n_reads + 127) / 128, 128, 0, st, rv, rv.seqs + pack_base,
                packed_record_bytes(hc.max_len), rel, ws.enc.as<ReadWord>());
  }
  if (p.ns == 2) {
    const uint32_t w_max = hc.max_len ? (hc.max_len + 63) / 64 : 1;
    const uint64_t threads = (uint64_t)n_reads * w_max;
    MTSV_LAUNCH(encode_rc_kernel, (unsigned)((threads + 255) / 256), 256, 0, st, rv, ws.enc.as<ReadWord>(),
                total_words, w_max);
  }
  end();
  return 0;
}

// ---- seed search, then the seed rule replayed and the hit offsets ----
int SubBatch::search() {
  for (DevBuf* b : {&ws.q_nseeds, &ws.q_nhits, &ws.hit_off}) MTSV_TRY(b->reserve(qn * 4));
  const uint32_t* slot_off = ws.slot_off.as<uint32_t>();
  begin(ST_SEARCH);
  if (n_slots)
    MTSV_LAUNCH(seed_search_kernel, (n_slots + 255) / 256, 256, 0, st, h->ix.fm_view(), h->ix.ktab_view(), rv, ev, p,
                slot_off, ws.slot_q.as<uint32_t>(), n_slots, ws.slot_lo.as<uint32_t>(),
                ws.slot_cnt.as<uint32_t>(), d_ctr, h->profiling ? 1 : 0, hc.max_len, uni_spq);
  end();
  begin(ST_SELECT);
  MTSV_LAUNCH(seed_select_kernel, qgrid(), 256, 0, st, rv, ev, p, slot_off, nq, ws.slot_cnt.as<uint32_t>(),
              ws.slot_hoff.as<uint32_t>(), ws.q_nseeds.as<uint32_t>(), ws.q_nhits.as<uint32_t>(), d_ctr);
  MTSV_TRY(exclusive_scan_u32(ws.q_nhits.as<uint32_t>(), ws.hit_off.as<uint32_t>(), nq, ws.scan_tmp,
                              (uint64_t*)&d_ctr->total_hits, st));
  end();
  MTSV_TRY(fetch());
  ln.stats.n_strands_over_hits += hc.overflow;
  const uint64_t hit_cap = h->opts.max_batch_hits ? h->opts.max_batch_hits : (1ull << 27);
  if (hc.total_hits > hit_cap || hc.total_hits > 0xfffffff0ull) {
    if (rv.n_reads == 1)
      return set_error(MTSVGPU_ELIMIT, "one read produced %llu seed hits (cap %llu)", hc.total_hits,
                       (unsigned long long)hit_cap);
    return 1;
  }
  n_hits = (uint32_t)hc.total_hits;
  ln.stats.n_seed_hits += n_hits;
  for (int i = 0; i < 32; ++i) ln.stats.rank_queries += hc.rank_steps[i];  // sectors touched by seed search
  return 0;
}

// ---- locate, sort per strand, coalesce into candidates, rank ----
int SubBatch::candidates() {
  const DeviceIndex& ix = h->ix;
  for (DevBuf* b : {&ws.q_ncand, &ws.cand_off}) MTSV_TRY(b->reserve(qn * 4));
  if (!n_hits) return 0;
  MTSV_TRY(ws.worklist.reserve(3 * qn * 4));
  MTSV_TRY(ws.hit_keys.reserve((size_t)n_hits * 8));
  MTSV_TRY(ws.cand_sparse.reserve((size_t)n_hits * sizeof(CandRec)));
  begin(ST_LOCATE);
  MTSV_LAUNCH(locate_kernel, qgrid(), 256, 0, st, ix.fm_view(), ix.sa_view(), p, ws.slot_off.as<uint32_t>(), nq,
              ws.slot_lo.as<uint32_t>(), ws.slot_cnt.as<uint32_t>(), ws.slot_hoff.as<uint32_t>(),
              ws.hit_off.as<uint32_t>(), ws.q_nhits.as<uint32_t>(), ws.hit_keys.as<uint64_t>());
  end();
  begin(ST_SORT);
  MTSV_TRY(run_segmented_sort(st, ws.worklist, ws.hit_keys.as<uint64_t>(), ws.hit_off.as<uint32_t>(),
                              ws.q_nhits.as<uint32_t>(), nq, kLightItems, d_ctr));
  end();
  begin(ST_COALESCE);
  MTSV_TRY(ws.cand_stage.reserve((size_t)n_hits * sizeof(CandRec)));
  MTSV_CUDA_TRY(cudaMemsetAsync(&d_ctr->n_heavy, 0, 3 * sizeof(unsigned int), st));
  MTSV_LAUNCH(coalesce_kernel, (rv.n_reads + 127) / 128, 128, 0, st, ix.bins_view(), rv, p, nq,
              ws.hit_off.as<uint32_t>(), ws.q_nhits.as<uint32_t>(), ws.q_nseeds.as<uint32_t>(),
              ws.hit_keys.as<uint64_t>(), ws.cand_sparse.as<CandRec>(), ws.q_ncand.as<uint32_t>(),
              ws.worklist.as<uint32_t>(), ws.worklist.as<uint32_t>() + nq, d_ctr);
  MTSV_LAUNCH(coalesce_heavy_kernel, sm_count() * 16, 128, 0, st, ix.bins_view(), rv, p, ws.hit_off.as<uint32_t>(),
              ws.q_nhits.as<uint32_t>(), ws.q_nseeds.as<uint32_t>(), ws.hit_keys.as<uint64_t>(),
              ws.cand_sparse.as<CandRec>(), ws.q_ncand.as<uint32_t>(), ws.worklist.as<uint32_t>(), d_ctr);
  MTSV_LAUNCH(coalesce_monster_kernel, sm_count(), 1024, 0, st, ix.bins_view(), rv, p, ws.hit_off.as<uint32_t>(),
              ws.q_nhits.as<uint32_t>(), ws.q_nseeds.as<uint32_t>(), ws.hit_keys.as<uint64_t>(),
              ws.cand_sparse.as<CandRec>(), ws.cand_stage.as<CandRec>(), ws.q_ncand.as<uint32_t>(),
              ws.worklist.as<uint32_t>() + nq, d_ctr);
  MTSV_TRY(exclusive_scan_u32(ws.q_ncand.as<uint32_t>(), ws.cand_off.as<uint32_t>(), nq, ws.scan_tmp,
                              (uint64_t*)&d_ctr->total_cands, st));
  end();
  MTSV_TRY(fetch());
  n_cand = (uint32_t)hc.total_cands;
  if (!n_cand) return 0;
  MTSV_TRY(ws.cand_dense.reserve((size_t)n_cand * sizeof(CandRec)));
  MTSV_TRY(ws.cand_q.reserve((size_t)n_cand * 4));
  begin(ST_RANK);
  MTSV_LAUNCH(rank_emit_kernel, qgrid(), 256, 0, st, nq, ws.hit_off.as<uint32_t>(), ws.q_ncand.as<uint32_t>(),
              ws.cand_off.as<uint32_t>(), ws.cand_sparse.as<CandRec>(), ws.cand_dense.as<CandRec>(),
              ws.cand_q.as<uint32_t>());
  end();
  return 0;
}

// ---- verify (sub-batches with candidates): the route is chosen up front ----
int SubBatch::verify() {
  const bool ssw = hc.max_len >= 254;  // reads the SW pre-filter is not implied for
  // several candidates per strand on average: verify TaxID group leaders first (see cand_leader_kernel).  Worth
  // trying only where some TaxID has several sequences (otherwise two candidates of one TaxID would have to be two
  // windows of the same sequence) and the sub-batch has more candidates than strands.
  bool grouped = !ssw && (group_verify ? group_verify[0] != '0' : n_cand > nq && h->ix.n_bins > h->ix.n_taxids);
  MTSV_TRY(ws.cand_edit.reserve((size_t)n_cand * 4));
  begin(ST_VERIFY);
  MTSV_TRY(ws.cand_flag.reserve(((size_t)n_cand + 1) * 4));
  MTSV_TRY(ws.cand_order.reserve((size_t)n_cand * 4));
  MTSV_LAUNCH(cand_class_kernel, (n_cand + 255) / 256, 256, 0, st, ws.cand_dense.as<CandRec>(), n_cand,
              ws.cand_flag.as<uint32_t>(), (h->profiling && !grouped) ? d_ctr : nullptr, 1);
  MTSV_TRY(exclusive_scan_u32(ws.cand_flag.as<uint32_t>(), ws.cand_flag.as<uint32_t>(), n_cand, ws.scan_tmp,
                              nullptr, st));
  MTSV_LAUNCH(cand_order_kernel, (n_cand + 255) / 256, 256, 0, st, ws.cand_dense.as<CandRec>(),
              ws.cand_flag.as<uint32_t>(), n_cand, ws.cand_order.as<uint32_t>());
  BinnerJobs jobs{rv, ev, p, ws.cand_dense.as<CandRec>(), ws.cand_q.as<uint32_t>(),
                  ws.cand_off.as<uint32_t>(), ws.cand_order.as<uint32_t>(), h->ix.text, n_cand};
  n_verified = n_cand;
  if (ssw) {
    MTSV_TRY(verify_ssw(jobs));
  } else {
    if (grouped) MTSV_TRY(verify_grouped(jobs, &grouped));
    if (!grouped) MTSV_TRY(launch_verify_warp(jobs));
  }
  end();
  return 0;
}

// the warp verifier (reads of at most 253 bases) over a job list
int SubBatch::launch_verify_warp(const BinnerJobs& jobs) {
  if (jobs.n == 0) return 0;
  const uint32_t words = (std::max(hc.max_len, 1u) + 63) / 64;
  if (words <= 1) return launch_verify_warp<1>(jobs);
  if (words == 2) return launch_verify_warp<2>(jobs);
  if (words == 3) return launch_verify_warp<3>(jobs);
  return launch_verify_warp<4>(jobs);
}
template <int W>
int SubBatch::launch_verify_warp(const BinnerJobs& jobs) {
  const unsigned grid = (jobs.n + kVerifyThreads - 1) / kVerifyThreads;
  const size_t smem = (size_t)5 * W * kVerifyThreads * sizeof(uint64_t);
  auto kernel = uniform ? verify_warp_kernel<W, true> : verify_warp_kernel<W, false>;
  MTSV_LAUNCH(kernel, grid, kVerifyThreads, smem, st, jobs, h->ix.text4, h->ix.text4_words - 1, ws.cand_edit.as<uint32_t>());
  MTSV_CUDA_TRY(cudaGetLastError());
  return 0;
}

// reads of 254 bases or more: the per-lane verifier, then the SW filter (band first, full matrices where it fails)
int SubBatch::verify_ssw(const BinnerJobs& jobs) {
  const uint32_t max_len = hc.max_len;
  for (DevBuf* b : {&ws.cand_end, &ws.ssw_list}) MTSV_TRY(b->reserve((size_t)n_cand * 4));
  uint32_t* cand_end = ws.cand_end.as<uint32_t>();
  MTSV_TRY(launch_verify<4>(jobs, max_len, ws.cand_edit.as<uint32_t>(), cand_end, h->profiling ? d_ctr : nullptr, st));
  // scratch of the full-matrix pass: 4 rows of max_len u16 per thread, about 64 MB in all
  const uint32_t full_threads =
      (uint32_t)std::min<size_t>(8192, std::max<size_t>(256, ((size_t)64 << 20) / ((size_t)max_len * 8))) / 128 * 128;
  MTSV_TRY(ws.ssw_scratch.reserve((size_t)full_threads * 4 * max_len * sizeof(uint16_t)));
  MTSV_CUDA_TRY(cudaMemsetAsync(&d_ctr->n_ssw_full, 0, sizeof(unsigned int), st));
  MTSV_LAUNCH(ssw_band_kernel, (n_cand + 127) / 128, 128, 0, st, jobs, cand_end, ws.cand_edit.as<uint32_t>(),
              ws.ssw_list.as<uint32_t>(), &d_ctr->n_ssw_full);
  MTSV_LAUNCH(ssw_full_kernel, full_threads / 128, 128, 0, st, jobs, ws.ssw_list.as<uint32_t>(), &d_ctr->n_ssw_full,
              ws.cand_edit.as<uint32_t>(), ws.ssw_scratch.as<uint16_t>(), max_len);
  return 0;
}

// Two rounds: the leaders, then the members whose leader did not pass.  The list lengths come back to the host (two
// short synchronisations per sub-batch, only on this route): the launches are sized exactly — a grid sized for every
// candidate costs more in empty blocks than the round saves.  *done = false (nothing verified) when more than 90 %
// of the candidates are leaders, or when forced, all of them: the caller takes the warp route instead.
int SubBatch::verify_grouped(const BinnerJobs& jobs, bool* done) {
  const unsigned grid = (n_cand + 255) / 256;
  BatchCounters* ctr = h->profiling ? d_ctr : nullptr;
  for (DevBuf* b : {&ws.cand_lead, &ws.cand_order2}) MTSV_TRY(b->reserve((size_t)n_cand * 4));
  uint32_t* flag = ws.cand_flag.as<uint32_t>();
  MTSV_LAUNCH(cand_leader_kernel, (nq + 127) / 128, 128, 0, st, h->ix.bins_view(), nq, ws.cand_off.as<uint32_t>(),
              ws.cand_dense.as<CandRec>(), ws.cand_lead.as<uint32_t>());
  MTSV_LAUNCH(cand_round_flags_kernel, grid, 256, 0, st, ws.cand_order.as<uint32_t>(), ws.cand_lead.as<uint32_t>(),
              ws.cand_edit.as<uint32_t>(), n_cand, 1, flag);
  MTSV_TRY(exclusive_scan_u32(flag, flag, n_cand, ws.scan_tmp, (uint64_t*)&d_ctr->verified[0], st));
  MTSV_TRY(fetch());
  const uint32_t n1 = (uint32_t)hc.verified[0];
  *done = !((uint64_t)n1 * 10 > (uint64_t)n_cand * 9 && !(group_verify && n1 < n_cand));
  if (!*done) {
    if (ctr)  // (the reference bytes the warp route will read)
      MTSV_LAUNCH(cand_class_kernel, grid, 256, 0, st, ws.cand_dense.as<CandRec>(), n_cand, (uint32_t*)nullptr, ctr, 0);
    return 0;
  }
  MTSV_CUDA_TRY(cudaMemsetAsync(ws.cand_edit.p, 0xff, (size_t)n_cand * 4, st));  // kNoEdit until verified
  BinnerJobs round_jobs = jobs;
  round_jobs.order = ws.cand_order2.as<uint32_t>();
  MTSV_LAUNCH(cand_compact_order_kernel, grid, 256, 0, st, ws.cand_order.as<uint32_t>(), flag, n_cand,
              ws.cand_dense.as<CandRec>(), ws.cand_order2.as<uint32_t>(), ctr);
  round_jobs.n = n1;
  MTSV_TRY(launch_verify_warp(round_jobs));
  MTSV_LAUNCH(cand_round_flags_kernel, grid, 256, 0, st, ws.cand_order.as<uint32_t>(), ws.cand_lead.as<uint32_t>(),
              ws.cand_edit.as<uint32_t>(), n_cand, 2, flag);
  MTSV_TRY(exclusive_scan_u32(flag, flag, n_cand, ws.scan_tmp, (uint64_t*)&d_ctr->verified[1], st));
  MTSV_TRY(fetch());
  const uint32_t n2 = (uint32_t)hc.verified[1];
  if (n2) {
    MTSV_LAUNCH(cand_compact_order_kernel, grid, 256, 0, st, ws.cand_order.as<uint32_t>(), flag, n_cand,
                ws.cand_dense.as<CandRec>(), ws.cand_order2.as<uint32_t>(), ctr);
    round_jobs.n = n2;
    MTSV_TRY(launch_verify_warp(round_jobs));
  }
  n_verified = (uint64_t)n1 + n2;
  return 0;
}

// ---- select, then append to the batch output: in slice order, after the other lane's previous append ----
int SubBatch::select_append(uint64_t* out_total) {
  for (DevBuf* b : {&ws.q_nout, &ws.out_off}) MTSV_TRY(b->reserve(qn * 4));
  uint64_t sub_out = 0;
  if (n_cand) {
    MTSV_TRY(ws.hit_tmp.reserve((size_t)n_cand * sizeof(HitRec)));
    begin(ST_EMIT);
    MTSV_LAUNCH(select_kernel, (nq + 127) / 128, 128, 0, st, h->ix.bins_view(), rv, p, nq, ws.cand_off.as<uint32_t>(),
                ws.cand_dense.as<CandRec>(), ws.cand_edit.as<uint32_t>(), ws.hit_tmp.as<HitRec>(),
                ws.q_nout.as<uint32_t>());
    MTSV_TRY(exclusive_scan_u32(ws.q_nout.as<uint32_t>(), ws.out_off.as<uint32_t>(), nq, ws.scan_tmp,
                                (uint64_t*)&d_ctr->total_out, st));
    end();
    MTSV_TRY(fetch());
    sub_out = hc.total_out;
    ln.stats.n_candidates += n_verified;
    for (int i = 0; i < 32; ++i) ln.stats.window_bytes += hc.window_bytes[i];
  } else {
    MTSV_CUDA_TRY(cudaMemsetAsync(ws.out_off.p, 0, qn * 4, st));
    MTSV_CUDA_TRY(cudaMemsetAsync(ws.cand_off.p, 0, qn * 4, st));
  }
  MTSV_TRY(emit_acquire(h, ln));
  Lane& other = h->lanes[&ln == &h->lanes[0] ? 1 : 0];
  if (other.emit_event) MTSV_CUDA_TRY(cudaStreamWaitEvent(st, other.emit_event, 0));
  BatchWorkspace& res = h->ws;  // batch results (shared, appended in slice order)
  MTSV_TRY(grow_preserve(res.out_hits, *out_total * sizeof(HitRec), (*out_total + sub_out + 1) * sizeof(HitRec), st));
  begin(ST_EMIT);
  MTSV_LAUNCH(gather_hits_kernel, (nq + 1 + 255) / 256, 256, 0, st, nq, p.ns, ws.cand_off.as<uint32_t>(),
              ws.out_off.as<uint32_t>(), ws.hit_tmp.as<HitRec>(), res.out_hits.as<HitRec>(), *out_total,
              res.out_hit_off.as<uint64_t>(), rv.read0);
  end();
  MTSV_CUDA_TRY(cudaGetLastError());
  if (!ln.emit_event) MTSV_CUDA_TRY(cudaEventCreateWithFlags(&ln.emit_event, cudaEventDisableTiming));
  MTSV_CUDA_TRY(cudaEventRecord(ln.emit_event, st));
  // host API: start copying this sub-batch's results out while the next one computes
  if (src) MTSV_TRY(src->results(*out_total, sub_out, rv.read0, rv.n_reads, st));
  resolve();
  *out_total += sub_out;
  ln.stats.n_hits += sub_out;
  ln.stats.n_queries += nq;
  return 0;
}

// One device sub-batch: reads [read0, read0 + n_reads).  Returns 1 when it exceeds the in-flight limits and the
// caller must split the range (nothing was emitted in that case).
static int run_sub_batch(const BatchCall& call, Lane& ln, uint64_t read0, uint32_t n_reads, uint64_t slot_bound,
                         uint64_t sub_bytes, uint64_t pack_base, uint64_t* out_total) {
  SubBatch s(call, ln, read0, n_reads);
  int rc = s.slots_encode(slot_bound, sub_bytes, pack_base);
  if (rc == 0) rc = s.search();
  if (rc != 0) return rc;
  MTSV_TRY(s.candidates());
  if (s.n_cand) MTSV_TRY(s.verify());
  return s.select_append(out_total);
}

// One uploaded slice [read0, read0 + n_reads): processed in groups of ln.chunk_reads reads.  A group whose seed
// hits overflow the in-flight cap (run_sub_batch returns 1, nothing emitted) is retried at half the size, and
// the smaller size is kept for what follows (repetitive references: hundreds of hits per read).
static int run_range(const BatchCall& call, Lane& ln, uint64_t read0, uint64_t n_reads, uint64_t off_lo,
                     uint64_t off_hi, uint64_t* out_total) {
  if (off_hi < off_lo) return set_error(MTSVGPU_EINVAL, "seq_off is not monotone");
  const Params& p = call.p;
  const uint64_t* h_off = call.src ? call.src->seq_off : nullptr;  // host copy of seq_off
  uint64_t r = read0, off_r = off_lo;
  // packed input: byte offset of the record of read r (the slice's first record was placed by the uploader)
  const bool packed = call.src && !call.src->pack_base.empty();
  uint64_t pack_r = packed ? call.src->pack_base[ln.slice] : 0;
  const uint64_t r_end = read0 + n_reads;
  while (r < r_end) {
    uint64_t nr = std::min(r_end - r, std::max<uint64_t>(ln.chunk_reads, 1));
    uint64_t off_e = off_hi;
    if (r + nr < r_end && h_off) {
      off_e = h_off[r + nr];
    } else if (r + nr < r_end) {
      MTSV_CUDA_TRY(cudaMemcpyAsync(&off_e, call.d_seq_off + r + nr, 8, cudaMemcpyDeviceToHost, ln.stream));
      MTSV_CUDA_TRY(cudaStreamSynchronize(ln.stream));
    }
    if (off_e < off_r) return set_error(MTSVGPU_EINVAL, "seq_off is not monotone");
    // bound on seed slots from the byte count: slots(L) <= L/G + 1 per strand
    const uint64_t bytes = off_e - off_r;
    const uint64_t slot_bound = (bytes / p.G + nr) * p.ns + 1;
    const bool too_big = slot_bound > 0xfffffff0ull || nr * p.ns > 0x7ffffff0ull;
    int rc = too_big ? 1 : run_sub_batch(call, ln, r, (uint32_t)nr, slot_bound, bytes, pack_r, out_total);
    if (rc == 1) {
      if (nr == 1) return set_error(MTSVGPU_ELIMIT, "a single read exceeds the device batch limits");
      ln.chunk_reads = std::max<uint64_t>(1, nr / 2);
      continue;
    }
    if (rc != 0) return rc;
    ln.stats.n_sub_batches += 1;
    if (packed && r + nr < r_end)  // (only after a split: a slice is normally one group)
      for (uint64_t i = r; i < r + nr; ++i) pack_r += packed_record_bytes((uint32_t)(h_off[i + 1] - h_off[i]));
    r += nr;
    off_r = off_e;
  }
  return 0;
}

static void add_stats(mtsvgpu_batch_stats& to, const mtsvgpu_batch_stats& from) {
  for (int i = 0; i < MTSVGPU_N_STAGES; ++i) to.ms[i] += from.ms[i];  // (launches[] is not filled)
  to.n_queries += from.n_queries;
  to.n_seed_slots += from.n_seed_slots;
  to.n_seed_hits += from.n_seed_hits;
  to.n_candidates += from.n_candidates;
  to.n_hits += from.n_hits;
  to.window_bytes += from.window_bytes;
  to.rank_queries += from.rank_queries;
  to.n_sub_batches += from.n_sub_batches;
  to.n_reads_over_limit += from.n_reads_over_limit;
  to.n_strands_over_hits += from.n_strands_over_hits;
}

int bin_batch_device(mtsvgpu_index* h, const uint8_t* d_seqs, const uint64_t* d_seq_off, uint64_t n_reads,
                     BatchSource* src, const mtsvgpu_params* params, const mtsvgpu_hit** d_hits,
                     const uint64_t** d_hit_off, uint64_t* n_hits) {
  if (!h) return set_error(MTSVGPU_EINVAL, "index is NULL");
  BatchCall call{h, {}, d_seqs, d_seq_off, src, getenv("MTSV_B200_GROUP_VERIFY")};
  MTSV_TRY(validate_params(params, &call.p));
  if (!d_seq_off) return set_error(MTSVGPU_EINVAL, "seq_off is NULL");
  MTSV_CUDA_TRY(cudaSetDevice(h->ix.device));
  cudaStream_t st = h->stream;
  memset(&h->stats, 0, sizeof h->stats);
  BatchWorkspace& ws = h->ws;
  MTSV_TRY(ws.out_hit_off.reserve((n_reads + 1) * 8));
  uint64_t total = 0;
  if (n_reads == 0) {
    MTSV_CUDA_TRY(cudaMemsetAsync(ws.out_hit_off.p, 0, 8, st));
    MTSV_TRY(grow_preserve(ws.out_hits, 0, sizeof(HitRec), st));
  }
  // ---- lanes: the slices of a batch alternate between two lanes (own stream, scratch and host thread each): the
  // synchronisation bubbles and kernel tails of one slice are filled by the other — ~10 % on the small slices of
  // the host API, 4 % on the large ones of device-resident input.  One lane for device-resident input when per-stage
  // timing is on, so that the event timers measure kernels that run alone. ----
  const bool two_lanes = src || !h->profiling;
  const std::vector<uint64_t> rb = src ? src->bounds : slice_bounds(n_reads, h->opts.batch_reads, false, two_lanes);
  const uint64_t n_sub = rb.size() - 1;
  std::vector<uint64_t> bounds(n_sub + 1, 0);
  if (n_reads) {
    if (src) {
      for (uint64_t i = 0; i <= n_sub; ++i) bounds[i] = src->seq_off[rb[i]];
    } else {
      // (boundaries are multiples of the first slice's size: one strided gather instead of copying 8 B per read)
      MTSV_CUDA_TRY(cudaMemcpy2DAsync(bounds.data(), 8, d_seq_off, rb[1] * 8, 8, n_sub, cudaMemcpyDeviceToHost, st));
      MTSV_CUDA_TRY(cudaMemcpyAsync(&bounds[n_sub], d_seq_off + n_reads, 8, cudaMemcpyDeviceToHost, st));
      MTSV_CUDA_TRY(cudaStreamSynchronize(st));
    }
  }
  const int n_lanes = n_sub >= 2 && two_lanes ? 2 : 1;
  h->lanes[0].stream = st;
  h->lanes[0].ws = &h->ws;
  h->lanes[1].ws = &h->ws1;
  if (n_lanes == 2) {
    if (!h->lane1_stream) MTSV_CUDA_TRY(cudaStreamCreateWithFlags(&h->lane1_stream, cudaStreamNonBlocking));
    if (!h->fork_event) MTSV_CUDA_TRY(cudaEventCreateWithFlags(&h->fork_event, cudaEventDisableTiming));
    if (!h->join_event) MTSV_CUDA_TRY(cudaEventCreateWithFlags(&h->join_event, cudaEventDisableTiming));
    h->lanes[1].stream = h->lane1_stream;
    // lane 1 starts after whatever the caller queued on the handle's stream (its inputs)
    MTSV_CUDA_TRY(cudaEventRecord(h->fork_event, st));
    MTSV_CUDA_TRY(cudaStreamWaitEvent(h->lane1_stream, h->fork_event, 0));
  }
  h->emit_turn = 0;
  h->abort_rc = 0;
  h->abort_msg.clear();
  for (Lane& ln : h->lanes) {
    ln.has_turn = false;
    ln.chunk_reads = UINT64_MAX;  // a whole slice
    memset(&ln.stats, 0, sizeof ln.stats);
  }
  const int device = h->ix.device;
  auto lane_main = [&](int li) {
    Lane& ln = h->lanes[li];
    if (li != 0) cudaSetDevice(device);
    for (uint64_t i = (uint64_t)li; i < n_sub; i += (uint64_t)n_lanes) {
      {
        std::lock_guard<std::mutex> lk(h->emit_mu);
        if (h->abort_rc != 0) return;
      }
      ln.slice = i;
      int rc = 0;
      if (src) rc = src->wait_slice(i, ln.stream);
      if (rc == 0) rc = run_range(call, ln, rb[i], rb[i + 1] - rb[i], bounds[i], bounds[i + 1], &total);
      if (rc != 0) {
        emit_abort(h, rc);
        return;
      }
      emit_release(h, ln);
    }
  };
  if (n_lanes == 2) {
    std::thread helper(lane_main, 1);
    lane_main(0);
    helper.join();
    // everything lane 1 did is ordered before what follows on the handle's stream
    MTSV_CUDA_TRY(cudaEventRecord(h->join_event, h->lane1_stream));
    MTSV_CUDA_TRY(cudaStreamWaitEvent(st, h->join_event, 0));
  } else {
    lane_main(0);
  }
  for (Lane& ln : h->lanes) add_stats(h->stats, ln.stats);
  if (h->abort_rc != 0) {
    cudaStreamSynchronize(st);
    if (h->lane1_stream) cudaStreamSynchronize(h->lane1_stream);
    return set_error(h->abort_rc, "%s", h->abort_msg.c_str());
  }
  MTSV_CUDA_TRY(cudaStreamSynchronize(st));
  if (d_hits) *d_hits = reinterpret_cast<const mtsvgpu_hit*>(ws.out_hits.p);
  if (d_hit_off) *d_hit_off = ws.out_hit_off.as<uint64_t>();
  if (n_hits) *n_hits = total;
  return 0;
}

// ------------------------------------------------------------------------------------------
// stage-level entry points
// ------------------------------------------------------------------------------------------
__global__ void bs_patterns_kernel(FmView fm, KtabView kt, ReadsView pv, EncView ev, uint32_t len, uint64_t n,
                                   uint64_t* __restrict__ lower, uint64_t* __restrict__ upper) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  // a pattern is a forward-strand "read" whose single seed covers it entirely
  uint32_t lo, cnt;
  const ReadWord* qw = ev.words + query_word_off(pv, ev, 1, (uint32_t)i);
  seed_search_item(fm, kt, qw, len, len, 0, &lo, &cnt, nullptr);
  if (cnt & kDirectHit) {  // this entry point reports SA rows: search again without the table
    KtabView none{nullptr, 0, 0, nullptr};
    seed_search_item(fm, none, qw, len, len, 0, &lo, &cnt, nullptr);
  }
  lower[i] = cnt ? lo : 0;
  upper[i] = cnt ? (uint64_t)lo + cnt : 0;
}

int backward_search_batch(mtsvgpu_index* h, const uint8_t* pats, uint32_t pat_len, uint64_t n_pats,
                          uint64_t* lower, uint64_t* upper) {
  if (!h || !pats || !lower || !upper) return set_error(MTSVGPU_EINVAL, "null argument");
  if (pat_len == 0) return set_error(MTSVGPU_EINVAL, "pattern length must be > 0");
  if (n_pats == 0) return 0;
  if (n_pats > 0x0fffffffull || n_pats * pat_len > 0x7fffffffull) return set_error(MTSVGPU_ELIMIT, "too many patterns");
  MTSV_CUDA_TRY(cudaSetDevice(h->ix.device));
  cudaStream_t st = h->stream;
  DevBuf dp, doff, dw, dl, du;
  int rc = 0;
  do {
    std::vector<uint64_t> off(n_pats + 1);
    for (uint64_t i = 0; i <= n_pats; ++i) off[i] = i * pat_len;
    const uint32_t w_max = (pat_len + 63) / 64;
    const uint32_t total_words = (uint32_t)((n_pats * pat_len) >> 6) + (uint32_t)n_pats;
    if ((rc = dp.reserve(n_pats * pat_len + 16))) break;
    if ((rc = doff.reserve((n_pats + 1) * 8))) break;
    if ((rc = dw.reserve(((size_t)total_words + 1) * sizeof(ReadWord)))) break;
    if ((rc = dl.reserve(n_pats * 8))) break;
    if ((rc = du.reserve(n_pats * 8))) break;
    cudaMemcpyAsync(dp.p, pats, n_pats * pat_len, cudaMemcpyHostToDevice, st);
    cudaMemcpyAsync(doff.p, off.data(), (n_pats + 1) * 8, cudaMemcpyHostToDevice, st);
    ReadsView pv{dp.as<uint8_t>(), doff.as<uint64_t>(), 0, (uint32_t)n_pats};
    EncView ev{dw.as<ReadWord>(), total_words};
    const uint64_t threads = n_pats * w_max;
    MTSV_LAUNCH(encode_fwd_kernel, (unsigned)((threads * 32 + 255) / 256), 256, 0, st, pv, dw.as<ReadWord>(), w_max, 0);
    MTSV_LAUNCH(bs_patterns_kernel, (unsigned)((n_pats + 127) / 128), 128, 0, st, h->ix.fm_view(),
                h->ix.ktab_view(), pv, ev, pat_len, n_pats, dl.as<uint64_t>(), du.as<uint64_t>());
    cudaMemcpyAsync(lower, dl.p, n_pats * 8, cudaMemcpyDeviceToHost, st);
    cudaMemcpyAsync(upper, du.p, n_pats * 8, cudaMemcpyDeviceToHost, st);
    cudaError_t e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) rc = set_error(MTSVGPU_ECUDA, "backward_search: %s", cudaGetErrorString(e));
  } while (0);
  dp.release();
  doff.release();
  dw.release();
  dl.release();
  du.release();
  return rc;
}

__global__ void locate_rows_kernel(FmView fm, SaView sv, const uint64_t* __restrict__ rows, uint64_t n,
                                   uint64_t* __restrict__ pos) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint64_t r = rows[i];
  pos[i] = r < fm.n ? (uint64_t)fm_locate(fm, sv, (uint32_t)r, nullptr) : ~0ull;
}

int locate_batch(mtsvgpu_index* h, const uint64_t* rows, uint64_t n_rows, uint64_t* pos) {
  if (!h || !rows || !pos) return set_error(MTSVGPU_EINVAL, "null argument");
  if (n_rows == 0) return 0;
  MTSV_CUDA_TRY(cudaSetDevice(h->ix.device));
  cudaStream_t st = h->stream;
  DevBuf dr, dp;
  int rc = 0;
  do {
    if ((rc = dr.reserve(n_rows * 8))) break;
    if ((rc = dp.reserve(n_rows * 8))) break;
    cudaMemcpyAsync(dr.p, rows, n_rows * 8, cudaMemcpyHostToDevice, st);
    MTSV_LAUNCH(locate_rows_kernel, (unsigned)((n_rows + 127) / 128), 128, 0, st, h->ix.fm_view(),
                h->ix.sa_view(), dr.as<uint64_t>(), n_rows, dp.as<uint64_t>());
    cudaMemcpyAsync(pos, dp.p, n_rows * 8, cudaMemcpyDeviceToHost, st);
    cudaError_t e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) rc = set_error(MTSVGPU_ECUDA, "locate: %s", cudaGetErrorString(e));
  } while (0);
  dr.release();
  dp.release();
  return rc;
}

int edit_distance_batch(int device, const uint8_t* pats, const uint64_t* pat_off, const uint8_t* texts,
                        const uint64_t* text_off, uint64_t n_pairs, uint32_t* edits) {
  if (!pat_off || !text_off || !edits) return set_error(MTSVGPU_EINVAL, "null argument");
  if (n_pairs == 0) return 0;
  if (n_pairs > 0x7fffffffull) return set_error(MTSVGPU_ELIMIT, "too many pairs");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    (void)cudaGetLastError();
    return set_error(MTSVGPU_ENODEVICE, "no CUDA device available (this library has no CPU path)");
  }
  MTSV_CUDA_TRY(cudaSetDevice(device));
  uint32_t max_len = 0;
  for (uint64_t i = 0; i < n_pairs; ++i) {
    if (pat_off[i + 1] < pat_off[i] || text_off[i + 1] < text_off[i])
      return set_error(MTSVGPU_EINVAL, "offsets not monotone");
    max_len = std::max<uint64_t>(max_len, pat_off[i + 1] - pat_off[i]);
  }
  if (max_len > kMaxReadLenDev) return set_error(MTSVGPU_ELIMIT, "pattern longer than %u", kMaxReadLenDev);
  uint64_t pb = pat_off[n_pairs], tb = text_off[n_pairs];
  DevBuf dp, dpo, dt, dto, de, dw;
  int rc = 0;
  do {
    if ((rc = dp.reserve(pb + 16))) break;
    if ((rc = dt.reserve(tb + 16))) break;
    if ((rc = dpo.reserve((n_pairs + 1) * 8))) break;
    if ((rc = dto.reserve((n_pairs + 1) * 8))) break;
    if ((rc = de.reserve(n_pairs * 4))) break;
    if (pb) cudaMemcpy(dp.p, pats, pb, cudaMemcpyHostToDevice);
    if (tb) cudaMemcpy(dt.p, texts, tb, cudaMemcpyHostToDevice);
    cudaMemcpy(dpo.p, pat_off, (n_pairs + 1) * 8, cudaMemcpyHostToDevice);
    cudaMemcpy(dto.p, text_off, (n_pairs + 1) * 8, cudaMemcpyHostToDevice);
    // encode the patterns (raw bytes: N is its own class) like a one-strand read batch
    const uint32_t w_max = std::max(1u, (max_len + 63) / 64);
    const uint32_t total_words = (uint32_t)(pb >> 6) + (uint32_t)n_pairs;
    if ((rc = dw.reserve(((size_t)total_words + 1) * sizeof(ReadWord)))) break;
    ReadsView pv{dp.as<uint8_t>(), dpo.as<uint64_t>(), 0, (uint32_t)n_pairs};
    EncView ev{dw.as<ReadWord>(), total_words};
    const uint64_t threads = n_pairs * w_max;
    MTSV_LAUNCH(encode_fwd_kernel, (unsigned)((threads * 32 + 255) / 256), 256, 0, 0, pv, dw.as<ReadWord>(), w_max, 1);
    PairJobs jobs{pv, ev, dt.as<uint8_t>(), dto.as<uint64_t>(), (uint32_t)n_pairs};
    if ((rc = launch_verify<5>(jobs, std::max(max_len, 1u), de.as<uint32_t>(), nullptr, nullptr, 0))) break;
    cudaError_t e = cudaMemcpy(edits, de.p, n_pairs * 4, cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) rc = set_error(MTSVGPU_ECUDA, "edit_distance: %s", cudaGetErrorString(e));
  } while (0);
  dp.release();
  dpo.release();
  dt.release();
  dto.release();
  de.release();
  dw.release();
  return rc;
}

}  // namespace mtsv
