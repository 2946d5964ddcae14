// emul.cpp — TEST-ONLY host harness that runs the per-item device logic of
// mtsv_tools_b200/csrc/core.cuh serially on the CPU (compiled with g++, no CUDA), so the
// arithmetic of every stage can be diffed against the oracle without a GPU.  It is not part of
// the product: libmtsv_b200.so never contains or calls this code and has no CPU path.
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <vector>

#define MTSV_COUNT_BLOCKS 1
#include "../../mtsv_tools_b200/csrc/core.cuh"

using namespace mtsv;

namespace {

struct EmulIndex {
  std::vector<FmBlock> blocks;
  std::vector<SuperCounts> super;
  std::vector<uint32_t> n_before;
  std::vector<uint32_t> sa;
  std::vector<uint2> ktab;
  std::vector<uint8_t> text;
  std::vector<uint32_t> bin_start, bin_end, bin_tax, bin_gi;
  uint32_t C[5] = {0, 0, 0, 0, 0};
  FmView fm{};
  SaView sv{};
  KtabView kt{};
  BinsView bv{};
};

}  // namespace

extern "C" {

struct emul_bin {
  uint32_t gi, tax_id;
  uint64_t start, end;
};

struct emul_params {
  double edit_rate;
  uint32_t seed_size, seed_gap;
  double min_seed;
  uint64_t max_hits, tune_max_hits;
  int64_t max_candidates, max_assignments;
  uint32_t strands, reserved;
};

void* emul_index_build(const uint8_t* text, uint64_t n, const emul_bin* bins, uint64_t n_bins,
                       const uint8_t* bwt, const uint64_t* sample, uint64_t n_sample, uint64_t s_file,
                       uint32_t sa_rate, uint32_t ktab_k) {
  EmulIndex* e = new EmulIndex;
  e->text.assign(text, text + n);
  e->text.resize(n + 16, 0);
  for (uint64_t i = 0; i < n_bins; ++i) {
    e->bin_start.push_back((uint32_t)bins[i].start);
    e->bin_end.push_back((uint32_t)bins[i].end);
    e->bin_tax.push_back(bins[i].tax_id);
    e->bin_gi.push_back(bins[i].gi);
  }
  uint64_t n_blocks = n / 64 + 1;
  uint64_t n_super = (n_blocks + kBlocksPerSuper - 1) / kBlocksPerSuper;
  e->blocks.assign(n_super * kBlocksPerSuper, FmBlock{0, 0, 0, 0});
  e->super.resize(n_super);
  e->n_before.assign(n_super * kBlocksPerSuper, 0);
  uint32_t run[5] = {0, 0, 0, 0, 0};
  uint32_t sup[4] = {0, 0, 0, 0};
  uint32_t dollar = 0;
  for (uint64_t blk = 0; blk < n_blocks; ++blk) {
    if (blk % kBlocksPerSuper == 0) {
      for (int a = 0; a < 4; ++a) {
        sup[a] = run[a];
        e->super[blk / kBlocksPerSuper].c[a] = run[a];
      }
    }
    FmBlock b{0, 0, 0, 0};
    for (int a = 0; a < 4; ++a) b.rel |= (uint64_t)(uint16_t)(run[a] - sup[a]) << (16 * a);
    e->n_before[blk] = run[4];
    for (uint32_t j = 0; j < 64; ++j) {
      uint64_t r = blk * 64 + j;
      if (r >= n) break;
      uint32_t c = text_code(bwt[r]);
      if (c < 4) {
        b.lo |= (uint64_t)(c & 1) << j;
        b.hi |= (uint64_t)(c >> 1) << j;
        run[c]++;
      } else {
        b.exc |= 1ull << j;
        if (c == SYM_N) run[4]++;
        else dollar = (uint32_t)r;
      }
    }
    e->blocks[blk] = b;
  }
  e->fm.blocks = e->blocks.data();
  e->fm.super = e->super.data();
  e->fm.n_before = e->n_before.data();
  e->fm.n = (uint32_t)n;
  e->fm.dollar_row = dollar;
  e->C[SYM_A] = 1;
  e->C[SYM_C] = 1 + run[0];
  e->C[SYM_G] = 1 + run[0] + run[1];
  e->C[SYM_N] = 1 + run[0] + run[1] + run[2];
  e->C[SYM_T] = 1 + run[0] + run[1] + run[2] + run[4];
  e->fm.C = e->C;
  // suffix array at the requested rate: same walk as sa_densify_kernel
  if (sa_rate == 0) sa_rate = 1;
  e->sa.assign((n + sa_rate - 1) / sa_rate, 0xffffffffu);
  for (uint64_t i = 0; i < n_sample; ++i) {
    uint32_t row = (uint32_t)(i * s_file), pos = (uint32_t)sample[i];
    if (row % sa_rate == 0) e->sa[row / sa_rate] = pos;
    for (;;) {
      FmBlock b = e->blocks[row >> 6];
      uint32_t c = fm_symbol(e->fm, b, row);
      if (c == SYM_DOLLAR) break;
      row = fm_lf(e->fm, c, b, row);
      pos -= 1;
      if (row % s_file == 0) break;
      if (row % sa_rate == 0) e->sa[row / sa_rate] = pos;
    }
  }
  e->sv.sa = e->sa.data();
  e->sv.rate = sa_rate;
  // k-mer table, level by level like ktab_level_kernel (key = lo | hi << t, base j at bit j)
  if (ktab_k) {
    std::vector<uint2> cur(1), next;
    cur[0].x = 0;
    cur[0].y = (uint32_t)n;
    for (uint32_t t = 1; t <= ktab_k; ++t) {
      next.resize(1ull << (2 * t));
      for (uint64_t key = 0; key < next.size(); ++key) {
        uint64_t lo = key & ((1ull << t) - 1), hi = key >> t;
        uint32_t c = (uint32_t)(lo & 1) | ((uint32_t)(hi & 1) << 1);
        uint64_t prev = (lo >> 1) | ((hi >> 1) << (t - 1));
        uint32_t l = cur[prev].x, u = cur[prev].y;
        if (l < u) fm_step(e->fm, c, l, u);
        if (l >= u) l = u = 0;
        next[key].x = l;
        next[key].y = u;
      }
      cur.swap(next);
    }
    // unique k-mers become direct entries, as ktab_direct_kernel does
    for (uint64_t key = 0; key < cur.size(); ++key)
      if (cur[key].y - cur[key].x == 1)
        cur[key] = ktab_direct_entry(fm_locate(e->fm, e->sv, cur[key].x, nullptr), e->text.data());
    e->ktab = cur;
  }
  e->kt.tab = e->ktab.data();
  e->kt.k = ktab_k;
  e->kt.direct = ktab_k ? 1 : 0;
  e->kt.text = e->text.data();
  e->bv = BinsView{e->bin_start.data(), e->bin_end.data(), e->bin_tax.data(), e->bin_gi.data(),
                   (uint32_t)n_bins};
  return e;
}

void emul_index_free(void* p) { delete (EmulIndex*)p; }

// rank, symbol, locate, backward search as the kernels compute them
uint32_t emul_occ(void* p, uint32_t a, uint32_t i) { return fm_occ(((EmulIndex*)p)->fm, a, i); }
uint32_t emul_locate(void* p, uint32_t row) {
  EmulIndex* e = (EmulIndex*)p;
  return fm_locate(e->fm, e->sv, row, nullptr);
}
static std::vector<ReadWord> encode_query(const uint8_t* seq, uint32_t L, bool rc, bool raw) {
  uint32_t W = (L + 63) / 64;
  std::vector<ReadWord> fwd(W ? W : 1, ReadWord{0, 0, 0});
  for (uint32_t w = 0; w < W; ++w) fwd[w] = encode_fwd_word(seq, L, w, raw);
  if (!rc) return fwd;
  std::vector<ReadWord> out(W ? W : 1, ReadWord{0, 0, 0});
  for (uint32_t w = 0; w < W; ++w) out[w] = encode_rc_word(fwd.data(), L, w);
  return out;
}

void emul_backward_search(void* p, const uint8_t* pat, uint32_t len, uint32_t* lo, uint32_t* cnt) {
  EmulIndex* e = (EmulIndex*)p;
  std::vector<ReadWord> q = encode_query(pat, len, false, false);
  seed_search_item(e->fm, e->kt, q.data(), len, len, 0, lo, cnt, nullptr);
}

// Myers recurrence exactly as verify_kernel evaluates it (ncls = 4: binner rule, 5: raw bytes)
static uint32_t edit_distance_k_end(const uint8_t* pat, uint32_t L, uint32_t rc, const uint8_t* txt, uint32_t T,
                                    int ncls, uint32_t k, uint32_t* end_col);

uint32_t emul_edit_distance_k(const uint8_t* pat, uint32_t L, uint32_t rc, const uint8_t* txt, uint32_t T,
                              int ncls, uint32_t k) {
  return edit_distance_k_end(pat, L, rc, txt, T, ncls, k, nullptr);
}

// The decision of src/index.rs:406 for reads >= 254 bases, as the device takes it (binner.cu ssw_band_kernel /
// ssw_full_kernel): banded lower bound of the 16-bit kernel around the edit alignment first, full matrices if
// that is not enough.  which: 0 = as the device, 1 = full matrices only, 2 = band only (lower-bound score).
uint32_t emul_ssw_accepts(const uint8_t* read, uint32_t L, const uint8_t* txt, uint32_t T, uint32_t k,
                          uint32_t edit, uint32_t end_col, int which) {
  std::vector<ReadWord> q = encode_query(read, L, false, false);
  auto rcode = [&](uint32_t x) { return plane_code(q.data(), x); };
  auto tcode = [&](uint32_t i) { return dna5_code(txt[i]); };
  const uint32_t thr = L - 2 * k;
  const uint32_t w = edit + 1;
  if (which != 1 && w <= kSswBandMaxW) {
    uint16_t H[kSswBandCap], E[kSswBandCap];
    uint32_t b = ssw_word_band(L, T, rcode, tcode, (int64_t)end_col - (int64_t)L, w, thr, H, E);
    if (which == 2) return b;
    if (b >= thr) return 1;
  }
  if (which == 2) return 0;
  std::vector<uint16_t> buf(4 * (size_t)L);
  return ssw_accepts_full(L, T, rcode, tcode, thr, buf.data(), buf.data() + L, buf.data() + 2 * L,
                          buf.data() + 3 * L)
             ? 1
             : 0;
}

// bounded edit distance (binner match rule, forward strand) + the end column of the first best alignment
uint32_t emul_edit_distance_end(const uint8_t* pat, uint32_t L, const uint8_t* txt, uint32_t T, uint32_t k,
                                uint32_t* end_col) {
  return edit_distance_k_end(pat, L, 0, txt, T, 4, k, end_col);
}

// both scores of the full matrices: the emulated sw_sse2_word and textbook SW
void emul_ssw_scores(const uint8_t* read, uint32_t L, const uint8_t* txt, uint32_t T, uint32_t* word,
                     uint32_t* exact) {
  std::vector<ReadWord> q = encode_query(read, L, false, false);
  auto rcode = [&](uint32_t x) { return plane_code(q.data(), x); };
  auto tcode = [&](uint32_t i) { return dna5_code(txt[i]); };
  std::vector<uint16_t> buf(4 * (size_t)L);
  ssw_accepts_full(L, T, rcode, tcode, 0xffffffffu, buf.data(), buf.data() + L, buf.data() + 2 * L,
                   buf.data() + 3 * L, word, exact);
}

static uint32_t edit_distance_k_end(const uint8_t* pat, uint32_t L, uint32_t rc, const uint8_t* txt, uint32_t T,
                                    int ncls, uint32_t k, uint32_t* end_col) {
  if (end_col) *end_col = 0;
  if (L == 0) return 0;
  if (L > 4096) return 0xffffffffu;
  // pattern masks from the bit planes, as verify_kernel builds them
  std::vector<ReadWord> q = encode_query(pat, L, rc != 0, ncls == 5);
  uint64_t peq[5][64];
  memset(peq, 0, sizeof peq);
  for (uint32_t w = 0; w < (L + 63) / 64; ++w)
    for (int c = 0; c < ncls; ++c) peq[c][w] = word_peq(q[w], c);
  auto pf = [&](uint32_t c, int w) { return peq[c][w]; };
  auto tf = [&](uint32_t j) {
    uint32_t c = text_code(txt[j]);
    return c < (uint32_t)ncls ? c : 7u;
  };
  return L <= 1024 ? myers_bounded<16>(L, T, k, pf, tf, end_col) : myers_bounded<64>(L, T, k, pf, tf, end_col);
}

// The warp-uniform fast path (core.cuh::myers_warp) as one lane.  The votes of the other 31 lanes are
// played by a PRNG: with probability `noise`/256 an `any` vote succeeds although this lane did not ask
// (early activation) and an `all` vote fails although this lane agreed (late drop / late exit).
struct NoisyVote {
  mutable uint64_t s;
  uint32_t noise;
  uint32_t other_T;  // a longer window of "another lane": this lane computes columns beyond its own T
  bool flip() const {
    s = s * 6364136223846793005ull + 1442695040888963407ull;
    return ((s >> 33) & 255) < noise;
  }
  bool any(bool x) const { return x || flip(); }
  bool all(bool x) const { return x && !flip(); }
  uint32_t umax(uint32_t x) const { return x; }
};
struct NoisyVoteT : NoisyVote {  // myers_warp takes three maxima: L, the initial last block, T
  mutable int calls = 0;
  uint32_t max_last = 0;
  uint32_t umax(uint32_t x) const {
    ++calls;
    if (calls == 2 && x < max_last && flip()) return x + 1;  // another lane starts with one more block
    if (calls == 3 && other_T > x) return other_T;           // another lane has a longer window
    return x;
  }
};

uint32_t emul_edit_distance_warp(const uint8_t* pat, uint32_t L, uint32_t rc, const uint8_t* txt, uint32_t T,
                                 uint32_t k, int uniform, uint32_t noise, uint64_t seed, uint32_t other_T) {
  if (L == 0) return 0;
  if (L > 256) return 0xffffffffu;
  std::vector<ReadWord> q = encode_query(pat, L, rc != 0, false);
  uint64_t peq[5][4];
  memset(peq, 0, sizeof peq);
  const uint32_t words = (L + 63) / 64;
  for (uint32_t w = 0; w < words; ++w)
    for (int c = 0; c < 4; ++c) peq[c][w] = word_peq(q[w], c);
  auto pf = [&](uint32_t c, int w) { return peq[c][w]; };
  // 4-bit codes of the window, followed by arbitrary codes (what another lane's longer window would make
  // this lane read)
  auto t16 = [&](uint32_t j0) {
    uint64_t v = 0;
    for (uint32_t i = 0; i < 16; ++i) {
      uint32_t j = j0 + i;
      uint32_t c = j < T ? upper_acgtn_code(txt[j]) : (j * 2654435761u >> 7) % 5;
      if (c > 4) c = 4;
      v |= (uint64_t)c << (4 * i);
    }
    return v;
  };
  NoisyVoteT vote;
  vote.s = seed;
  vote.noise = noise;
  vote.other_T = other_T;
  vote.max_last = words - 1;
#define CASE(WW)                                                                                     \
  if (words == WW)                                                                                   \
    return uniform ? myers_warp<WW, true>(L, T, k, true, pf, t16, vote)                              \
                   : myers_warp<WW, false>(L, T, k, true, pf, t16, vote);
  CASE(1) CASE(2) CASE(3) CASE(4)
#undef CASE
  // non-uniform lanes may sit in a wider kernel than they need
  return 0xffffffffu;
}

// a short read in a kernel instantiated for longer ones (ragged batch): words < W
uint32_t emul_edit_distance_warp_wide(const uint8_t* pat, uint32_t L, const uint8_t* txt, uint32_t T, uint32_t k,
                                      uint32_t noise, uint64_t seed, uint32_t other_T) {
  if (L == 0 || L > 256) return 0xffffffffu;
  std::vector<ReadWord> q = encode_query(pat, L, false, false);
  uint64_t peq[5][4];
  memset(peq, 0, sizeof peq);
  for (uint32_t w = 0; w < (L + 63) / 64; ++w)
    for (int c = 0; c < 4; ++c) peq[c][w] = word_peq(q[w], c);
  auto pf = [&](uint32_t c, int w) { return peq[c][w]; };
  auto t16 = [&](uint32_t j0) {
    uint64_t v = 0;
    for (uint32_t i = 0; i < 16; ++i) {
      uint32_t j = j0 + i;
      uint32_t c = j < T ? upper_acgtn_code(txt[j]) : (j * 2654435761u >> 7) % 5;
      if (c > 4) c = 4;
      v |= (uint64_t)c << (4 * i);
    }
    return v;
  };
  NoisyVoteT vote;
  vote.s = seed;
  vote.noise = noise;
  vote.other_T = other_T;
  vote.max_last = 3;
  return myers_warp<4, false>(L, T, k, true, pf, t16, vote);
}

uint32_t emul_edit_distance(const uint8_t* pat, uint32_t L, uint32_t rc, const uint8_t* txt, uint32_t T,
                            int ncls) {
  return emul_edit_distance_k(pat, L, rc, txt, T, ncls, 0xfffffffeu);
}

// the whole pipeline, one query at a time, in the stage order of binner.cu
int emul_bin_reads(void* p, const uint8_t* seqs, const uint64_t* seq_off, uint64_t n_reads,
                   const emul_params* ep, HitRec** hits_out, uint64_t** off_out) {
  EmulIndex* e = (EmulIndex*)p;
  Params prm;
  prm.edit_rate = ep->edit_rate;
  prm.min_seed = ep->min_seed;
  prm.S = ep->seed_size;
  prm.G = ep->seed_gap;
  prm.max_hits = ep->max_hits;
  prm.tune_max_hits = ep->tune_max_hits;
  prm.max_candidates = ep->max_candidates < 0 ? -1 : ep->max_candidates;
  prm.max_assignments = ep->max_assignments < 0 ? -1 : ep->max_assignments;
  prm.ns = ep->strands == 1 ? 1 : 2;
  ReadsView rv{seqs, seq_off, 0, (uint32_t)n_reads};
  std::vector<HitRec> all;
  std::vector<uint64_t> offs(n_reads + 1, 0);
  const uint32_t nq = (uint32_t)n_reads * prm.ns;
  for (uint32_t q = 0; q < nq; ++q) {
    if (q % prm.ns == 0) offs[q / prm.ns] = all.size();
    uint32_t L = query_len(rv, prm.ns, q);
    const uint8_t* seq = seqs + seq_off[q / prm.ns];
    uint32_t rc = q % prm.ns;
    std::vector<ReadWord> qwords = encode_query(seq, L, rc != 0, false);
    uint32_t nslots = seed_slots(L, prm.S, prm.G);
    std::vector<uint32_t> lo(nslots), cnt(nslots), hoff(nslots);
    for (uint32_t j = 0; j < nslots; ++j)
      seed_search_item(e->fm, e->kt, qwords.data(), L, prm.S, j * prm.G, &lo[j], &cnt[j], nullptr);
    uint32_t nseeds = 0, nhits = 0, ovf = 0;
    if (nslots && query_hopeless(qwords.data(), L, edit_budget(L, prm.edit_rate))) {
      for (uint32_t j = 0; j < nslots; ++j) hoff[j] = kUnused;
    } else {
      seed_select_item(prm, nslots, cnt.data(), hoff.data(), &nseeds, &nhits, &ovf);
    }
    if (ovf) return -7;
    std::vector<uint64_t> keys(nhits);
    for (uint32_t j = 0; j < nslots; ++j)
      if (hoff[j] != kUnused)
        for (uint32_t r = 0; r < (cnt[j] & kSlotCountMask); ++r)
          keys[hoff[j] + r] = (cnt[j] & kDirectHit) ? make_hit_key(lo[j], j * prm.G)
                                                    : make_hit_key(fm_locate(e->fm, e->sv, lo[j] + r, nullptr), j * prm.G);
    std::sort(keys.begin(), keys.end());
    uint32_t k = edit_budget(L, prm.edit_rate);
    std::vector<CandRec> cand(nhits ? nhits : 1);
    uint32_t nc = nhits ? coalesce_item(e->bv, keys.data(), nhits, min_seeds_of(nseeds, prm.min_seed), L, k,
                                        cand.data())
                        : 0;
    std::vector<uint64_t> rkeys(nc ? nc : 1);
    for (uint32_t i = 0; i < nc; ++i) rkeys[i] = make_rank_key(cand[i].num_seeds, i);
    std::sort(rkeys.begin(), rkeys.begin() + nc);
    std::vector<CandRec> dense(nc ? nc : 1);
    std::vector<uint32_t> edits(nc ? nc : 1);
    for (uint32_t i = 0; i < nc; ++i) {
      dense[i] = cand[(uint32_t)(rkeys[i] & 0xffffffffu)];
      bool skip = (prm.max_candidates >= 0 && (uint64_t)i >= (uint64_t)prm.max_candidates) ||
                  2ull * k > (uint64_t)L || L == 0;
      uint32_t ed = kNoEdit;
      if (!skip) {
        const uint8_t* win = e->text.data() + dense[i].start;
        const uint32_t T = dense[i].end - dense[i].start;
        uint32_t end_col = 0;
        ed = edit_distance_k_end(seq, L, rc, win, T, 4, k, &end_col);
        if (ed > k) ed = kNoEdit;
        if (ed != kNoEdit && L >= 254) {  // the SW pre-filter is no longer implied (core.cuh, ssw_word_*)
          auto rcode = [&](uint32_t x) { return plane_code(qwords.data(), x); };
          auto tcode = [&](uint32_t c) { return dna5_code(win[c]); };
          const uint32_t thr = L - 2 * k, w = ed + 1;
          bool ok = false;
          if (w <= kSswBandMaxW) {
            uint16_t Hb[kSswBandCap], Eb[kSswBandCap];
            ok = ssw_word_band(L, T, rcode, tcode, (int64_t)end_col - (int64_t)L, w, thr, Hb, Eb) >= thr;
          }
          if (!ok) {
            std::vector<uint16_t> buf(4 * (size_t)L);
            ok = ssw_accepts_full(L, T, rcode, tcode, thr, buf.data(), buf.data() + L, buf.data() + 2 * L,
                                  buf.data() + 3 * L);
          }
          if (!ok) ed = kNoEdit;
        }
      }
      edits[i] = ed;
    }
    std::vector<HitRec> out(nc ? nc : 1);
    uint32_t no = select_item(e->bv, prm, dense.data(), edits.data(), nc, k, out.data());
    all.insert(all.end(), out.begin(), out.begin() + no);
  }
  offs[n_reads] = all.size();
  *hits_out = (HitRec*)malloc((all.size() ? all.size() : 1) * sizeof(HitRec));
  if (!all.empty()) memcpy(*hits_out, all.data(), all.size() * sizeof(HitRec));
  *off_out = (uint64_t*)malloc((n_reads + 1) * 8);
  memcpy(*off_out, offs.data(), (n_reads + 1) * 8);
  return 0;
}

// slice schedule of one batch call (core.cuh::sub_batch_bounds); returns the number of boundaries
uint32_t emul_sub_batch_bounds(uint64_t n_reads, uint64_t step, int ramp, uint64_t* out, uint32_t cap) {
  std::vector<uint64_t> b = sub_batch_bounds(n_reads, step, ramp != 0);
  for (size_t i = 0; i < b.size() && i < cap; ++i) out[i] = b[i];
  return (uint32_t)b.size();
}

// the slices one batch call computes (core.cuh::slice_bounds); returns the number of boundaries
uint32_t emul_slice_bounds(uint64_t n_reads, uint64_t step, int host_input, int two_lanes, uint64_t* out,
                           uint32_t cap) {
  std::vector<uint64_t> b = slice_bounds(n_reads, step, host_input != 0, two_lanes != 0);
  for (size_t i = 0; i < b.size() && i < cap; ++i) out[i] = b[i];
  return (uint32_t)b.size();
}

// packed reads: the device's unpacker (core.cuh::unpack_word) applied to a record, next to the planes the device
// computes from the raw bytes (encode_fwd_word).  out: W words of {lo, hi, nn} for each of the two routes.
// `from_record`: a record made elsewhere (the product's AVX2 / SWAR packer); NULL = core.cuh::pack_read.
uint32_t emul_packed_words(const uint8_t* seq, uint32_t L, const uint8_t* from_record, uint64_t* unpacked,
                           uint64_t* encoded) {
  std::vector<uint8_t> rec(packed_record_bytes(L) + 1);
  if (from_record) memcpy(rec.data(), from_record, packed_record_bytes(L));
  else pack_read(seq, L, rec.data());
  const uint32_t W = (L + 63) >> 6;
  for (uint32_t w = 0; w < W; ++w) {
    ReadWord a = unpack_word(rec.data(), L, w), b = encode_fwd_word(seq, L, w, false);
    unpacked[3 * w] = a.lo, unpacked[3 * w + 1] = a.hi, unpacked[3 * w + 2] = a.nn;
    encoded[3 * w] = b.lo, encoded[3 * w + 1] = b.hi, encoded[3 * w + 2] = b.nn;
  }
  return W;
}

void emul_free(void* p) { free(p); }

void emul_myers_counters(unsigned long long* blocks, unsigned long long* cols, int reset) {
  *blocks = mtsv::g_myers_blocks;
  *cols = mtsv::g_myers_cols;
  if (reset) mtsv::g_myers_blocks = mtsv::g_myers_cols = 0;
}

}  // extern "C"
