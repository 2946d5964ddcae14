// core.cuh — device data layout and the per-work-item logic of every hot-path stage.
//
// Everything here is `__host__ __device__` so that tests/emul/ can compile the very same
// arithmetic with g++ and diff it against the oracle without a GPU (test-only; the product
// library has no CPU path).  Kernels in binner.cu / index.cu are thin grids over these items.
//
// Reference (FofanovLab/mtsv_tools v2.1.0) lines restated by each item are cited inline.
#pragma once
#include <stdint.h>

#include <algorithm>
#include <vector>

#if defined(__CUDACC__)
#define MTSV_HD __host__ __device__ __forceinline__
#else
#define MTSV_HD inline
struct uint2 {  // CUDA vector type, for the g++ build of tests/emul/
  uint32_t x, y;
};
#endif

namespace mtsv {

// ---------------------------------------------------------------------------------------------
// small helpers
// ---------------------------------------------------------------------------------------------
MTSV_HD int popc64(uint64_t x) {
#ifdef __CUDA_ARCH__
  return __popcll(x);
#else
  return __builtin_popcountll(x);
#endif
}

template <typename T>
MTSV_HD T ldg(const T* p) {
#ifdef __CUDA_ARCH__
  return __ldg(p);
#else
  return *p;
#endif
}

// symbol codes used on the device: A C G T in 2 bits, N and '$' are "exceptions"
enum : uint32_t { SYM_A = 0, SYM_C = 1, SYM_G = 2, SYM_T = 3, SYM_N = 4, SYM_DOLLAR = 5, SYM_OTHER = 6 };

// Branch-free byte -> symbol code.  (b >> 1) & 7 separates the five letters: A 0, C 1, T 2, G 3,
// N 7; a 3-bit-per-entry table maps that to the code and a comparison against the canonical byte of
// the code rejects every other byte.  (A `switch` here compiles to a divergent branch tree, which the
// verifier would execute once per DP column.)
MTSV_HD uint32_t upper_acgtn_code(uint32_t b) {  // A,C,G,T,N (upper case) -> 0..4, anything else -> 7
  const uint32_t lut = (0u << 0) | (1u << 3) | (3u << 6) | (2u << 9) | (7u << 12) | (7u << 15) | (7u << 18) |
                       (4u << 21);
  uint32_t code = (lut >> (3 * ((b >> 1) & 7))) & 7;
  const uint64_t canon = 0x4E54474341ull;  // "ACGTN" little-endian
  uint32_t want = (uint32_t)(canon >> (8 * (code & 7))) & 0xff;  // code 7 -> 0 (never a letter)
  return (code < 5 && want == b) ? code : 7u;
}

// read normalisation of src/binner.rs:88-100 fused with the 0..4 encoding: upper/lower case ACGT
// keep their base, everything else (N, n, IUPAC, garbage) is N
MTSV_HD uint32_t read_code(uint8_t b) {
  uint32_t u = (uint32_t)b & 0xDFu;  // fold lower case onto upper case
  uint32_t c = upper_acgtn_code(u);
  // bytes whose folded value is a letter but which are not letters themselves (0x01/0x03/0x07/0x14
  // | 0x20 variants are letters; only b in 0x41..0x5A or 0x61..0x7A can fold to a letter) are fine:
  // folding only clears bit 5, so u is a letter iff b is that letter in either case.
  return c < 4 ? c : (uint32_t)SYM_N;
}
// reference text bytes are already upper-case ACGTN (src/index.rs:543-553)
MTSV_HD uint32_t text_code(uint8_t b) {
  uint32_t c = upper_acgtn_code(b);
  return c < 5 ? c : (b == '$' ? (uint32_t)SYM_DOLLAR : (uint32_t)SYM_OTHER);
}
// bio::alphabets::dna::revcomp on the normalised alphabet (src/binner.rs:115): A<->T C<->G N->N
MTSV_HD uint32_t comp_code(uint32_t c) { return c < 4 ? 3u - c : c; }

// ---------------------------------------------------------------------------------------------
// FM-index layout in HBM
//
// One 32-byte sector per 64 BWT rows: relative A/C/G/T counts (u16, relative to the enclosing
// 32768-row superblock), a 64-bit exception plane (rows holding N or '$'), and the two bit
// planes of the 2-bit symbol code.  A rank query = one sector from here + 16 bytes from the tiny
// (n/2048 bytes) superblock table that lives in L2.  Replaces rust-bio's byte BWT + 11 separate
// u64 checkpoint arrays (Occ::get, SURVEY app. B) — same counts, different bytes.
// ---------------------------------------------------------------------------------------------
struct __attribute__((aligned(32))) FmBlock {
  uint64_t rel;  // four u16 relative counts: A | C << 16 | G << 32 | T << 48
  uint64_t exc;
  uint64_t lo;
  uint64_t hi;
};
static_assert(sizeof(FmBlock) == 32, "FmBlock must be one 32-byte sector");

constexpr uint32_t kRowsPerBlock = 64;
constexpr uint32_t kBlocksPerSuper = 512;  // 32768 rows: relative counts fit u16

struct SuperCounts {  // absolute counts of A,C,G,T before the superblock
  uint32_t c[4];
};

struct FmView {
  const FmBlock* blocks;      // n/64 + 1
  const SuperCounts* super;   // per 512 blocks
  const uint32_t* n_before;   // per block: number of N in bwt[0 .. 64*blk)
  const uint32_t* C;          // device array[5]: `less` for A,C,G,T,N (byte order $ < A < C < G < N < T)
  uint32_t n;                 // rows (= text length incl. '$')
  uint32_t dollar_row;        // the single row whose BWT symbol is '$'
};

MTSV_HD FmBlock load_block(const FmBlock* p) {
#ifdef __CUDA_ARCH__
  // the whole 32-byte sector in ONE 256-bit read-only load (sm_100: ld.global.nc.v8.u32; tools/randbench2.cu found
  // it the fastest flavour for dependent random sector fetches, ahead of two 128-bit loads)
  FmBlock b;
  uint32_t x0, x1, x2, x3, x4, x5, x6, x7;
  asm("ld.global.nc.v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(x0), "=r"(x1), "=r"(x2), "=r"(x3), "=r"(x4), "=r"(x5), "=r"(x6), "=r"(x7)
               : "l"(p));
  b.rel = (uint64_t)x0 | ((uint64_t)x1 << 32);
  b.exc = (uint64_t)x2 | ((uint64_t)x3 << 32);
  b.lo = (uint64_t)x4 | ((uint64_t)x5 << 32);
  b.hi = (uint64_t)x6 | ((uint64_t)x7 << 32);
  return b;
#else
  return *p;
#endif
}

// occurrences of symbol a (0..3) among the first j (0..63) rows of the block, plus its rel count
MTSV_HD uint32_t block_occ(const FmBlock& b, uint32_t a, uint32_t j) {
  uint64_t m = ~b.exc & ((a & 1) ? b.lo : ~b.lo) & ((a & 2) ? b.hi : ~b.hi);
  return (uint32_t)((b.rel >> (16 * a)) & 0xffff) + (uint32_t)popc64(m & ((1ull << j) - 1));
}

// occ(a, i) = number of `a` in bwt[0 .. i)   (== bio Occ::get(bwt, i-1, a) for i > 0)
MTSV_HD uint32_t fm_occ(const FmView& fm, uint32_t a, uint32_t i) {
  uint32_t blk = i >> 6, j = i & 63;
  if (a < 4) {
    uint32_t sup = ldg(&fm.super[blk >> 9].c[a]);
    FmBlock b = load_block(fm.blocks + blk);
    return sup + block_occ(b, a, j);
  }
  // N: absolute per-block count (side array, touched only by N queries) + exception plane
  FmBlock b = load_block(fm.blocks + blk);
  uint32_t c = ldg(&fm.n_before[blk]) + (uint32_t)popc64(b.exc & ((1ull << j) - 1));
  uint32_t base = blk << 6;
  if (fm.dollar_row >= base && fm.dollar_row < i) c -= 1;
  return c;
}

// BWT symbol at a row
MTSV_HD uint32_t fm_symbol(const FmView& fm, const FmBlock& b, uint32_t row) {
  uint32_t j = row & 63;
  if ((b.exc >> j) & 1) return row == fm.dollar_row ? SYM_DOLLAR : SYM_N;
  return (uint32_t)((b.lo >> j) & 1) | ((uint32_t)((b.hi >> j) & 1) << 1);
}

// One backward-search step on the half-open interval [l,u) — bio FMIndexable::backward_search
// body: l = less[a] + occ(l-1,a) ; r = less[a] + occ(r,a) - 1  with u = r + 1.
MTSV_HD uint32_t fm_step(const FmView& fm, uint32_t a, uint32_t& l, uint32_t& u) {
  uint32_t sectors = 1;  // FmBlock sectors touched (the roofline's unit of work)
  if (a < 4) {
    uint32_t bl = l >> 6, bu = u >> 6;
    uint32_t sup_l = ldg(&fm.super[bl >> 9].c[a]);
    FmBlock b1 = load_block(fm.blocks + bl);
    uint32_t ol = sup_l + block_occ(b1, a, l & 63);
    uint32_t ou;
    if (bu == bl) {
      ou = sup_l + block_occ(b1, a, u & 63);
    } else {
      FmBlock b2 = load_block(fm.blocks + bu);
      ou = ldg(&fm.super[bu >> 9].c[a]) + block_occ(b2, a, u & 63);
      sectors = 2;
    }
    uint32_t ca = ldg(&fm.C[a]);
    l = ca + ol;
    u = ca + ou;
  } else {
    uint32_t ol = fm_occ(fm, SYM_N, l), ou = fm_occ(fm, SYM_N, u);
    uint32_t cn = ldg(&fm.C[SYM_N]);
    l = cn + ol;
    u = cn + ou;
    sectors = 4;  // two FmBlock sectors + two n_before sectors
  }
  return sectors;
}

// LF mapping used by locate — bio SampledSuffixArray::get: pos = less[c] + occ(pos-1, c)
MTSV_HD uint32_t fm_lf(const FmView& fm, uint32_t c, const FmBlock& b, uint32_t row) {
  uint32_t blk = row >> 6, j = row & 63;
  if (c < 4) return ldg(&fm.C[c]) + ldg(&fm.super[blk >> 9].c[c]) + block_occ(b, c, j);
  uint32_t cnt = ldg(&fm.n_before[blk]) + (uint32_t)popc64(b.exc & ((1ull << j) - 1));
  uint32_t base = blk << 6;
  if (fm.dollar_row >= base && fm.dollar_row < row) cnt -= 1;
  return ldg(&fm.C[SYM_N]) + cnt;
}

// Suffix array as kept on the device: rows 0, s', 2s', ... (s' = 1 means the full array).
struct SaView {
  const uint32_t* sa;
  uint32_t rate;  // s'
};

// SampledSuffixArray::get (bio 3.0.0; SURVEY §8 a-3) on the device layout.  The '$' row needs no
// extra_rows entry here: its suffix is text position 0.
MTSV_HD uint32_t fm_locate(const FmView& fm, const SaView& sv, uint32_t row, uint32_t* lf_steps) {
  uint32_t off = 0;
  for (;;) {
    if (sv.rate == 1) break;
    if (row % sv.rate == 0) break;
    FmBlock b = load_block(fm.blocks + (row >> 6));
    uint32_t c = fm_symbol(fm, b, row);
    if (c == SYM_DOLLAR) {
      if (lf_steps) *lf_steps += off;
      return off;  // SA[dollar_row] = 0
    }
    row = fm_lf(fm, c, b, row);
    ++off;
  }
  if (lf_steps) *lf_steps += off;
  return ldg(&sv.sa[row / sv.rate]) + off;
}

// k-mer interval table: entry for a k-mer w (key = lo plane | hi plane << k, base j at bit j)
// = SA interval [l,u) of w, or l == u when absent.  Legal shortcut 5 of SURVEY app. A.
//
// "Direct" entries: a k-mer that occurs exactly ONCE in the text does not need its SA interval — whatever longer
// seed ends with it can only occur at that one place.  Such an entry holds the text position of the k-mer and
// the 8 symbols that precede it (3 bits each): the remaining S - k symbols of a seed are compared right there
// (further back than 8: against the text itself), and the seed's hit is (position - (S - k)) without any
// rank query and without touching the suffix array.  On a 1 Gbp index that is every true seed outside repeats:
// one 128-byte line per seed instead of one table line + two FM lines + one SA line.
struct KtabView {
  const uint2* tab;
  uint32_t k;           // 0 = no table
  uint32_t direct;      // 1 = unique k-mers are stored as direct entries
  const uint8_t* text;  // the reference text (only read for seeds longer than k + 8)
};
constexpr uint32_t kKtabDirectTag = 0xFFu;       // e.y >> 24 of a direct entry (needs n < 0xFF000000)
constexpr uint32_t kKtabDirectCtx = 8;           // preceding symbols kept in the entry
constexpr uint32_t kDirectHit = 0x80000000u;     // flag in a slot's count: `lo` is a text position, count 1
constexpr uint32_t kSlotCountMask = 0x7fffffffu;

// symbol class used to compare text with seed symbols: A,C,G,T = 0..3, N = 4, anything else 5
MTSV_HD uint32_t ktab_ctx_code(uint8_t b) {
  uint32_t c = upper_acgtn_code(b);
  return c <= 4 ? c : 5u;
}
MTSV_HD uint2 ktab_direct_entry(uint32_t pos, const uint8_t* text) {
  uint32_t ctx = 0;
  for (uint32_t t = 1; t <= kKtabDirectCtx; ++t) {
    uint32_t c = pos >= t ? ktab_ctx_code(ldg(text + pos - t)) : 5u;
    ctx |= c << (3 * (t - 1));
  }
  uint2 e;
  e.x = pos;
  e.y = (kKtabDirectTag << 24) | ctx;
  return e;
}

// ---------------------------------------------------------------------------------------------
// batch description
// ---------------------------------------------------------------------------------------------
struct Params {  // mtsvgpu_params, validated
  double edit_rate, min_seed;
  uint32_t S, G;
  uint64_t max_hits, tune_max_hits;
  int64_t max_candidates, max_assignments;
  uint32_t ns;  // strands per read: 1 or 2
};

struct ReadsView {
  const uint8_t* seqs;
  const uint64_t* seq_off;  // indexed by absolute read id
  uint64_t read0;           // first read of this sub-batch
  uint32_t n_reads;
};

MTSV_HD uint32_t query_len(const ReadsView& rv, uint32_t ns, uint32_t q) {
  uint64_t r = rv.read0 + q / ns;
  return (uint32_t)(ldg(&rv.seq_off[r + 1]) - ldg(&rv.seq_off[r]));
}

// ---------------------------------------------------------------------------------------------
// reads as bit planes
//
// Every read-strand ("query") is encoded once per batch into 64-base words of three bit planes:
// lo/hi = the two bits of the base code (A 0, C 1, G 2, T 3), nn = "not a base" (N after the
// normalisation of src/binner.rs:88-100).  Seed search then takes a seed's bases and its k-mer table
// key with a couple of shifts, and the verifier gets its pattern-match masks with a few logic ops,
// instead of one byte load + classification per base per use.
// ---------------------------------------------------------------------------------------------
struct ReadWord {
  uint64_t lo, hi, nn;
};

MTSV_HD uint64_t brev64(uint64_t x) {
#ifdef __CUDA_ARCH__
  return __brevll(x);
#else
  x = ((x >> 1) & 0x5555555555555555ull) | ((x & 0x5555555555555555ull) << 1);
  x = ((x >> 2) & 0x3333333333333333ull) | ((x & 0x3333333333333333ull) << 2);
  x = ((x >> 4) & 0x0f0f0f0f0f0f0f0full) | ((x & 0x0f0f0f0f0f0f0f0full) << 4);
  return __builtin_bswap64(x);
#endif
}

MTSV_HD uint64_t low_mask(uint32_t nbits) { return nbits >= 64 ? ~0ull : ((1ull << nbits) - 1); }

// word w (bases 64w .. 64w+63) of the forward strand.  raw = false: binner normalisation (upper and
// lower case ACGT are bases, everything else is N).  raw = true: bytes as they are (stage-level
// edit-distance entry point): A,C,G,T bases, 'N' is nn with lo = hi = 0, any other byte is nn with lo = 1
// ("matches nothing").
MTSV_HD ReadWord encode_fwd_word(const uint8_t* seq, uint32_t L, uint32_t w, bool raw) {
  ReadWord r{0, 0, 0};
  uint32_t base = w * 64;
  uint32_t lim = L > base ? (L - base < 64 ? L - base : 64) : 0;
  for (uint32_t b = 0; b < lim; ++b) {
    uint8_t byte = ldg(seq + base + b);
    uint32_t c = raw ? text_code(byte) : read_code(byte);
    uint64_t is_base = c < 4;
    r.lo |= (uint64_t)((c & 1) & is_base) << b;
    r.hi |= (uint64_t)(((c >> 1) & 1) & is_base) << b;
    r.nn |= (uint64_t)(1 - is_base) << b;
    if (raw && c > 4) r.lo |= 1ull << b;
  }
  return r;
}

// Eight read bytes at once (SWAR): returns the lo / hi / nn plane bits of the 8 bases in the low 8 bits
// of each output.  Same normalisation as read_code (src/binner.rs:88-100).
MTSV_HD void encode8(uint64_t x, uint32_t* lo, uint32_t* hi, uint32_t* nn) {
  const uint64_t k7f = 0x7f7f7f7f7f7f7f7full, k80 = 0x8080808080808080ull;
  uint64_t u = x & 0xdfdfdfdfdfdfdfdfull;  // fold lower case onto upper case
  // zero-byte detector: 0x80 in every byte of v that is zero (exact, no cross-byte borrow)
#define MTSV_ZB(v) (~((((v) & k7f) + k7f) | (v)) & k80)
  uint64_t za = MTSV_ZB(u ^ 0x4141414141414141ull), zc = MTSV_ZB(u ^ 0x4343434343434343ull);
  uint64_t zg = MTSV_ZB(u ^ 0x4747474747474747ull), zt = MTSV_ZB(u ^ 0x5454545454545454ull);
#undef MTSV_ZB
  uint64_t l = zc | zt, h = zg | zt, b = za | l | zg;
  // gather bit 7 of every byte into 8 adjacent bits: (z >> 7) * 0x0102040810204080 puts byte i's flag at bit 56 + i
  const uint64_t mul = 0x0102040810204080ull;
  *lo = (uint32_t)(((l >> 7) * mul) >> 56);
  *hi = (uint32_t)(((h >> 7) * mul) >> 56);
  *nn = (uint32_t)((((b ^ k80) >> 7) * mul) >> 56);
}

// word w of the reverse-complement strand from the forward words (bio::alphabets::dna::revcomp on the
// normalised alphabet, src/binner.rs:115): rc[i] = comp(fwd[L-1-i]), N stays N.
MTSV_HD ReadWord encode_rc_word(const ReadWord* fwd, uint32_t L, uint32_t w) {
  const uint32_t W = (L + 63) >> 6;
  const uint32_t s = W * 64 - L;  // 0..63
  ReadWord out{0, 0, 0};
  // R[x] = bit-reversed complement of fwd[W-1-x]; rc = R >> s (multi-word)
  for (uint32_t t = 0; t < 2; ++t) {
    uint32_t x = w + t;
    if (x >= W) break;
    if (t == 1 && s == 0) break;
    ReadWord f = fwd[W - 1 - x];
    uint32_t fbits = (W - 1 - x) == W - 1 ? L - (W - 1) * 64 : 64;
    uint64_t valid = low_mask(fbits) & ~f.nn;
    uint64_t rlo = brev64(~f.lo & valid), rhi = brev64(~f.hi & valid), rnn = brev64(f.nn & low_mask(fbits));
    if (t == 0) {
      out.lo |= rlo >> s;
      out.hi |= rhi >> s;
      out.nn |= rnn >> s;
    } else {
      out.lo |= rlo << (64 - s);
      out.hi |= rhi << (64 - s);
      out.nn |= rnn << (64 - s);
    }
  }
  return out;
}

// ---------------------------------------------------------------------------------------------
// packed reads (mtsvgpu_bin_batch_packed): what a host parser hands over instead of raw bytes.  The record of a
// read of L bases is three bit planes of ceil(L/8) bytes each — lo, hi (the two bits of the base code, A 0, C 1,
// G 2, T 3) and nn (1 = not a base after the normalisation of src/binner.rs:88-100; lo = hi = 0 there) — base j
// at bit j % 8 of byte j / 8.  Records follow each other without padding: 57 bytes for a 150-base read.
// ---------------------------------------------------------------------------------------------
MTSV_HD uint32_t packed_plane_bytes(uint32_t L) { return (L + 7) >> 3; }
MTSV_HD uint32_t packed_record_bytes(uint32_t L) { return 3 * packed_plane_bytes(L); }

// word w (64 bases) of a packed record
MTSV_HD ReadWord unpack_word(const uint8_t* rec, uint32_t L, uint32_t w) {
  const uint32_t pb = packed_plane_bytes(L);
  const uint32_t b0 = w * 8;
  const uint32_t nb = pb > b0 ? (pb - b0 < 8 ? pb - b0 : 8) : 0;
  uint64_t v[3] = {0, 0, 0};
  for (uint32_t pl = 0; pl < 3; ++pl)
    for (uint32_t i = 0; i < nb; ++i) v[pl] |= (uint64_t)ldg(rec + pl * pb + b0 + i) << (8 * i);
  const uint32_t bits = L > w * 64 ? (L - w * 64 < 64 ? L - w * 64 : 64) : 0;
  const uint64_t m = low_mask(bits);
  ReadWord r;
  r.nn = v[2] & m;
  r.lo = v[0] & m & ~r.nn;
  r.hi = v[1] & m & ~r.nn;
  return r;
}

// host side of the format (also what tests/emul compiles): one read
inline void pack_read(const uint8_t* seq, uint32_t L, uint8_t* rec) {
  const uint32_t pb = packed_plane_bytes(L);
  for (uint32_t i = 0; i < 3 * pb; ++i) rec[i] = 0;
  for (uint32_t j = 0; j < L; ++j) {
    const uint32_t c = read_code(seq[j]);
    const uint32_t bit = 1u << (j & 7);
    if (c < 4) {
      if (c & 1) rec[j >> 3] |= (uint8_t)bit;
      if (c & 2) rec[pb + (j >> 3)] |= (uint8_t)bit;
    } else {
      rec[2 * pb + (j >> 3)] |= (uint8_t)bit;
    }
  }
}

// where a query's words live: reads are laid out by a closed form of their byte offset, so no scan
// is needed: woff(r) = floor((seq_off[r] - seq_off[read0]) / 64) + (r - read0); the second strand
// follows the first at + total_words.
struct EncView {
  const ReadWord* words;
  uint32_t total_words;  // woff(n_reads): words of one strand
};

MTSV_HD uint32_t query_word_off(const ReadsView& rv, const EncView& ev, uint32_t ns, uint32_t q) {
  uint32_t r = q / ns;
  uint64_t rel = ldg(&rv.seq_off[rv.read0 + r]) - ldg(&rv.seq_off[rv.read0]);
  return (uint32_t)(rel >> 6) + r + (q % ns) * ev.total_words;
}

// 64 consecutive bases starting at `pos` as plane windows (bit i = base pos + i)
MTSV_HD ReadWord plane_window(const ReadWord* qw, uint32_t n_words, uint32_t pos) {
  uint32_t w0 = pos >> 6, sh = pos & 63;
  ReadWord a = qw[w0];
  if (sh == 0) return a;
  ReadWord out{a.lo >> sh, a.hi >> sh, a.nn >> sh};
  if (w0 + 1 < n_words) {
    ReadWord b = qw[w0 + 1];
    out.lo |= b.lo << (64 - sh);
    out.hi |= b.hi << (64 - sh);
    out.nn |= b.nn << (64 - sh);
  }
  return out;
}

// k = ceil(len * edit_freq) in f64 — src/index.rs:281-282
MTSV_HD uint32_t edit_budget(uint32_t L, double edit_rate) {
  double v = (double)L * edit_rate;
  double c = (double)(int64_t)v;
  if (c < v) c += 1.0;
  if (c < 0) c = 0;
  if (c > 4294967295.0) c = 4294967295.0;
  return (uint32_t)c;
}

// number of seed start offsets: (0..len+1-S).step(G) — src/index.rs:284-286.  len < S-1 makes the
// reference panic (usize wrap + out-of-range slice); defined here as no seeds.
MTSV_HD uint32_t seed_slots(uint32_t L, uint32_t S, uint32_t G) {
  if (L + 1 < S || L + 1 == S) return 0;
  uint32_t starts = L + 1 - S;
  return (starts + G - 1) / G;
}

// ---------------------------------------------------------------------------------------------
// stage: seed search (one item per seed slot) — src/index.rs:305 + bio backward_search
// Only `Complete` results matter to the caller (src/index.rs:312-332): cnt = 0 otherwise.
// ---------------------------------------------------------------------------------------------
// The k-mer table is keyed by the bit planes of the k-mer: key = lo | hi << k with base j at bit j.
MTSV_HD void seed_search_item(const FmView& fm, const KtabView& kt, const ReadWord* qw, uint32_t L,
                              uint32_t S, uint32_t seed_off, uint32_t* out_lo, uint32_t* out_cnt,
                              uint32_t* rank_steps) {
  const uint32_t n_words = (L + 63) >> 6;
  uint32_t l = 0, u = fm.n;
  uint32_t steps = 0;
  if (S <= 64) {
    // the whole seed in one window: bit i = base seed_off + i
    ReadWord win = plane_window(qw, n_words, seed_off);
    int i = (int)S - 1;
    if (kt.k && kt.k <= S) {
      // the table replaces the first k steps (the last k bases of the seed) when none is N
      uint32_t sh = S - kt.k;
      uint64_t km = low_mask(kt.k);
      if (((win.nn >> sh) & km) == 0) {
        uint64_t key = ((win.lo >> sh) & km) | (((win.hi >> sh) & km) << kt.k);
        uint2 e = ldg(&kt.tab[key]);
        steps = 1;  // one table sector
        if (kt.direct && (e.y >> 24) == kKtabDirectTag) {
          // the k-mer occurs once, at text position e.x: compare the other S - k symbols with what precedes it
          const uint32_t m = sh, pos = e.x;
          bool ok = pos >= m;
          for (uint32_t t = 1; t <= m && ok; ++t) {
            const uint32_t j = m - t;  // seed symbol index
            const uint32_t a = ((win.nn >> j) & 1) ? (uint32_t)SYM_N
                                                   : ((uint32_t)((win.lo >> j) & 1) | ((uint32_t)((win.hi >> j) & 1) << 1));
            const uint32_t c = t <= kKtabDirectCtx ? (e.y >> (3 * (t - 1))) & 7u : ktab_ctx_code(ldg(kt.text + pos - t));
            ok = c == a;
          }
          if (rank_steps) *rank_steps = steps + (m > kKtabDirectCtx ? 1u : 0u);
          *out_lo = ok ? pos - m : 0;
          *out_cnt = ok ? (1u | kDirectHit) : 0;
          return;
        }
        l = e.x;
        u = e.y;
        i -= (int)kt.k;
      }
    }
    for (; i >= 0 && l < u; --i) {
      uint32_t a = ((win.nn >> i) & 1) ? (uint32_t)SYM_N
                                       : ((uint32_t)((win.lo >> i) & 1) | ((uint32_t)((win.hi >> i) & 1) << 1));
      steps += fm_step(fm, a, l, u);
    }
  } else {
    // long seeds: one plane read per base, no table
    for (int i = (int)S - 1; i >= 0 && l < u; --i) {
      uint32_t pos = seed_off + (uint32_t)i;
      ReadWord w = qw[pos >> 6];
      uint32_t b = pos & 63;
      uint32_t a = ((w.nn >> b) & 1) ? (uint32_t)SYM_N
                                     : ((uint32_t)((w.lo >> b) & 1) | ((uint32_t)((w.hi >> b) & 1) << 1));
      steps += fm_step(fm, a, l, u);
    }
  }
  if (rank_steps) *rank_steps = steps;
  if (l < u) {
    // bit 31 of the count is the direct-hit flag: an interval of 2^31 rows or more (possible beyond 2 Gbp with a
    // very short seed) is clamped — far above any usable max_hits, and above kMaxQueryHits, so the strand is either
    // dropped by the max-hits rule or counted as over the hit limit, exactly as with the true count
    *out_lo = l;
    *out_cnt = u - l < kSlotCountMask ? u - l : kSlotCountMask;
  } else {
    *out_lo = 0;
    *out_cnt = 0;
  }
}

// pattern-match masks of one 64-base word for the verifier: class 0..3 = A,C,G,T; class 4 = N
// (only used by the raw-byte entry point, where N equals N; the binner never matches an N,
// src/index.rs:272-279)
MTSV_HD uint64_t word_peq(const ReadWord& w, uint32_t cls) {
  uint64_t base = ~w.nn;
  switch (cls) {
    case 0: return base & ~w.lo & ~w.hi;
    case 1: return base & w.lo & ~w.hi;
    case 2: return base & ~w.lo & w.hi;
    case 3: return base & w.lo & w.hi;
    default: return w.nn & ~w.lo & ~w.hi;
  }
}

// ---------------------------------------------------------------------------------------------
// stage: seed selection (one item per query) — replays src/index.rs:293-355 over the
// speculatively searched slots.  slot_hoff[slot] = offset of the slot's hits inside the query's
// hit list, or kUnused.
// ---------------------------------------------------------------------------------------------
constexpr uint32_t kUnused = 0xffffffffu;
constexpr uint32_t kMaxQueryHits = 1u << 26;  // per query; beyond this the batch fails loudly

MTSV_HD void seed_select_item(const Params& p, uint32_t nslots, const uint32_t* slot_cnt,
                              uint32_t* slot_hoff, uint32_t* n_seeds, uint32_t* n_hits,
                              uint32_t* overflow) {
  uint64_t next_offset = 0, seed_interval = p.G;
  uint32_t seeds = 0;
  uint64_t total = 0;
  for (uint32_t j = 0; j < nslots; ++j) {
    uint64_t offset = (uint64_t)j * p.G;
    uint32_t cnt = slot_cnt[j] & kSlotCountMask;  // (a direct hit counts 1)
    uint32_t ho = kUnused;
    if (offset >= next_offset && cnt != 0 && (uint64_t)cnt <= p.max_hits) {  // :300-302,:330,:335
      if ((uint64_t)cnt > p.tune_max_hits) {                                 // :338-344
        seed_interval *= 2;
        next_offset = offset + seed_interval;
      }
      if (total + cnt > kMaxQueryHits) {
        *overflow = 1;
      } else {
        ho = (uint32_t)total;
        total += cnt;
      }
      seeds += 1;  // :354
    }
    slot_hoff[j] = ho;
  }
  *n_seeds = seeds;
  *n_hits = (uint32_t)total;
}

// A read-strand that cannot produce a hit whatever its seeds find (result-preserving shortcut):
//  * every N of the read is compared as '.' (src/index.rs:272-279), which equals no reference byte, so each
//    N costs at least one edit in any alignment: more than k of them => min_edit_distance > k (:410);
//  * 2k > L: the SW threshold L - 2k wraps (:406) and nothing is ever accepted.
// Such strands skip locate / coalesce / verify altogether.  (Typical source: reads sampled across an
// N run of the reference, whose N-rich seeds match hundreds of other N runs.)
MTSV_HD bool query_hopeless(const ReadWord* qw, uint32_t L, uint32_t k) {
  if (2ull * k > (uint64_t)L) return true;
  uint32_t n_n = 0;
  for (uint32_t w = 0; w * 64 < L; ++w) {
#ifdef __CUDA_ARCH__
    n_n += (uint32_t)__popcll(qw[w].nn);
#else
    n_n += (uint32_t)__builtin_popcountll(qw[w].nn);
#endif
  }
  return n_n > k;
}

// hit key: (reference_offset << 16) | query_offset — sorts as the derived Ord of SeedHit
// (src/index.rs:109-113, :443)
MTSV_HD uint64_t make_hit_key(uint32_t pos, uint32_t q_off) { return ((uint64_t)pos << 16) | q_off; }

// ---------------------------------------------------------------------------------------------
// stage: candidate windows
// ---------------------------------------------------------------------------------------------
struct BinsView {
  const uint32_t* start;  // nbins
  const uint32_t* end;    // nbins
  const uint32_t* tax;
  const uint32_t* gi;
  uint32_t n;
};

// SeedHit::candidate_indices — src/index.rs:118-153 (u64 wrapping arithmetic of a release build)
MTSV_HD bool candidate_window(uint64_t site, uint64_t seed_offset, uint64_t bin_start,
                              uint64_t bin_end, uint64_t read_len, uint64_t k, uint32_t* ws,
                              uint32_t* we) {
  uint64_t start_offset = seed_offset + k;
  uint64_t cand_start =
      ((uint64_t)(site - start_offset) < bin_start || start_offset > site) ? bin_start
                                                                           : site - start_offset;
  uint64_t cand_end = site + (read_len - seed_offset) + k;
  if (cand_end > bin_end) cand_end = bin_end;
  if (cand_start > cand_end || cand_start < bin_start || cand_end > bin_end ||
      cand_end - cand_start < read_len - k)
    return false;
  *ws = (uint32_t)cand_start;
  *we = (uint32_t)cand_end;
  return true;
}

// first bin with end > site — the `while curr_bin.end <= site` walk of src/index.rs:455-458
MTSV_HD uint32_t find_bin(const BinsView& bv, uint32_t site) {
  uint32_t lo = 0, hi = bv.n;  // answer in [lo, hi)
  while (lo < hi) {
    uint32_t mid = (lo + hi) >> 1;
    if (ldg(&bv.end[mid]) <= site) lo = mid + 1;
    else hi = mid;
  }
  return lo;
}

// min_seeds = max(floor(n_seeds * pct), 1) — src/index.rs:358
MTSV_HD uint32_t min_seeds_of(uint32_t n_seeds, double pct) {
  double v = (double)n_seeds * pct;
  double f = (double)(int64_t)v;  // v >= 0: truncation == floor
  if (f < 1.0) f = 1.0;
  if (f > 4294967295.0) f = 4294967295.0;
  return (uint32_t)f;
}

struct CandRec {  // ReferenceCandidate (src/index.rs:158-165), 16 bytes
  uint32_t start, end, bin, num_seeds;
};

// candidate ranking = `refs.sort_by(|a,b| b.num_seeds.cmp(&a.num_seeds))` (stable, src/index.rs:369):
// by num_seeds descending, ties in discovery order.  Key form of that order (ascending):
MTSV_HD uint64_t make_rank_key(uint32_t num_seeds, uint32_t idx) {
  return ((uint64_t)(~num_seeds) << 32) | idx;
}

// coalesce_seed_sites (src/index.rs:435-487) over the query's sorted hit keys.
// Writes candidates (in discovery order) to cand[0..); returns their number.
MTSV_HD uint32_t coalesce_item(const BinsView& bv, const uint64_t* keys, uint32_t n_hits,
                               uint32_t min_seeds, uint32_t L, uint32_t k, CandRec* cand) {
  uint32_t nc = 0;
  bool have = false;
  CandRec cur{0, 0, 0, 0};
  uint32_t b = 0, b_start = 0, b_end = 0;
  bool b_valid = false;
  for (uint32_t h = 0; h < n_hits; ++h) {
    uint64_t key = keys[h];
    uint32_t site = (uint32_t)(key >> 16), q_off = (uint32_t)(key & 0xffff);
    if (!b_valid || site >= b_end) {  // hits are sorted by site, bins only move forward
      b = find_bin(bv, site);
      b_start = ldg(&bv.start[b]);
      b_end = ldg(&bv.end[b]);
      b_valid = true;
    }
    uint32_t ws = 0, we = 0;
    bool some = candidate_window(site, q_off, b_start, b_end, L, k, &ws, &we);
    bool merged = false;
    if (have && some && b == cur.bin &&
        ((cur.start <= ws && ws < cur.end) || (cur.start < we && we <= cur.end))) {  // :216-221
      cur.start = ws < cur.start ? ws : cur.start;
      cur.end = we > cur.end ? we : cur.end;
      cur.num_seeds += 1;
      merged = true;
    }
    if (!merged) {
      if (have && cur.num_seeds >= min_seeds) {  // :467-469
        cand[nc] = cur;
        ++nc;
      }
      have = some;  // :472 / :475
      if (some) cur = CandRec{ws, we, b, 1};
    }
  }
  if (have && cur.num_seeds >= min_seeds) {  // :481-485
    cand[nc] = cur;
    ++nc;
  }
  return nc;
}

// ---------------------------------------------------------------------------------------------
// stage: verification — Aligner::min_edit_distance (src/align.rs:28-85) as a Myers/Hyyrö
// bit-vector recurrence (semi-global: free start in the text, min over the last row).
// By SURVEY §8 a-7 the SSW pre-filter of src/index.rs:402-406 is implied for reads <= 253 bp.
// ---------------------------------------------------------------------------------------------
constexpr uint32_t kNoEdit = 0xffffffffu;

// One 64-row block of the recurrence for one text column.  phin/mhin: horizontal delta entering
// from the block above (+1 / -1 as separate bits); returns the pre-shift Ph/Mh for score tracking.
MTSV_HD void myers_block(uint64_t Eq, uint64_t& Pv, uint64_t& Mv, uint32_t& phin, uint32_t& mhin,
                         uint64_t& Ph_out, uint64_t& Mh_out) {
  uint64_t Xv = Eq | Mv;
  Eq |= (uint64_t)mhin;
  uint64_t Xh = (((Eq & Pv) + Pv) ^ Pv) | Eq;
  uint64_t Ph = Mv | ~(Xh | Pv);
  uint64_t Mh = Pv & Xh;
  Ph_out = Ph;
  Mh_out = Mh;
  uint32_t pho = (uint32_t)(Ph >> 63), mho = (uint32_t)(Mh >> 63);
  Ph = (Ph << 1) | (uint64_t)phin;
  Mh = (Mh << 1) | (uint64_t)mhin;
  Pv = Mh | ~(Xv | Ph);
  Mv = Ph & Xv;
  phin = pho;
  mhin = mho;
}

// Bounded semi-global edit distance over W 64-row blocks: returns min_j D[L][j] when that is <= k and
// some value > k otherwise (only values <= k are observable at src/index.rs:410).  Pattern masks come
// from peq(class, word) -> u64, the text from text(j) -> class (0..4 match classes, > 4 = matches nothing).
//
// Three exact prunings (SURVEY app. A, transformation 6), all of the form "cells that cannot lie on a
// complete alignment of cost <= k are not computed and are treated as +infinity (over-estimated)":
//   * Ukkonen cut-off, per 64-row block as in Myers' block algorithm: blocks below `last` hold only
//     values > k; block last+1 is (re)activated in the column where the bottom cell of block `last`
//     is <= k in this or the previous column, initialised with vertical deltas +1; a block whose
//     bottom value is >= k + rows holds only values > k and is dropped.
//   * static band: rows above j - (T - L) - k at column j cannot reach row L by column T; whole blocks
//     above it are dropped, the block below receives a horizontal delta of +1 (an over-estimate).
//   * early exit when the active rows can no longer reach row L within the remaining columns.
// Used by the verify kernel (binner.cu) and, compiled with g++, by tests/emul/.
#ifdef MTSV_COUNT_BLOCKS
static unsigned long long g_myers_blocks = 0, g_myers_cols = 0;  // test-only instrumentation
#endif

template <int W, typename PeqF, typename TextF>
MTSV_HD uint32_t myers_bounded(uint32_t L, uint32_t T, uint32_t k, PeqF peq, TextF text,
                               uint32_t* end_col = nullptr) {
  // end_col (optional): number of text columns consumed by the first best alignment found (0 = D[L][0])
  if (end_col) *end_col = 0;
  if (L == 0) return 0;
  if (k > L) k = L;  // D[L][0] = L bounds the answer; also keeps k + rows small
  uint64_t Pv[W], Mv[W];
  uint32_t bs[W];  // bs[w] = D[bottom row of block w][current column]
  const int nb = (int)((L - 1) >> 6);
  const uint32_t sbit = (L - 1) & 63;
#pragma unroll
  for (int w = 0; w < W; ++w) {
    Pv[w] = ~0ull;
    Mv[w] = 0;
    uint32_t bottom = (uint32_t)(w + 1) * 64;
    bs[w] = bottom < L ? bottom : L;
  }
  // column 0: D[i][0] = i, so block w (rows 64w+1..) is active iff 64w + 1 <= k; block 0 always
  int last = k ? (int)((k - 1) >> 6) : 0;
  if (last > nb) last = nb;
  int first = 0;
  uint32_t best = last == nb ? L : k + 1;
  const uint32_t slack = T + k;  // a row i at column j is useful only if i + slack >= L + j
  for (uint32_t j = 0; j < T; ++j) {
    // House-keeping every 8th column only: early exit, band advance and (below) block drops merely
    // prune work, so doing them late is always safe; activation of the next block is checked every column.
    if ((j & 7) == 0) {
      uint32_t reach = (uint32_t)(last + 1) * 64;  // bottom row of the active region
      if (reach < L && (L - reach) > (T - j) + k) break;
      // blocks entirely above the band at column j+1: 64(w+1) + slack < L + j + 1.  The bottom-most
      // active block is never dropped this way: the activation of the block below needs its bottom cell.
#pragma unroll
      for (int w = 0; w < W - 1; ++w)
        if (w == first && w < last && (uint32_t)(w + 1) * 64 + slack < L + j + 1) first = w + 1;
    }
    const uint32_t c = text(j);
#ifdef MTSV_COUNT_BLOCKS
    ++g_myers_cols;
#endif
    uint32_t phin = first > 0 ? 1u : 0u, mhin = 0;
    uint32_t prev_old = 0, prev_new = 0, bottom_score = k + 1;
    bool prev_valid = false;
#pragma unroll
    for (int w = 0; w < W; ++w) {
      if (w <= nb) {
        bool active = w >= first && w <= last;
        if (!active && w == last + 1 && prev_valid && (prev_old <= k || prev_new <= k)) {
          uint32_t rows = w == nb ? L - (uint32_t)w * 64 : 64u;
          Pv[w] = ~0ull;
          Mv[w] = 0;
          bs[w] = prev_old + rows;
          last = w;
          active = true;
        }
        if (active) {
          uint64_t Eq = c <= 4 ? peq(c, w) : 0ull;
          uint64_t Ph, Mh;
          prev_old = bs[w];
          myers_block(Eq, Pv[w], Mv[w], phin, mhin, Ph, Mh);
#ifdef MTSV_COUNT_BLOCKS
          ++g_myers_blocks;
#endif
          const uint32_t bit = w == nb ? sbit : 63u;
          bs[w] += (uint32_t)((Ph >> bit) & 1);
          bs[w] -= (uint32_t)((Mh >> bit) & 1);
          prev_new = bs[w];
          prev_valid = true;
          if (w == nb) bottom_score = bs[w];
        } else {
          prev_valid = false;
        }
      }
    }
    // drop blocks that hold only values > k (keep the top-most active one)
    if ((j & 7) == 7) {
#pragma unroll
      for (int w = W - 1; w >= 1; --w) {
        if (w <= nb && w == last && w > first) {
          uint32_t rows = w == nb ? L - (uint32_t)w * 64 : 64u;
          if (bs[w] >= k + rows) last = w - 1;
        }
      }
    }
    if (bottom_score < best) {
      best = bottom_score;
      if (end_col) *end_col = j + 1;
    }
  }
  return best;
}

// ---------------------------------------------------------------------------------------------
// The same bounded recurrence with WARP-UNIFORM control, for reads of at most W <= 4 words (the
// verifier's fast path).  Lanes of a warp run in lock step anyway, so the set of computed blocks
// [first, last] is kept per warp instead of per lane: every decision that only prunes work is taken by
// a vote — a block is activated as soon as ANY lane needs it, dropped / banded out / the loop left only
// when ALL lanes agree.  For a lane this means blocks are activated earlier and dropped later than it
// would on its own, both of which are exact (a block activated early holds true values > k or the
// +1-per-row over-estimate of them; a block kept longer holds exact values).  What this buys: no
// per-lane activity predicates, no divergent sections, and with all reads of one length (UNIFORM)
// the score of every block but the last is tracked with the carry bits the recurrence produces anyway.
//
// Text arrives 16 columns at a time as 4-bit codes (0..3 = A,C,G,T, 4 = matches nothing): text16(j0)
// returns the codes of columns j0 .. j0+15, and may be asked for columns beyond the lane's own T (up to the
// warp's longest window); those columns are computed but never scored.
// Vote: any(bool), all(bool), umax(u32) over the warp (tests/emul supplies a one-lane version that
// perturbs the votes to exercise early activation and late drops).
// ---------------------------------------------------------------------------------------------
// four columns of the recurrence over the blocks F..Z (compile time), straight-line
template <int W, bool UNIFORM, int F, int Z, typename PeqF>
MTSV_HD void myers_cols4(uint32_t codes, uint32_t ncols, uint64_t (&Pv)[W], uint64_t (&Mv)[W], uint32_t (&bs)[W],
                         uint32_t& best, PeqF peq, int nb, uint32_t sbit, uint32_t j, uint32_t T) {
#pragma unroll
  for (uint32_t jj = 0; jj < 4; ++jj) {
    if (jj >= ncols) break;  // warp-uniform
    const uint32_t c = (codes >> (4 * jj)) & 7u;
    uint32_t phin = F > 0 ? 1u : 0u, mhin = 0;
#pragma unroll
    for (int w = F; w <= Z; ++w) {
      uint64_t Ph, Mh;
#ifdef MTSV_COUNT_BLOCKS
      ++g_myers_blocks;
#endif
      myers_block(peq(c, w), Pv[w], Mv[w], phin, mhin, Ph, Mh);  // leaves the carries in phin / mhin
      if (UNIFORM && w < W - 1) {
        bs[w] += phin;
        bs[w] -= mhin;
      } else {
        const uint32_t bit = (UNIFORM || w == nb) ? sbit : 63u;
        bs[w] += (uint32_t)(Ph >> bit) & 1u;
        bs[w] -= (uint32_t)(Mh >> bit) & 1u;
      }
    }
    if (UNIFORM) {
      if (Z == W - 1 && j + jj < T && bs[W - 1] < best) best = bs[W - 1];
    } else if (Z >= nb && F <= nb && j + jj < T) {
      uint32_t v = bs[W - 1];
#pragma unroll
      for (int w = 0; w < W - 1; ++w)
        if (w == nb) v = bs[w];
      if (v < best) best = v;
    }
  }
}

template <int W, bool UNIFORM, int F, typename PeqF>
MTSV_HD void myers_cols4_z(int last, uint32_t codes, uint32_t ncols, uint64_t (&Pv)[W], uint64_t (&Mv)[W],
                           uint32_t (&bs)[W], uint32_t& best, PeqF peq, int nb, uint32_t sbit, uint32_t j,
                           uint32_t T) {
  if (last == F) myers_cols4<W, UNIFORM, F, F>(codes, ncols, Pv, Mv, bs, best, peq, nb, sbit, j, T);
  if (W > F + 1 && last == F + 1)
    myers_cols4<W, UNIFORM, F, (F + 1 < W ? F + 1 : F)>(codes, ncols, Pv, Mv, bs, best, peq, nb, sbit, j, T);
  if (W > F + 2 && last == F + 2)
    myers_cols4<W, UNIFORM, F, (F + 2 < W ? F + 2 : F)>(codes, ncols, Pv, Mv, bs, best, peq, nb, sbit, j, T);
  if (W > F + 3 && last == F + 3)
    myers_cols4<W, UNIFORM, F, (F + 3 < W ? F + 3 : F)>(codes, ncols, Pv, Mv, bs, best, peq, nb, sbit, j, T);
}

template <int W, bool UNIFORM, typename Vote, typename PeqF, typename Text16F>
MTSV_HD uint32_t myers_warp(uint32_t L, uint32_t T, uint32_t k, bool live, PeqF peq, Text16F text16,
                            Vote vote) {
  static_assert(W >= 1 && W <= 4, "fast path: at most 4 words");
  if (!live) {
    L = 0;
    T = 0;
    k = 0;
  }
  const uint32_t Lw = vote.umax(L);
  if (Lw == 0) return 0;
  if (!live) L = Lw;  // idle lanes borrow a length so that their (unused) state stays well defined
  if (k > L) k = L;
  const int nb = UNIFORM ? W - 1 : (int)((L - 1) >> 6);
  const uint32_t sbit = (L - 1) & 63;
  const uint32_t rows_nb = L - (uint32_t)nb * 64;
  uint64_t Pv[W], Mv[W];
  uint32_t bs[W];
#pragma unroll
  for (int w = 0; w < W; ++w) {
    Pv[w] = ~0ull;
    Mv[w] = 0;
    uint32_t bottom = (uint32_t)(w + 1) * 64;
    bs[w] = bottom < L ? bottom : L;
  }
  // column 0: D[i][0] = i, so the blocks holding rows <= k start active
  int lane_last = k ? (int)((k - 1) >> 6) : 0;
  if (lane_last > nb) lane_last = nb;
  int last = (int)vote.umax((uint32_t)lane_last), first = 0;
  uint32_t best = L < k + 1 ? L : k + 1;
  const uint32_t slack = T + k;
  const uint32_t Tw = vote.umax(T);
  for (uint32_t j0 = 0; j0 < Tw; j0 += 16) {
    // ---- pruning votes, once per 16 columns (late pruning is always exact) ----
    const uint32_t reach = (uint32_t)(last + 1) * 64;
    // Value-based pruning of the top block: a cell (i, j) with value D lies on an alignment of cost <= k only if
    // D + (L - i) - (T - j) <= k (the rows still to come need that many vertical moves).  Inside a block
    // D[i] >= D[bottom] - (bottom - i), so D[bottom] + L + j > k + bottom + T rules out every cell of the block
    // at this column; once row 0 can no longer start an alignment (j + L > T + k) everything that enters the
    // block later descends from such cells.
    uint32_t bf = bs[0];
#pragma unroll
    for (int w = 1; w < W; ++w)
      if (w == first) bf = bs[w];
    const uint32_t bottom_f = (uint32_t)(first + 1) * 64 < L ? (uint32_t)(first + 1) * 64 : L;
    const bool top_useless = j0 + L > T + k && bf + L + j0 > k + bottom_f + T;
    const bool done = !live || j0 >= T || (reach < L && (L - reach) > (T - j0) + k) || (first == last && top_useless);
    if (vote.all(done)) break;
    if (first < last) {  // top block entirely above the band: 64(first+1) + slack < L + j0 + 1
      bool can = done || ((uint32_t)(first + 1) * 64 + slack < L + j0 + 1) || top_useless;
      if (vote.all(can)) ++first;
    }
    if (last > first) {  // bottom block holds only values > k (with the margin of the activation rule below)
      uint32_t rows = last == nb ? rows_nb : 64u;
      uint32_t bl = bs[0], bp = bs[0];
#pragma unroll
      for (int w = 1; w < W; ++w) {
        if (w == last) bl = bs[w];
        if (w == last - 1) bp = bs[w];
      }
      bool can = done || last > nb || (bl >= k + rows && bp > k + 4 + 16);
      if (vote.all(can)) --last;
    }
    const uint64_t tw = text16(j0);
    const uint32_t ncols16 = Tw - j0 < 16u ? Tw - j0 : 16u;
    for (uint32_t j4 = 0; j4 < ncols16; j4 += 4) {
      // ---- activation, every 4 columns: the bottom cell of block `last` moves by at most 1 per column, so
      //      block last+1 cannot hold a value <= k within the next 4 columns unless that cell is <= k + 4 now.
      //      The new block starts from the +1-per-row over-estimate below that cell (state of column j-1). ----
      if (last < W - 1) {
        uint32_t bl = bs[0];
#pragma unroll
        for (int w = 1; w < W - 1; ++w)
          if (w == last) bl = bs[w];
        bool want = live && !done && last < nb && bl <= k + 4;
        if (vote.any(want)) {
          ++last;
          const uint32_t init = bl + (last == nb ? rows_nb : 64u);
#pragma unroll
          for (int w = 1; w < W; ++w)
            if (w == last) {
              Pv[w] = ~0ull;
              Mv[w] = 0;
              bs[w] = init;
            }
        }
      }
      const uint32_t codes = (uint32_t)(tw >> (4 * j4)) & 0xffffu;
      const uint32_t ncols = ncols16 - j4 < 4u ? ncols16 - j4 : 4u;
      const uint32_t j = j0 + j4;
      if (first == 0) myers_cols4_z<W, UNIFORM, 0>(last, codes, ncols, Pv, Mv, bs, best, peq, nb, sbit, j, T);
      if (W > 1 && first == 1)
        myers_cols4_z<W, UNIFORM, (W > 1 ? 1 : 0)>(last, codes, ncols, Pv, Mv, bs, best, peq, nb, sbit, j, T);
      if (W > 2 && first == 2)
        myers_cols4_z<W, UNIFORM, (W > 2 ? 2 : 0)>(last, codes, ncols, Pv, Mv, bs, best, peq, nb, sbit, j, T);
      if (W > 3 && first == 3)
        myers_cols4_z<W, UNIFORM, (W > 3 ? 3 : 0)>(last, codes, ncols, Pv, Mv, bs, best, peq, nb, sbit, j, T);
    }
  }
  return best;
}

// ---------------------------------------------------------------------------------------------
// The SW pre-filter of src/index.rs:402-406 for reads of 254 bases and more.
//
// For shorter reads the test `score >= L - 2k` is implied by `min_edit_distance <= k` (SURVEY §8 a-7):
// ssw_align's 8-bit kernel is textbook local SW.  Once the true SW score reaches 254 the 8-bit kernel
// overflows (ssw.c:271,302) and ssw_align re-runs sw_sse2_word (ssw.c:789-792, :354-530), which is NOT
// textbook SW: with gap open == gap extend (the reference passes 1, 1: src/index.rs:402) its lazy-F loop
// (ssw.c:444-455) always leaves after its first vector — after `vH = max(vH, vF)` the exit test
// `vF - gapE > vH - gapO` can never hold.  In scalar terms (query row q sits in SIMD lane q / segLen at
// position q % segLen, segLen = ceil(L / 8)): the vertical-gap value F restarts from 0 at every lane
// boundary row (q % segLen == 0); the F that arrives there from the row above only lifts the STORED H of
// that one row (used as the next column's diagonal and for the maximum), while E and the F of the rows
// below continue from the uncorrected H.  Scores come out up to a few points lower than SW, which can
// push a candidate with edit distance <= k under the threshold.  The functions below reproduce the kernel
// cell for cell (16-bit saturation never triggers: scores < 32767).
//
// Codes: 0..3 = A,C,G,T, 4 = anything else; 4 matches 4 (ssw/src/lib.rs:11-16,93-99).
// ---------------------------------------------------------------------------------------------
MTSV_HD int32_t ssw_sub(uint32_t rc, uint32_t tc) { return rc == tc ? 1 : -1; }

// One column of sw_sse2_word over rows [q_lo, q_hi]; H/E are indexed through `slot(q)`.  diag_in = stored H of
// row q_lo - 1 in the previous column (0 above the matrix / outside a band).  Returns the column maximum.
template <typename ReadF, typename SlotF>
MTSV_HD uint32_t ssw_word_column(uint32_t q_lo, uint32_t q_hi, uint32_t seg_len, uint32_t tc, ReadF rcode,
                                 uint16_t* H, uint16_t* E, SlotF slot, uint32_t diag_in) {
  uint32_t colmax = 0, F = 0, diag = diag_in;
  for (uint32_t q = q_lo; q <= q_hi; ++q) {
    const uint32_t sl = slot(q);
    const uint32_t e = E[sl];
    int32_t h = (int32_t)diag + ssw_sub(rcode(q), tc);  // _mm_adds_epi16(vH, profile)
    if (h < (int32_t)e) h = (int32_t)e;                  // e >= 0, so h >= 0 from here on
    uint32_t carry = 0;
    if (q % seg_len == 0) {  // first row of a SIMD lane: F restarts; the carry only corrects the stored H
      carry = q == q_lo ? 0 : F;
      F = 0;
    }
    if ((uint32_t)h < F) h = (int32_t)F;
    const uint32_t t = h > 0 ? (uint32_t)h - 1 : 0;  // _mm_subs_epu16(vH, vGapO)
    const uint32_t e1 = e > 0 ? e - 1 : 0;
    E[sl] = (uint16_t)(e1 > t ? e1 : t);
    const uint32_t f1 = F > 0 ? F - 1 : 0;
    F = f1 > t ? f1 : t;
    uint32_t hst = (uint32_t)h > carry ? (uint32_t)h : carry;  // lazy-F, j == 0 of every lane only
    diag = H[sl];
    H[sl] = (uint16_t)hst;
    if (hst > colmax) colmax = hst;
  }
  return colmax;
}

// Lower bound of the sw_sse2_word score from the cells within `w` of the diagonal text_col - row == d0
// (cells outside count as 0; every operation of the kernel is monotone, so restricting it can only lower the
// result).  Stops as soon as `thr` is reached.  H/E: 2 x kSswBandCap entries, used circularly.
constexpr uint32_t kSswBandCap = 256;
constexpr uint32_t kSswBandMaxW = kSswBandCap / 2 - 1;  // rows q_lo-1 .. q_hi of a column must fit the ring
template <typename ReadF, typename TextF>
MTSV_HD uint32_t ssw_word_band(uint32_t L, uint32_t T, ReadF rcode, TextF tcode, int64_t d0, uint32_t w,
                               uint32_t thr, uint16_t* H, uint16_t* E) {
  const uint32_t seg_len = (L + 7) / 8;
  for (uint32_t x = 0; x < kSswBandCap; ++x) H[x] = E[x] = 0;
  int64_t i_lo = d0 - (int64_t)w, i_hi = d0 + (int64_t)(L - 1) + (int64_t)w;
  if (i_lo < 0) i_lo = 0;
  if (i_hi > (int64_t)T - 1) i_hi = (int64_t)T - 1;
  uint32_t best = 0;
  auto slot = [](uint32_t q) { return q & (kSswBandCap - 1); };
  for (int64_t i = i_lo; i <= i_hi; ++i) {
    int64_t ql = i - d0 - (int64_t)w, qh = i - d0 + (int64_t)w;
    if (qh < 0 || ql > (int64_t)L - 1) continue;
    if (qh <= (int64_t)L - 1 && i > i_lo) H[slot((uint32_t)qh)] = E[slot((uint32_t)qh)] = 0;  // row enters the band
    if (ql < 0) ql = 0;
    if (qh > (int64_t)L - 1) qh = (int64_t)L - 1;
    uint32_t diag_in = 0;
    if (ql > 0 && i > i_lo) diag_in = H[slot((uint32_t)ql - 1)];  // top row of the previous column's band
    uint32_t m = ssw_word_column((uint32_t)ql, (uint32_t)qh, seg_len, tcode((uint32_t)i), rcode, H, E, slot, diag_in);
    if (m > best) best = m;
    if (best >= thr) return best;
  }
  return best;
}

// The reference's decision at src/index.rs:406 from the full matrices: textbook SW (what the 8-bit kernel
// returns while it does not overflow) and the 16-bit kernel, in one pass.  H/E/H2/E2: L entries each.
template <typename ReadF, typename TextF>
MTSV_HD bool ssw_accepts_full(uint32_t L, uint32_t T, ReadF rcode, TextF tcode, uint32_t thr, uint16_t* H,
                              uint16_t* E, uint16_t* H2, uint16_t* E2, uint32_t* word_out = nullptr,
                              uint32_t* exact_out = nullptr) {  // (scores are only complete when thr is unreachable)
  const uint32_t seg_len = (L + 7) / 8;
  for (uint32_t q = 0; q < L; ++q) H[q] = E[q] = H2[q] = E2[q] = 0;
  uint32_t word_best = 0, exact_best = 0;
  auto slot = [](uint32_t q) { return q; };
  for (uint32_t i = 0; i < T; ++i) {
    const uint32_t tc = tcode(i);
    uint32_t m = ssw_word_column(0, L - 1, seg_len, tc, rcode, H, E, slot, 0);
    if (m > word_best) word_best = m;
    if (word_best >= thr) return true;  // (and if the 8-bit kernel did not overflow, SW itself is >= this)
    // textbook SW, linear gap 1 (== sw_sse2_byte below its overflow point)
    uint32_t diag = 0, F = 0;
    for (uint32_t q = 0; q < L; ++q) {
      int32_t h = (int32_t)diag + ssw_sub(rcode(q), tc);
      const uint32_t e = E2[q];
      if (h < (int32_t)e) h = (int32_t)e;
      if ((uint32_t)h < F) h = (int32_t)F;
      const uint32_t t = h > 0 ? (uint32_t)h - 1 : 0;
      const uint32_t e1 = e > 0 ? e - 1 : 0;
      E2[q] = (uint16_t)(e1 > t ? e1 : t);
      const uint32_t f1 = F > 0 ? F - 1 : 0;
      F = f1 > t ? f1 : t;
      diag = H2[q];
      H2[q] = (uint16_t)h;
      if ((uint32_t)h > exact_best) exact_best = (uint32_t)h;
    }
  }
  // ssw_align: the 8-bit result unless it overflowed (max + bias >= 255, bias = 1), then the 16-bit kernel's
  if (word_out) *word_out = word_best;
  if (exact_out) *exact_out = exact_best;
  const uint32_t score = exact_best >= 254 ? word_best : exact_best;
  return score >= thr;
}

// read code of row q from the bit planes: 0..3, N -> 4
MTSV_HD uint32_t plane_code(const ReadWord* qw, uint32_t q) {
  const ReadWord& w = qw[q >> 6];
  const uint32_t b = q & 63;
  if ((w.nn >> b) & 1) return 4;
  return (uint32_t)((w.lo >> b) & 1) | ((uint32_t)((w.hi >> b) & 1) << 1);
}
// reference byte -> dna5 code (ssw/src/lib.rs:93-99)
MTSV_HD uint32_t dna5_code(uint8_t b) {
  uint32_t c = upper_acgtn_code(b);
  return c < 4 ? c : 4;
}

// ---------------------------------------------------------------------------------------------
// stage: selection (one item per query) — the verification loop control of src/index.rs:375-431
// over already computed edit distances, in rank order.
// ---------------------------------------------------------------------------------------------
struct HitRec {  // mtsvgpu_hit layout
  uint32_t tax_id, gi;
  uint64_t offset;
  uint32_t edit, reserved;
};
static_assert(sizeof(HitRec) == 24, "HitRec must match mtsvgpu_hit");

MTSV_HD uint32_t select_item(const BinsView& bv, const Params& p, const CandRec* cand,
                             const uint32_t* edits, uint32_t n_cand, uint32_t k, HitRec* out) {
  uint32_t n_out = 0;
  for (uint32_t c = 0; c < n_cand; ++c) {
    if (p.max_candidates >= 0 && (uint64_t)c >= (uint64_t)p.max_candidates) break;  // :385-389
    // (the edit test comes first here: a candidate that fails :406/:410 never changes the loop's
    //  state, so testing it before the "TaxID already matched" scan of :393-396 gives the same hits)
    uint32_t e = edits[c];
    if (e == kNoEdit || e > k) continue;  // :406,:410
    uint32_t bin = cand[c].bin;
    uint32_t tax = ldg(&bv.tax[bin]);
    bool seen = false;
    for (uint32_t m = 0; m < n_out; ++m) seen |= out[m].tax_id == tax;  // :393-396
    if (seen) continue;
    HitRec h;
    h.tax_id = tax;
    h.gi = ldg(&bv.gi[bin]);
    uint32_t bs = ldg(&bv.start[bin]);
    h.offset = cand[c].start >= bs ? cand[c].start - bs : 0;  // saturating_sub, :416
    h.edit = e;
    h.reserved = 0;
    out[n_out++] = h;
    if (p.max_assignments >= 0 && (uint64_t)n_out >= (uint64_t)p.max_assignments) break;  // :421-425
  }
  return n_out;
}

// ---------------------------------------------------------------------------------------------
// host-side schedule (no device code; here so that tests/emul can check it)
// ---------------------------------------------------------------------------------------------
// Read boundaries of slices of at most `step` reads.  Without the ramp: equal slices of `step` reads.  With the
// ramp (host input): the slices are uploaded one by one while earlier ones compute, so the call lasts about
// (upload of everything) + (upload of the first slice) + (compute of the last slice): the first slices grow
// geometrically from step/16 and the last ones shrink to step/8.
inline std::vector<uint64_t> sub_batch_bounds(uint64_t n_reads, uint64_t step, bool ramp) {
  std::vector<uint64_t> b{0};
  if (step == 0) step = 1;
  std::vector<uint64_t> up, down;
  if (ramp && step >= 1024) {
    up = {step / 16, step / 8, step / 4, step / 2};
    down = {step / 2, step / 4, step / 8};
  }
  uint64_t edge = 0;
  for (uint64_t x : up) edge += x;
  for (uint64_t x : down) edge += x;
  uint64_t r = 0;
  if (!up.empty() && n_reads > edge + step / 2) {
    for (uint64_t x : up) b.push_back(r += x);
    const uint64_t middle = n_reads - edge, n_full = (middle + step - 1) / step;
    for (uint64_t i = 1; i <= n_full; ++i) b.push_back(r + middle * i / n_full);
    r += middle;
    for (uint64_t x : down) b.push_back(r += x);
  } else {
    for (uint64_t x : up) {  // short batch: geometric slices until it is used up
      if (r + x >= n_reads) break;
      b.push_back(r += x);
    }
    while (r < n_reads) b.push_back(r = std::min(n_reads, r + step));
  }
  return b;
}

// The slices of one batch call, for the uploader of host input and the compute lanes alike.  step = reads per slice,
// 0 for the default of the input's kind.  Host input: the ramped slices above.  Device-resident input: k = ceil(n /
// step) slices of equal size; with two lanes an even number, so that both lanes get the same share, and a batch that
// fits one slice is still cut in two when it is large enough (kSplitMinReads: +3 % at 2.5 M reads; at 1.25 M reads
// the halves gain 3 % on an idle host and lose as much with eight ranks' threads competing for it).  Bound i is
// min(n, i * ceil(n / k)), so the last slice can be empty.
constexpr uint64_t kDefaultStepDevice = 1ull << 22, kDefaultStepHost = 1ull << 20, kSplitMinReads = 1ull << 21;
inline std::vector<uint64_t> slice_bounds(uint64_t n_reads, uint64_t step, bool host_input, bool two_lanes) {
  if (step == 0) step = host_input ? kDefaultStepHost : kDefaultStepDevice;
  if (host_input) return sub_batch_bounds(n_reads, step, true);
  uint64_t k = (n_reads + step - 1) / step;
  if (two_lanes && ((k >= 2 && (k & 1)) || (k == 1 && n_reads >= kSplitMinReads))) ++k;
  const uint64_t stride = k ? (n_reads + k - 1) / k : step;
  std::vector<uint64_t> b{0};
  for (uint64_t i = 1; i <= k; ++i) b.push_back(std::min(n_reads, i * stride));
  return b;
}

}  // namespace mtsv
