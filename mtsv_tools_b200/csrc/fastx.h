// FASTA / FASTQ records (bio::io::{fasta,fastq}) for mtsv-binner and mtsv-build: the one record grammar, and a block
// reader that hands out runs of whole records; gz or plain via zlib (src/binner.rs:21-33).
#pragma once
#include <ctype.h>
#include <fcntl.h>
#include <stdint.h>
#include <string.h>
#include <sys/stat.h>
#include <unistd.h>
#include <zlib.h>

#include <algorithm>
#include <string>

// lines of a text span; '\r' before '\n' is dropped; `terminated` tells whether the line ended in a newline
// (the last line of a span may be cut by the span's end)
struct Lines {
  const char *p, *end;
  bool terminated = true;
  bool next(const char** b, const char** e) {
    if (p >= end) return false;
    const char* nl = (const char*)memchr(p, '\n', (size_t)(end - p));
    terminated = nl != nullptr;
    *b = p;
    *e = nl ? nl : end;
    p = nl ? nl + 1 : end;
    if (*e > *b && (*e)[-1] == '\r') --*e;
    return true;
  }
};

struct FastxRecord {
  const char *id, *id_end;  // the header up to the first whitespace, without its '>' / '@'
  const char *seq, *seq_end;  // the sequence lines as they stand in the text, newlines included (Lines splits them)
  uint64_t seq_lines;         // with one line, the bases are [seq, seq + len)
  uint64_t len;               // bases
};

// Reads the record at `ln` and moves `ln` past it (1).  A record starts with '>' (FASTA) or '@' (FASTQ); blank lines
// before it are skipped; its sequence may span lines and ends at the next '>' line (FASTA) or at a '+' line, which
// in FASTQ is followed by as many quality characters as there are bases.  0: the text ends before the record is
// complete, or holds no further record; -1: malformed record.  `eof`: the text is the rest of the file, so a last
// line without newline is whole and a FASTA record needs no following header to be complete.
inline int next_record(Lines& ln, bool fastq, bool eof, FastxRecord* r) {
  const char *b, *e;
  do {  // blank lines between records
    if (!ln.next(&b, &e) || (!ln.terminated && !eof)) return 0;
  } while (e == b);
  if (*b != (fastq ? '@' : '>')) return -1;
  r->id = r->id_end = b + 1;
  while (r->id_end < e && !isspace((unsigned char)*r->id_end)) ++r->id_end;
  r->seq = r->seq_end = ln.p;
  r->seq_lines = r->len = 0;
  for (;;) {  // sequence lines
    if (ln.p >= ln.end) return !eof ? 0 : fastq ? -1 : 1;
    if (!fastq && *ln.p == '>') return 1;
    ln.next(&b, &e);
    if (!ln.terminated && !eof) return 0;
    if (fastq && e > b && *b == '+') break;
    r->seq_end = ln.p;
    ++r->seq_lines;
    r->len += (uint64_t)(e - b);
  }
  uint64_t q = 0;
  while (q < r->len) {  // quality lines
    if (!ln.next(&b, &e)) return eof ? -1 : 0;
    if (!ln.terminated && !eof) return 0;
    q += (uint64_t)(e - b);
  }
  return q == r->len ? 1 : -1;
}

// Reads a FASTA / FASTQ file, gz or plain, in large blocks of whole records.
class FastxBlocks {
 public:
  FastxBlocks(const char* path, bool fastq) : fastq_(fastq) {
    gz_ = gzopen(path, "rb");  // reads uncompressed files too (magic 1f 8b sniffing)
    if (!gz_) return;
    gzbuffer(gz_, 1 << 20);
    // an uncompressed file is read with plain read(2): no pass through zlib's copy-through mode
    struct stat st;
    if (stat(path, &st) == 0 && S_ISREG(st.st_mode) && gzdirect(gz_)) {
      fd_ = open(path, O_RDONLY);
#ifdef POSIX_FADV_SEQUENTIAL
      if (fd_ >= 0) posix_fadvise(fd_, 0, 0, POSIX_FADV_SEQUENTIAL);
#endif
    }
  }
  ~FastxBlocks() {
    if (gz_) gzclose(gz_);
    if (fd_ >= 0) close(fd_);
  }
  FastxBlocks(const FastxBlocks&) = delete;
  FastxBlocks& operator=(const FastxBlocks&) = delete;
  bool ok() const { return gz_ != nullptr; }
  // a malformed record follows the block last handed out (the next call reports it)
  bool malformed_next() const { return malformed_; }

  // 1: *text is the next run of whole records, *n of them; 0: end of input; -1: malformed record (the good records
  // before it come first, as a block of their own); -2: read error.  Each block is read straight into the string
  // handed out: only the cut-off tail (the beginning of the record the block edge fell into) is copied, into the
  // string *text held before.
  int next(std::string* text, uint64_t* n) {
    for (;;) {
      if (malformed_) return -1;
      if (!eof_) {
        // a read that completed no record is followed by one at least as large as the carry: a record of any
        // length is scanned a bounded number of times
        const size_t have = carry_.size(), want = std::max(kBlockBytes, have);
        carry_.resize(have + want);
        size_t filled = 0;
        while (filled < want) {  // (short reads happen on pipes and at gzip member boundaries)
          const size_t ask = std::min(want - filled, (size_t)1 << 30);
          const long got = fd_ >= 0 ? (long)read(fd_, &carry_[have + filled], ask)
                                    : (long)gzread(gz_, &carry_[have + filled], (unsigned)ask);
          if (got < 0) return -2;
          if (got == 0) {
            eof_ = true;
            break;
          }
          filled += (size_t)got;
        }
        carry_.resize(have + filled);
      }
      Lines ln{carry_.data(), carry_.data() + carry_.size()};
      FastxRecord r;
      const char* cut = ln.p;
      uint64_t k = 0;
      int rc;
      while ((rc = next_record(ln, fastq_, eof_, &r)) == 1) {
        cut = ln.p;
        ++k;
      }
      malformed_ = rc < 0;
      if (k == 0) {
        if (malformed_) return -1;
        if (eof_) return 0;
        continue;
      }
      const size_t used = (size_t)(cut - carry_.data());
      text->swap(carry_);  // (the caller's previous block becomes the next carry's buffer)
      carry_.assign(*text, used, std::string::npos);
      text->resize(used);
      *n = k;
      return 1;
    }
  }

 private:
  static constexpr size_t kBlockBytes = 4u << 20;
  gzFile gz_ = nullptr;
  int fd_ = -1;
  bool fastq_, eof_ = false, malformed_ = false;
  std::string carry_;
};
