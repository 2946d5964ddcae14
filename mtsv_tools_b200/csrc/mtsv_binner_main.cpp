// mtsv-binner (B200) — host driver with the reference's command line above the C ABI.
//
// Mirrors src/bin/mtsv-binner.rs:21-331 (flags, defaults, validation, exit codes, resume-by-results
// :347-411) and the host part of src/binner.rs (gz sniffing :21-33, FASTA/FASTQ records via their
// id = header up to the first whitespace, --read-offset skipping :169-199, write_assignments :310-379).
// The per-read work (normalisation, both strands, matching_tax_ids, and for the default results format the
// per-TaxID minimum edit) is one mtsvgpu_assign_batch_packed call per batch of reads (mtsvgpu_bin_batch_packed
// for --output-format long).  The reference's host is Rust; no Rust toolchain exists in this image, so the
// driver is C++ over the same C ABI a Rust build.rs would link (INTEGRATION.md).
//
// Host pipeline (the reference: cue's reader -> N workers -> single writer, src/binner.rs:149-217):
//   reader thread     inflates / reads the file in large blocks of whole records (fastx.h)
//   --threads workers parse the records of a block (id, sequence) and pack each sequence straight into the
//                     bit planes the device consumes (mtsvgpu_pack_read: no intermediate copy of the bases);
//                     the same pool later formats result lines
//   one thread per GPU (--gpus) gathers parsed blocks into batches in page-locked memory, calls the library,
//                     keeps the results; batches go to the GPUs round-robin
//   writer thread     appends the formatted batches in input order (so results are deterministic and
//                     resume-by-results is exact)
//
// Exit codes (SURVEY §5): 0 ok, 2 query error, 3 no results path, 4 resume error, 11 write error,
// 12 read-parse error.
#include <ctype.h>
#include <errno.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <sys/stat.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <deque>
#include <functional>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <tuple>
#include <unordered_set>
#include <vector>

#include "../../include/mtsv_b200.h"
#include "fastx.h"

namespace {

bool g_verbose = false;
void logf(const char* level, const char* fmt, ...) {
  if (!g_verbose && strcmp(level, "DEBUG") == 0) return;
  va_list ap;
  va_start(ap, fmt);
  fprintf(stderr, "[%s mtsv_binner] ", level);
  vfprintf(stderr, fmt, ap);
  fputc('\n', stderr);
  va_end(ap);
}

// ---- write_assignments (src/binner.rs:310-379) ----
inline void put_u64(std::string* out, uint64_t v) {
  char tmp[24];
  int n = 0;
  do {
    tmp[n++] = (char)('0' + v % 10);
    v /= 10;
  } while (v);
  while (n) out->push_back(tmp[--n]);
}

// one result line, or nothing when the read has no assignment (:316-318).  Default format (:330-352): the
// library's merged records are already one per TaxID with its minimum edit, by TaxID (BTreeMap order).
void format_taxhits(const char* id, size_t id_len, const mtsvgpu_taxhit* recs, uint64_t n, std::string* out) {
  if (n == 0) return;
  out->append(id, id_len);
  out->push_back(':');
  for (uint64_t i = 0; i < n; ++i) {
    if (i) out->push_back(',');
    put_u64(out, recs[i].tax_id);
    out->push_back('=');
    put_u64(out, recs[i].edit);
  }
  out->push_back('\n');
}

// long format (:354-376): minimum edit per (TaxID, GI, offset), in that order
void format_hits_long(const char* id, size_t id_len, const mtsvgpu_hit* hits, uint64_t n, std::string* out) {
  if (n == 0) return;
  out->append(id, id_len);
  out->push_back(':');
  constexpr uint64_t kSmall = 16;
  const mtsvgpu_hit* order[kSmall];
  std::vector<const mtsvgpu_hit*> big;
  const mtsvgpu_hit** v = order;
  if (n > kSmall) {
    big.resize(n);
    v = big.data();
  }
  for (uint64_t i = 0; i < n; ++i) v[i] = hits + i;
  auto less = [](const mtsvgpu_hit* a, const mtsvgpu_hit* b) {
    if (a->tax_id != b->tax_id) return a->tax_id < b->tax_id;
    if (a->gi != b->gi) return a->gi < b->gi;
    if (a->offset != b->offset) return a->offset < b->offset;
    return a->edit < b->edit;
  };
  if (n > 1) std::sort(v, v + n, less);
  bool first = true;
  for (uint64_t i = 0; i < n; ++i) {
    if (i) {
      const mtsvgpu_hit *a = v[i - 1], *b = v[i];
      const bool same = a->tax_id == b->tax_id && a->gi == b->gi && a->offset == b->offset;
      if (same) continue;  // the smaller edit of the key came first
    }
    if (!first) out->push_back(',');
    first = false;
    put_u64(out, v[i]->tax_id);
    out->push_back('-');
    put_u64(out, v[i]->gi);
    out->push_back('-');
    put_u64(out, v[i]->offset);
    out->push_back('=');
    put_u64(out, v[i]->edit);
  }
  out->push_back('\n');
}

// ---- resume (src/bin/mtsv-binner.rs:347-411) ----
bool read_ids_from_results(const char* path, std::unordered_set<std::string>* ids, std::string* err) {
  FILE* f = fopen(path, "r");
  if (!f) {
    *err = strerror(errno);
    return false;
  }
  char* line = nullptr;
  size_t cap = 0;
  ssize_t n;
  while ((n = getline(&line, &cap, f)) >= 0) {
    std::string s(line, (size_t)n);
    while (!s.empty() && isspace((unsigned char)s.back())) s.pop_back();
    size_t b = 0;
    while (b < s.size() && isspace((unsigned char)s[b])) ++b;
    if (b == s.size()) continue;
    size_t colon = s.rfind(':');  // rsplitn(2, ':')
    if (colon == std::string::npos || colon == 0) {
      *err = "Missing read id";
      free(line);
      fclose(f);
      return false;
    }
    ids->insert(s.substr(0, colon));
  }
  free(line);
  fclose(f);
  return true;
}

bool resume_offset(const char* results, const char* input, bool fastq, uint64_t* offset, std::string* err) {
  struct stat sb;
  if (stat(results, &sb) != 0) {
    *offset = 0;
    return true;
  }
  std::unordered_set<std::string> ids;
  if (!read_ids_from_results(results, &ids, err)) return false;
  FastxBlocks in(input, fastq);
  if (!in.ok()) {
    *err = "cannot open input";
    return false;
  }
  std::string text, id;
  uint64_t n, idx = 0, last = 0;
  bool any = false;
  int rc;
  while ((rc = in.next(&text, &n)) == 1) {
    Lines ln{text.data(), text.data() + text.size()};
    FastxRecord r;
    while (next_record(ln, fastq, true, &r) == 1) {
      if (ids.count(id.assign(r.id, r.id_end))) {
        last = idx;
        any = true;
      }
      ++idx;
    }
  }
  if (rc < 0) {
    *err = rc == -1 ? "parse error while scanning input" : "cannot read input";
    return false;
  }
  *offset = any ? last + 1 : 0;
  return true;
}

void usage() {
  fprintf(stderr,
          "mtsv-binner (B200)\n"
          "USAGE: mtsv-binner (--fasta <FASTA> | --fastq <FASTQ>) --index <INDEX> --results <RESULTS_PATH> [FLAGS]\n"
          "  -i, --index <INDEX>            Path to MG-index file.\n"
          "  -m, --results <RESULTS_PATH>   Path to write results file.\n"
          "      --fasta / --fastq <PATH>   Path to FASTA / FASTQ reads (gz detected automatically).\n"
          "  -e, --edit-rate <f>            [default: 0.13]\n"
          "      --seed-size <n>            [default: 18]\n"
          "      --seed-interval <n>        [default: 15]\n"
          "      --min-seed <f>             [default: 0.015]\n"
          "      --max-hits <n>             [default: 2000]\n"
          "      --tune-max-hits <n>        [default: 200]\n"
          "      --max-assignments <n>      --max-candidates <n>\n"
          "      --read-offset <n>          [default: 0]\n"
          "      --output-format default|long\n"
          "      --force-overwrite          -v\n"
          "  -t, --threads <n>              parser / formatter threads [default: all cores]\n"
          "      --gpu <id>                 first CUDA device [default: 0]\n"
          "      --gpus <n>                 number of CUDA devices; batches go round-robin [default: 1]\n"
          "      --batch-reads <n>          reads per library call [default: 524288]\n"
          "      --strict-limits            exit 2 when a read exceeded a limit of this implementation (reads longer\n"
          "                                 than 4096 bases get no assignments; default: warn and go on)\n");
}


// ------------------------------------------------------------------------------------------
// pipeline
// ------------------------------------------------------------------------------------------
struct TextBlock {  // whole records, as they stand in the file
  uint64_t seq = 0;
  std::string text;
  uint64_t n_records = 0;
};

struct ParsedBlock {
  uint32_t n = 0;
  std::vector<uint8_t> packed;    // records of core.cuh "packed reads"
  std::vector<uint32_t> len;      // bases per read
  std::vector<uint32_t> id_end;   // end of each id inside `ids`
  std::string ids;
  bool bad = false;
};

struct Batch {
  uint64_t seq = 0;
  std::vector<std::unique_ptr<ParsedBlock>> parts;
  uint64_t n_reads = 0;
  std::vector<mtsvgpu_hit> hits;        // long format: the Hit records
  std::vector<mtsvgpu_taxhit> taxhits;  // default format: merged (TaxID, edit) records
  std::vector<uint64_t> hit_off;
  std::vector<std::string> text;  // one per part, filled by the formatter tasks
  std::atomic<uint32_t> pending{0};
  uint64_t lines = 0;
};

class Pool {  // fixed set of workers running queued tasks
 public:
  explicit Pool(int n) {
    for (int i = 0; i < n; ++i) th_.emplace_back([this] { run(); });
  }
  ~Pool() {
    {
      std::lock_guard<std::mutex> lk(mu_);
      stop_ = true;
    }
    cv_.notify_all();
    for (auto& t : th_) t.join();
  }
  void submit(std::function<void()> f) {
    {
      std::lock_guard<std::mutex> lk(mu_);
      q_.push_back(std::move(f));
    }
    cv_.notify_one();
  }

 private:
  void run() {
    for (;;) {
      std::function<void()> f;
      {
        std::unique_lock<std::mutex> lk(mu_);
        cv_.wait(lk, [this] { return stop_ || !q_.empty(); });
        if (q_.empty()) return;
        f = std::move(q_.front());
        q_.pop_front();
      }
      f();
    }
  }
  std::mutex mu_;
  std::condition_variable cv_;
  std::deque<std::function<void()>> q_;
  std::vector<std::thread> th_;
  bool stop_ = false;
};

struct Shared {
  std::mutex mu;
  std::condition_variable cv;
  int exit_code = 0;
  std::string error;
  void fail(int code, const std::string& msg) {
    std::lock_guard<std::mutex> lk(mu);
    if (exit_code == 0) {
      exit_code = code;
      error = msg;
    }
    cv.notify_all();
  }
  bool failed() {
    std::lock_guard<std::mutex> lk(mu);
    return exit_code != 0;
  }
};

// parse + pack one block of whole records, all but the first `skip` (a pool task)
void parse_block(const TextBlock& tb, bool fastq, uint64_t skip, ParsedBlock* out) {
  out->n = 0;
  out->len.reserve(tb.n_records - skip);
  out->id_end.reserve(tb.n_records - skip);
  out->packed.reserve(tb.text.size() / 4);
  Lines ln{tb.text.data(), tb.text.data() + tb.text.size()};
  FastxRecord r;
  std::string multi;
  for (uint64_t i = 0; next_record(ln, fastq, true, &r) == 1; ++i) {
    if (i < skip) continue;
    if (r.len > 0xfffffff0ull) {
      out->bad = true;
      return;
    }
    out->ids.append(r.id, r.id_end);
    out->id_end.push_back((uint32_t)out->ids.size());
    const char* seq = r.seq;
    if (r.seq_lines > 1) {  // only a multi-line sequence is copied
      multi.clear();
      Lines sl{r.seq, r.seq_end};
      const char *b, *e;
      while (sl.next(&b, &e)) multi.append(b, e);
      seq = multi.data();
    }
    const size_t at = out->packed.size();
    out->packed.resize(at + 3 * ((r.len + 7) >> 3));
    if (r.len) mtsvgpu_pack_read((const uint8_t*)seq, (uint32_t)r.len, out->packed.data() + at);
    out->len.push_back((uint32_t)r.len);
    ++out->n;
  }
}

}  // namespace

int main(int argc, char** argv) {
  const char *fasta = nullptr, *fastq = nullptr, *index = nullptr, *results = nullptr;
  mtsvgpu_params p{0.13, 18, 15, 0.015, 2000, 200, -1, -1, 2, 0};
  uint64_t read_offset = 0, batch_reads = 1u << 19;
  bool long_fmt = false, force = false, dump_reads = false, strict_limits = false;
  int device = 0, n_gpus = 1, n_threads = 0;
  auto need = [&](int& i) -> const char* {
    if (i + 1 >= argc) {
      fprintf(stderr, "error: %s requires a value\n", argv[i]);
      exit(1);
    }
    return argv[++i];
  };
  for (int i = 1; i < argc; ++i) {
    std::string a = argv[i];
    if (a == "--fasta" || a == "-fa" || a == "-f") fasta = need(i);
    else if (a == "--fastq" || a == "-fq") fastq = need(i);
    else if (a == "--index" || a == "-i") index = need(i);
    else if (a == "--results" || a == "-m") results = need(i);
    else if (a == "--threads" || a == "-t") n_threads = atoi(need(i));
    else if (a == "--edit-rate" || a == "-e") p.edit_rate = atof(need(i));
    else if (a == "--seed-size") p.seed_size = (uint32_t)strtoul(need(i), nullptr, 10);
    else if (a == "--seed-interval") p.seed_gap = (uint32_t)strtoul(need(i), nullptr, 10);
    else if (a == "--min-seed") p.min_seed = atof(need(i));
    else if (a == "--max-hits") p.max_hits = strtoull(need(i), nullptr, 10);
    else if (a == "--tune-max-hits") p.tune_max_hits = strtoull(need(i), nullptr, 10);
    else if (a == "--max-assignments") p.max_assignments = strtoll(need(i), nullptr, 10);
    else if (a == "--max-candidates") p.max_candidates = strtoll(need(i), nullptr, 10);
    else if (a == "--read-offset") read_offset = strtoull(need(i), nullptr, 10);
    else if (a == "--output-format") long_fmt = std::string(need(i)) == "long";
    else if (a == "--force-overwrite") force = true;
    else if (a == "-v") g_verbose = true;
    else if (a == "--gpu") device = atoi(need(i));
    else if (a == "--gpus") n_gpus = atoi(need(i));
    else if (a == "--strict-limits") strict_limits = true;
    else if (a == "--dump-reads") dump_reads = true;  // test hook: parse the input, print "id<TAB>seq", no GPU
    else if (a == "--dump-reads-mt") dump_reads = true, n_threads = n_threads ? n_threads : -1;  // same through the pipeline's scanner + parser
    else if (a == "--batch-reads") batch_reads = strtoull(need(i), nullptr, 10);
    else if (a == "-h" || a == "--help") {
      usage();
      return 0;
    } else {
      fprintf(stderr, "error: unknown argument %s\n", a.c_str());
      usage();
      return 1;
    }
  }
  const bool dump_mt = dump_reads && n_threads != 0;
  if (dump_reads && !dump_mt && (fasta || fastq)) {
    FastxBlocks in(fasta ? fasta : fastq, fastq != nullptr);
    if (!in.ok()) return 2;
    std::string text;
    uint64_t n, idx = 0;
    int rc;
    while ((rc = in.next(&text, &n)) == 1) {
      Lines ln{text.data(), text.data() + text.size()};
      FastxRecord r;
      while (next_record(ln, fastq != nullptr, true, &r) == 1) {
        if (idx++ < read_offset) continue;
        fwrite(r.id, 1, (size_t)(r.id_end - r.id), stdout);
        putchar('\t');
        Lines sl{r.seq, r.seq_end};
        const char *b, *e;
        while (sl.next(&b, &e)) fwrite(b, 1, (size_t)(e - b), stdout);
        putchar('\n');
      }
    }
    return rc < 0 ? 12 : 0;
  }
  if ((!fasta && !fastq) || (fasta && fastq) || (!index && !dump_mt)) {
    usage();
    return 1;
  }
  // validation as src/bin/mtsv-binner.rs:151,195 (the reference panics; exit code 101 there)
  if (p.edit_rate < 0.0 || p.edit_rate > 1.0) {
    logf("ERROR", "Edit tolerance proportion must be between 0 and 1, inclusive");
    return 101;
  }
  if (p.min_seed <= 0.0 || p.min_seed > 1.0) {
    logf("ERROR", "Min seed percent must be between 0 and 1");
    return 101;
  }
  if (p.seed_size < 16) logf("WARN", "Seed size may be small enough that it causes performance issues.");
  else if (p.seed_size > 24) logf("WARN", "Seed size may be large enough that significant results are ignored.");
  if (!results && !dump_mt) {
    logf("ERROR", "No results path provided!");
    return 3;  // :262-265
  }
  if (n_gpus < 1) n_gpus = 1;
  if (n_threads <= 0) n_threads = (int)std::max(1u, std::thread::hardware_concurrency());
  if (batch_reads == 0) batch_reads = 1;
  const char* input = fasta ? fasta : fastq;
  const bool is_fastq = fastq != nullptr;
  struct stat sb;
  const bool append = !dump_mt && !force && stat(results, &sb) == 0;
  uint64_t resume = 0;
  if (!force && !dump_mt) {
    std::string err;
    if (!resume_offset(results, input, is_fastq, &resume, &err)) {
      logf("ERROR", "Error computing resume offset: %s", err.c_str());
      return 4;  // :288-291
    }
    if (append) logf("INFO", "Existing results detected at %s; resuming after read offset %llu", results,
                     (unsigned long long)resume);
  }
  read_offset += resume;

  FILE* out = dump_mt ? stdout : fopen(results, append ? "a" : "w");  // src/binner.rs:54-61
  if (!out) {
    logf("ERROR", "Error running query: cannot open %s: %s", results, strerror(errno));
    return 2;
  }
  FastxBlocks blocks(input, is_fastq);  // src/binner.rs:21-33
  if (!blocks.ok()) {
    logf("ERROR", "Error running query: cannot open %s", input);
    if (!dump_mt) fclose(out);
    return 2;
  }
  std::vector<mtsvgpu_index*> handles((size_t)n_gpus, nullptr);
  if (!dump_mt) {
    logf("INFO", "Deserializing candidate filter ...");
    std::vector<std::thread> openers;
    std::vector<std::string> errs((size_t)n_gpus);
    for (int g = 0; g < n_gpus; ++g)
      openers.emplace_back([&, g] {
        if (mtsvgpu_index_open(index, device + g, nullptr, &handles[(size_t)g]) != 0) {
          errs[(size_t)g] = mtsvgpu_last_error();
          return;
        }
        // a first small batch brings in what a fresh process pays once (kernel images, workspaces, page-locked
        // result buffers) while the other devices and the reader start up; its results are discarded
        std::vector<uint8_t> wseq(256 * 150);
        std::vector<uint64_t> woff(257);
        uint32_t x = 12345u + (uint32_t)g;
        for (auto& c : wseq) c = (uint8_t)"ACGT"[(x = x * 1664525u + 1013904223u) >> 30];
        for (size_t i = 0; i <= 256; ++i) woff[i] = i * 150;
        const uint64_t* wo = nullptr;
        uint64_t wn = 0;
        if (long_fmt) {
          const mtsvgpu_hit* wh = nullptr;
          (void)mtsvgpu_bin_batch_pinned(handles[(size_t)g], wseq.data(), woff.data(), 256, &p, &wh, &wo, &wn);
        } else {
          const mtsvgpu_taxhit* wt = nullptr;
          (void)mtsvgpu_assign_batch_pinned(handles[(size_t)g], wseq.data(), woff.data(), 256, &p, &wt, &wo, &wn);
        }
      });
    for (auto& t : openers) t.join();
    for (int g = 0; g < n_gpus; ++g)
      if (!handles[(size_t)g]) {
        logf("ERROR", "Error running query: %s", errs[(size_t)g].c_str());
        for (auto h : handles) mtsvgpu_index_close(h);
        fclose(out);
        return 2;
      }
  }
  logf("INFO", "Beginning queries.");
  auto t0 = std::chrono::steady_clock::now();

  Shared sh;
  // a failure anywhere in the pipeline is raised through `sh`, not through every stage's condition variable: waits
  // re-check it at short intervals
  auto wait_on = [](std::condition_variable& cv, std::unique_lock<std::mutex>& lk, auto pred) {
    while (!pred()) cv.wait_for(lk, std::chrono::milliseconds(50));
  };
  Pool pool(n_threads);
  // ---- reader -> parsed blocks (ordered by block sequence number) ----
  std::mutex pmu;
  std::condition_variable pcv;
  std::map<uint64_t, std::unique_ptr<ParsedBlock>> parsed;  // finished blocks waiting for their turn
  uint64_t blocks_issued = 0, blocks_taken = 0;
  bool reader_done = false;
  const uint64_t max_blocks_in_flight = (uint64_t)std::max(8, 4 * n_threads) + batch_reads / 8192;
  std::thread reader([&] {
    uint64_t records_seen = 0;  // complete records read so far (including skipped ones)
    while (!sh.failed()) {
      auto tb = std::make_shared<TextBlock>();
      const int rc = blocks.next(&tb->text, &tb->n_records);
      if (rc == 0) break;
      if (rc < 0 || blocks.malformed_next()) {  // (the records of a block that ends at a malformed one are not binned)
        std::string msg = "Unable to read from input file";
        if (rc != -2) msg += ": malformed record after " + std::to_string(records_seen) + " reads";
        sh.fail(12, msg);  // src/binner.rs:81-84
        break;
      }
      // .skip(read_offset) (src/binner.rs:176,199): whole blocks are dropped, the parser skips the first records of
      // a straddling block
      const uint64_t first = records_seen;
      records_seen += tb->n_records;
      if (records_seen <= read_offset) continue;
      const uint64_t skip = read_offset > first ? read_offset - first : 0;
      uint64_t seq;
      {
        std::unique_lock<std::mutex> lk(pmu);
        wait_on(pcv, lk, [&] { return blocks_issued - blocks_taken < max_blocks_in_flight || sh.failed(); });
        seq = blocks_issued++;
      }
      tb->seq = seq;
      pool.submit([&, tb, skip] {
        auto pb = std::make_unique<ParsedBlock>();
        if (!sh.failed()) parse_block(*tb, is_fastq, skip, pb.get());
        if (pb->bad) sh.fail(12, "Unable to read from input file: malformed record");
        std::lock_guard<std::mutex> lk(pmu);
        parsed[tb->seq] = std::move(pb);
        pcv.notify_all();
      });
    }
    std::lock_guard<std::mutex> lk(pmu);
    reader_done = true;
    pcv.notify_all();
  });

  // ---- batches: GPU threads take consecutive parsed blocks; formatted batches are written in order ----
  std::mutex bmu;  // serialises "take the next blocks" so that batches are consecutive runs of blocks
  uint64_t batch_seq = 0;
  std::mutex wmu;
  std::condition_variable wcv;
  std::map<uint64_t, std::shared_ptr<Batch>> done;  // formatted (or empty) batches by sequence number
  uint64_t batches_total = ~0ull;                   // known once the input is exhausted
  std::atomic<uint64_t> total_reads{0}, total_lines{0}, over_len{0}, over_hits{0};

  auto take_batch = [&]() -> std::shared_ptr<Batch> {
    std::lock_guard<std::mutex> blk(bmu);
    auto b = std::make_shared<Batch>();
    std::unique_lock<std::mutex> lk(pmu);
    for (;;) {
      wait_on(pcv, lk, [&] { return parsed.count(blocks_taken) || (reader_done && blocks_taken == blocks_issued) || sh.failed(); });
      if (sh.failed()) return nullptr;
      if (!parsed.count(blocks_taken)) break;  // input exhausted
      auto it = parsed.find(blocks_taken);
      b->n_reads += it->second->n;
      b->parts.push_back(std::move(it->second));
      parsed.erase(it);
      ++blocks_taken;
      pcv.notify_all();
      if (b->n_reads >= batch_reads) break;
    }
    if (b->parts.empty()) return nullptr;
    b->seq = batch_seq++;
    return b;
  };

  auto gpu_main = [&](int g) {
    mtsvgpu_index* ix = handles[(size_t)g];
    uint8_t* pin_packed = nullptr;
    uint64_t* pin_off = nullptr;
    size_t cap_packed = 0, cap_off = 0;
    for (;;) {
      std::shared_ptr<Batch> b = take_batch();
      if (!b) break;
      size_t pbytes = 0;
      for (auto& part : b->parts) pbytes += part->packed.size();
      const auto tb0 = std::chrono::steady_clock::now();
      auto since = [&](std::chrono::steady_clock::time_point t) {
        return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t).count();
      };
      double ms_gather = 0, ms_call = 0;
      if (!dump_mt) {
        if (pbytes + 64 > cap_packed) {
          mtsvgpu_host_free(pin_packed);
          cap_packed = pbytes + pbytes / 4 + 4096;
          pin_packed = (uint8_t*)mtsvgpu_host_alloc(cap_packed);
        }
        if ((b->n_reads + 1) * 8 > cap_off) {
          mtsvgpu_host_free(pin_off);
          cap_off = (b->n_reads + 1) * 8 + (b->n_reads / 4) * 8 + 4096;
          pin_off = (uint64_t*)mtsvgpu_host_alloc(cap_off);
        }
        if (!pin_packed || !pin_off) {
          sh.fail(2, std::string("Error running query: ") + mtsvgpu_last_error());
          break;
        }
        size_t at = 0;
        uint64_t r = 0, bases = 0;
        pin_off[0] = 0;
        for (auto& part : b->parts) {
          memcpy(pin_packed + at, part->packed.data(), part->packed.size());
          at += part->packed.size();
          for (uint32_t i = 0; i < part->n; ++i) pin_off[++r] = (bases += part->len[i]);
          std::vector<uint8_t>().swap(part->packed);
        }
        // default format: the library merges each read's hits into its TaxID=edit list; long: the Hit records
        const mtsvgpu_hit* hits = nullptr;
        const mtsvgpu_taxhit* taxhits = nullptr;
        const uint64_t* hit_off = nullptr;
        uint64_t n_hits = 0;
        ms_gather = since(tb0);
        const auto tc0 = std::chrono::steady_clock::now();
        const int rc = long_fmt ? mtsvgpu_bin_batch_packed(ix, pin_packed, pbytes, pin_off, b->n_reads, &p, &hits,
                                                           &hit_off, &n_hits)
                                : mtsvgpu_assign_batch_packed(ix, pin_packed, pbytes, pin_off, b->n_reads, &p, &taxhits,
                                                              &hit_off, &n_hits);
        if (rc != 0) {
          sh.fail(2, std::string("Error running query: ") + mtsvgpu_last_error());
          break;
        }
        ms_call = since(tc0);
        mtsvgpu_batch_stats bst;
        if (mtsvgpu_last_batch_stats(ix, &bst) == 0) {
          over_len += bst.n_reads_over_limit;
          over_hits += bst.n_strands_over_hits;
        }
        if (long_fmt)  // (the handle's buffers are reused by its next batch)
          b->hits.assign(hits, hits + n_hits);
        else
          b->taxhits.assign(taxhits, taxhits + n_hits);
        b->hit_off.assign(hit_off, hit_off + b->n_reads + 1);
        logf("DEBUG", "gpu %d batch %llu: %llu reads, %llu %s; waited+gathered %.1f ms, library call %.1f ms, results copied %.1f ms",
             g, (unsigned long long)b->seq, (unsigned long long)b->n_reads, (unsigned long long)n_hits,
             long_fmt ? "hits" : "assignments", ms_gather, ms_call,
             since(tc0) - ms_call);
      }
      // format: one pool task per parsed block of the batch
      b->text.resize(b->parts.size());
      b->pending.store((uint32_t)b->parts.size());
      uint64_t first = 0;
      for (size_t k = 0; k < b->parts.size(); ++k) {
        const uint64_t r0 = first;
        first += b->parts[k]->n;
        pool.submit([&, b, k, r0] {
          const ParsedBlock& part = *b->parts[k];
          std::string& text = b->text[k];
          uint64_t lines = 0;
          uint32_t id0 = 0;
          for (uint32_t i = 0; i < part.n; ++i) {
            const uint32_t id1 = part.id_end[i];
            if (dump_mt) {
              text.append(part.ids, id0, id1 - id0);
              text.push_back('\t');
              put_u64(&text, part.len[i]);
              text.push_back('\n');
            } else {
              const uint64_t h0 = b->hit_off[r0 + i], h1 = b->hit_off[r0 + i + 1];
              const size_t before = text.size();
              if (long_fmt)
                format_hits_long(part.ids.data() + id0, id1 - id0, b->hits.data() + h0, h1 - h0, &text);
              else
                format_taxhits(part.ids.data() + id0, id1 - id0, b->taxhits.data() + h0, h1 - h0, &text);
              lines += text.size() != before;
            }
            id0 = id1;
          }
          total_lines += lines;
          if (b->pending.fetch_sub(1) == 1) {
            std::lock_guard<std::mutex> lk(wmu);
            done[b->seq] = b;
            wcv.notify_all();
          }
        });
      }
      total_reads += b->n_reads;
    }
    mtsvgpu_host_free(pin_packed);
    mtsvgpu_host_free(pin_off);
  };

  std::thread writer([&] {
    uint64_t next = 0;
    for (;;) {
      std::shared_ptr<Batch> b;
      {
        std::unique_lock<std::mutex> lk(wmu);
        wait_on(wcv, lk, [&] { return done.count(next) || next == batches_total || sh.failed(); });
        if (!done.count(next)) return;
        b = done[next];
        done.erase(next);
      }
      for (const std::string& t : b->text)
        if (!t.empty() && fwrite(t.data(), 1, t.size(), out) != t.size()) {
          sh.fail(11, std::string("Error writing to result file (") + strerror(errno) + ")");  // src/binner.rs:136-139
          return;
        }
      ++next;
    }
  });

  std::vector<std::thread> gpus;
  for (int g = 0; g < n_gpus; ++g) gpus.emplace_back(gpu_main, g);
  for (auto& t : gpus) t.join();
  reader.join();
  {
    std::lock_guard<std::mutex> lk(wmu);
    batches_total = batch_seq;
    wcv.notify_all();
  }
  writer.join();
  for (auto h : handles) mtsvgpu_index_close(h);
  int code = 0;
  {
    std::lock_guard<std::mutex> lk(sh.mu);
    code = sh.exit_code;
    if (code) logf("ERROR", "%s", sh.error.c_str());
  }
  if (!dump_mt && fclose(out) != 0 && code == 0) {
    logf("ERROR", "Error writing to result file (%s)", strerror(errno));
    code = 11;
  }
  if (code) return code;
  if (over_len.load() || over_hits.load()) {
    // the reference has no such limits: say so loudly (README "Limits"); --strict-limits turns it into a failure
    logf("WARN", "%llu read(s) longer than %d bases and %llu read strand(s) with more than 2^26 seed hits were reported "
                 "without assignments (limits of this implementation)",
         (unsigned long long)over_len.load(), MTSVGPU_MAX_READ_LEN, (unsigned long long)over_hits.load());
    if (strict_limits) return 2;
  }
  double secs = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
  logf("INFO", "All reads binned: %llu reads, %llu result lines. Took %.3f seconds.",
       (unsigned long long)total_reads.load(), (unsigned long long)total_lines.load(), secs);
  return 0;
}
