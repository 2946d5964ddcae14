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
//                     keeps the results; each GPU takes the next batch whenever it is free
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
  bool ok = true;
  while (ok && (n = getline(&line, &cap, f)) >= 0) {
    std::string s(line, (size_t)n);
    while (!s.empty() && isspace((unsigned char)s.back())) s.pop_back();
    if (s.empty()) continue;  // (a blank line)
    const size_t colon = s.rfind(':');  // rsplitn(2, ':')
    ok = colon != std::string::npos && colon != 0;
    if (ok) ids->insert(s.substr(0, colon));
  }
  free(line);
  fclose(f);
  if (!ok) *err = "Missing read id";
  return ok;
}

// f(record) for every record of a FASTA / FASTQ file; 0 at its end, else FastxBlocks::next's error or -3 (no file)
template <class F>
int for_each_record(const char* path, bool fastq, F f) {
  FastxBlocks in(path, fastq);
  if (!in.ok()) return -3;
  std::string text;
  uint64_t n;
  int rc;
  while ((rc = in.next(&text, &n)) == 1) {
    Lines ln{text.data(), text.data() + text.size()};
    FastxRecord r;
    while (next_record(ln, fastq, true, &r) == 1) f(r);
  }
  return rc;
}

// the number of input records up to the last one that has a line in the results file (0 when none has)
bool resume_offset(const char* results, const char* input, bool fastq, uint64_t* offset, std::string* err) {
  std::unordered_set<std::string> ids;
  if (!read_ids_from_results(results, &ids, err)) return false;
  std::string id;
  uint64_t idx = 0;
  *offset = 0;
  const int rc = for_each_record(input, fastq, [&](const FastxRecord& r) {
    if (ids.count(id.assign(r.id, r.id_end))) *offset = idx + 1;
    ++idx;
  });
  if (rc == 0) return true;
  *err = rc == -3 ? "cannot open input" : rc == -1 ? "parse error while scanning input" : "cannot read input";
  return false;
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

struct Options {
  const char *fasta = nullptr, *fastq = nullptr, *index = nullptr, *results = nullptr;
  mtsvgpu_params p{0.13, 18, 15, 0.015, 2000, 200, -1, -1, 2, 0};
  uint64_t read_offset = 0, batch_reads = 1u << 19;
  bool long_fmt = false, force = false, dump_reads = false, strict_limits = false;
  int device = 0, n_gpus = 1, n_threads = 0;
  bool dump_mt = false;  // test hook: the pipeline without a GPU, printing "id<TAB>length" of each read to stdout
  const char* input() const { return fasta ? fasta : fastq; }
  bool is_fastq() const { return fastq != nullptr; }
};

constexpr int kGoOn = -1;  // the steps of main return this when the run goes on, else the process's exit code

int parse_args(int argc, char** argv, Options* o) {
  auto need = [&](int& i) -> const char* {
    if (i + 1 >= argc) {
      fprintf(stderr, "error: %s requires a value\n", argv[i]);
      exit(1);
    }
    return argv[++i];
  };
  mtsvgpu_params& p = o->p;
  for (int i = 1; i < argc; ++i) {
    std::string a = argv[i];
    if (a == "--fasta" || a == "-fa" || a == "-f") o->fasta = need(i);
    else if (a == "--fastq" || a == "-fq") o->fastq = need(i);
    else if (a == "--index" || a == "-i") o->index = need(i);
    else if (a == "--results" || a == "-m") o->results = need(i);
    else if (a == "--threads" || a == "-t") o->n_threads = atoi(need(i));
    else if (a == "--edit-rate" || a == "-e") p.edit_rate = atof(need(i));
    else if (a == "--seed-size") p.seed_size = (uint32_t)strtoul(need(i), nullptr, 10);
    else if (a == "--seed-interval") p.seed_gap = (uint32_t)strtoul(need(i), nullptr, 10);
    else if (a == "--min-seed") p.min_seed = atof(need(i));
    else if (a == "--max-hits") p.max_hits = strtoull(need(i), nullptr, 10);
    else if (a == "--tune-max-hits") p.tune_max_hits = strtoull(need(i), nullptr, 10);
    else if (a == "--max-assignments") p.max_assignments = strtoll(need(i), nullptr, 10);
    else if (a == "--max-candidates") p.max_candidates = strtoll(need(i), nullptr, 10);
    else if (a == "--read-offset") o->read_offset = strtoull(need(i), nullptr, 10);
    else if (a == "--output-format") o->long_fmt = std::string(need(i)) == "long";
    else if (a == "--force-overwrite") o->force = true;
    else if (a == "-v") g_verbose = true;
    else if (a == "--gpu") o->device = atoi(need(i));
    else if (a == "--gpus") o->n_gpus = atoi(need(i));
    else if (a == "--strict-limits") o->strict_limits = true;
    else if (a == "--dump-reads") o->dump_reads = true;  // test hook: parse the input, print "id<TAB>seq", no GPU
    else if (a == "--dump-reads-mt") o->dump_reads = true, o->n_threads = o->n_threads ? o->n_threads : -1;  // same through the pipeline's scanner + parser
    else if (a == "--batch-reads") o->batch_reads = strtoull(need(i), nullptr, 10);
    else if (a == "-h" || a == "--help") {
      usage();
      return 0;
    } else {
      fprintf(stderr, "error: unknown argument %s\n", a.c_str());
      usage();
      return 1;
    }
  }
  o->dump_mt = o->dump_reads && o->n_threads != 0;
  return kGoOn;
}

int check_options(Options* o) {
  if ((!o->fasta && !o->fastq) || (o->fasta && o->fastq) || (!o->index && !o->dump_mt)) {
    usage();
    return 1;
  }
  // validation as src/bin/mtsv-binner.rs:151,195 (the reference panics; exit code 101 there)
  if (o->p.edit_rate < 0.0 || o->p.edit_rate > 1.0) {
    logf("ERROR", "Edit tolerance proportion must be between 0 and 1, inclusive");
    return 101;
  }
  if (o->p.min_seed <= 0.0 || o->p.min_seed > 1.0) {
    logf("ERROR", "Min seed percent must be between 0 and 1");
    return 101;
  }
  if (o->p.seed_size < 16) logf("WARN", "Seed size may be small enough that it causes performance issues.");
  else if (o->p.seed_size > 24) logf("WARN", "Seed size may be large enough that significant results are ignored.");
  if (!o->results && !o->dump_mt) {
    logf("ERROR", "No results path provided!");
    return 3;  // :262-265
  }
  if (o->n_gpus < 1) o->n_gpus = 1;
  if (o->n_threads <= 0) o->n_threads = (int)std::max(1u, std::thread::hardware_concurrency());
  if (o->batch_reads == 0) o->batch_reads = 1;
  return kGoOn;
}

// test hook --dump-reads: parse the input on this thread, print "id<TAB>seq" of every record from --read-offset on
int dump_reads(const Options& o) {
  uint64_t idx = 0;
  const int rc = for_each_record(o.input(), o.is_fastq(), [&](const FastxRecord& r) {
    if (idx++ < o.read_offset) return;
    fwrite(r.id, 1, (size_t)(r.id_end - r.id), stdout);
    putchar('\t');
    Lines sl{r.seq, r.seq_end};
    const char *b, *e;
    while (sl.next(&b, &e)) fwrite(b, 1, (size_t)(e - b), stdout);
    putchar('\n');
  });
  return rc == -3 ? 2 : rc < 0 ? 12 : 0;
}

// An existing results file is appended to, and the run resumes after the last read it holds, unless
// --force-overwrite is given (src/binner.rs:54-61).  --dump-reads-mt writes to stdout.
int open_results(Options* o, FILE** out) {
  *out = stdout;
  if (o->dump_mt) return kGoOn;
  struct stat sb;
  const bool append = !o->force && stat(o->results, &sb) == 0;
  if (append) {
    uint64_t resume = 0;
    std::string err;
    if (!resume_offset(o->results, o->input(), o->is_fastq(), &resume, &err)) {
      logf("ERROR", "Error computing resume offset: %s", err.c_str());
      return 4;  // :288-291
    }
    logf("INFO", "Existing results detected at %s; resuming after read offset %llu", o->results,
         (unsigned long long)resume);
    o->read_offset += resume;
  }
  if (!(*out = fopen(o->results, append ? "a" : "w"))) {
    logf("ERROR", "Error running query: cannot open %s: %s", o->results, strerror(errno));
    return 2;
  }
  return kGoOn;
}

struct IndexClose {
  void operator()(mtsvgpu_index* ix) const { mtsvgpu_index_close(ix); }
};
struct HostFree {
  void operator()(void* p) const { mtsvgpu_host_free(p); }
};
using Index = std::unique_ptr<mtsvgpu_index, IndexClose>;

// A first small batch brings in what a fresh process pays once (kernel images, workspaces, page-locked result
// buffers) while the other devices and the reader start up.  Its results are discarded.
void warm_up(mtsvgpu_index* ix, int g, const Options& o) {
  std::vector<uint8_t> seq(256 * 150);
  std::vector<uint64_t> off(257);
  uint32_t x = 12345u + (uint32_t)g;
  for (auto& c : seq) c = (uint8_t)"ACGT"[(x = x * 1664525u + 1013904223u) >> 30];
  for (size_t i = 0; i <= 256; ++i) off[i] = i * 150;
  const mtsvgpu_hit* wh = nullptr;
  const mtsvgpu_taxhit* wt = nullptr;
  const uint64_t* wo = nullptr;
  uint64_t wn = 0;
  if (o.long_fmt) (void)mtsvgpu_bin_batch_pinned(ix, seq.data(), off.data(), 256, &o.p, &wh, &wo, &wn);
  else (void)mtsvgpu_assign_batch_pinned(ix, seq.data(), off.data(), 256, &o.p, &wt, &wo, &wn);
}

// One handle per GPU, opened and warmed up side by side (null handles for --dump-reads-mt); none when one fails.
std::vector<Index> open_indexes(const Options& o) {
  std::vector<Index> ix((size_t)o.n_gpus);
  if (o.dump_mt) return ix;
  logf("INFO", "Deserializing candidate filter ...");
  std::vector<std::thread> openers;
  std::vector<std::string> errs((size_t)o.n_gpus);
  for (int g = 0; g < o.n_gpus; ++g)
    openers.emplace_back([&, g] {
      mtsvgpu_index* h = nullptr;
      if (mtsvgpu_index_open(o.index, o.device + g, nullptr, &h) == 0) warm_up(h, g, o);
      else errs[(size_t)g] = mtsvgpu_last_error();
      ix[(size_t)g].reset(h);
    });
  for (auto& t : openers) t.join();
  for (int g = 0; g < o.n_gpus; ++g)
    if (!ix[(size_t)g]) {
      logf("ERROR", "Error running query: %s", errs[(size_t)g].c_str());
      return {};
    }
  return ix;
}

// ---- pipeline ----
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
};

// parse + pack one block of whole records, all but the first `skip` (a worker's task); false at a read too long
bool parse_block(const TextBlock& tb, bool fastq, uint64_t skip, ParsedBlock* out) {
  out->len.reserve(tb.n_records - skip);
  out->id_end.reserve(tb.n_records - skip);
  out->packed.reserve(tb.text.size() / 4);
  Lines ln{tb.text.data(), tb.text.data() + tb.text.size()};
  FastxRecord r;
  std::string multi;
  for (uint64_t i = 0; next_record(ln, fastq, true, &r) == 1; ++i) {
    if (i < skip) continue;
    if (r.len > 0xfffffff0ull) return false;
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
  return true;
}

// page-locked memory for a GPU thread's batch input
struct PinnedBuf {
  std::unique_ptr<void, HostFree> p;
  size_t cap = 0;
  bool fit(size_t need, size_t grown) {  // false: `need` bytes do not fit and `grown` bytes cannot be allocated
    if (need > cap) {
      p.reset();  // (the old buffer is freed before the new one is allocated)
      p.reset(mtsvgpu_host_alloc(cap = grown));
    }
    return p != nullptr;
  }
};

// The threads of one run (see the top of the file), their shared state and their stages.  One mutex guards the queues
// and the failure, so a failure wakes every wait.  run() returns once all threads, workers included, have ended.
class Pipeline {
 public:
  Pipeline(const Options& o, FastxBlocks& blocks, FILE* out, const std::vector<Index>& ix)
      : o_(o), blocks_(blocks), out_(out), ix_(ix) {}
  std::atomic<uint64_t> total_reads{0}, total_lines{0}, over_len{0}, over_hits{0};

  int run() {
    std::vector<std::thread> workers, gpus;
    for (int i = 0; i < o_.n_threads; ++i) workers.emplace_back([this] { work(); });
    std::thread reader([this] { read_blocks(); });
    std::thread writer([this] { write_batches(); });
    for (int g = 0; g < o_.n_gpus; ++g)
      gpus.emplace_back([this, g] {
        PinnedBuf packed, off;
        while (std::shared_ptr<Batch> b = take_batch()) {
          if (!o_.dump_mt && !compute(g, b.get(), &packed, &off)) break;
          queue_format(b);
        }
      });
    for (auto& t : gpus) t.join();
    reader.join();
    {
      std::lock_guard<std::mutex> lk(mu_);  // no task is queued after this: the workers end once the queue is empty
      batches_total_ = batch_seq_;
      stop_ = true;
      done_cv_.notify_all();
      task_cv_.notify_all();
    }
    writer.join();
    for (auto& t : workers) t.join();
    if (code_) logf("ERROR", "%s", error_.c_str());
    return code_;
  }

 private:
  void fail(int code, const std::string& msg) {
    std::lock_guard<std::mutex> lk(mu_);
    if (code_ == 0) {
      error_ = msg;
      code_ = code;
    }
    parsed_cv_.notify_all();
    done_cv_.notify_all();
  }

  void submit(std::function<void()> task) {
    std::lock_guard<std::mutex> lk(mu_);
    tasks_.push_back(std::move(task));
    task_cv_.notify_one();
  }
  void work() {
    for (;;) {
      std::function<void()> task;
      {
        std::unique_lock<std::mutex> lk(mu_);
        task_cv_.wait(lk, [this] { return stop_ || !tasks_.empty(); });
        if (tasks_.empty()) return;
        task = std::move(tasks_.front());
        tasks_.pop_front();
      }
      task();
    }
  }

  // blocks of whole records to the parser tasks, with at most max_in_flight of them issued and not yet taken
  void read_blocks() {
    const uint64_t max_in_flight = (uint64_t)std::max(8, 4 * o_.n_threads) + o_.batch_reads / 8192;
    uint64_t records_seen = 0;  // complete records read so far (including skipped ones)
    while (!code_) {
      auto tb = std::make_shared<TextBlock>();
      const int rc = blocks_.next(&tb->text, &tb->n_records);
      if (rc == 0) break;
      if (rc < 0 || blocks_.malformed_next()) {  // (the records of a block that ends at a malformed one are not binned)
        std::string msg = "Unable to read from input file";
        if (rc != -2) msg += ": malformed record after " + std::to_string(records_seen) + " reads";
        fail(12, msg);  // src/binner.rs:81-84
        break;
      }
      // .skip(read_offset) (src/binner.rs:176,199): whole blocks are dropped, the parser skips the first records of
      // a straddling block
      const uint64_t first = records_seen;
      records_seen += tb->n_records;
      if (records_seen <= o_.read_offset) continue;
      const uint64_t skip = o_.read_offset > first ? o_.read_offset - first : 0;
      {
        std::unique_lock<std::mutex> lk(mu_);
        parsed_cv_.wait(lk, [&] { return issued_ - taken_ < max_in_flight || code_; });
        tb->seq = issued_++;
      }
      submit([this, tb, skip] {
        auto pb = std::make_unique<ParsedBlock>();
        if (!code_ && !parse_block(*tb, o_.is_fastq(), skip, pb.get()))
          fail(12, "Unable to read from input file: malformed record");
        std::lock_guard<std::mutex> lk(mu_);
        parsed_[tb->seq] = std::move(pb);
        parsed_cv_.notify_all();
      });
    }
    std::lock_guard<std::mutex> lk(mu_);
    reader_done_ = true;
    parsed_cv_.notify_all();
  }

  // consecutive parsed blocks until they hold batch_reads reads or the input ends; null when none is left or failed
  std::shared_ptr<Batch> take_batch() {
    std::lock_guard<std::mutex> tlk(take_mu_);
    auto b = std::make_shared<Batch>();
    std::unique_lock<std::mutex> lk(mu_);
    for (;;) {
      parsed_cv_.wait(lk, [&] { return parsed_.count(taken_) || (reader_done_ && taken_ == issued_) || code_; });
      if (code_) return nullptr;
      auto it = parsed_.find(taken_);
      if (it == parsed_.end()) break;  // input exhausted
      b->n_reads += it->second->n;
      b->parts.push_back(std::move(it->second));
      parsed_.erase(it);
      ++taken_;
      parsed_cv_.notify_all();
      if (b->n_reads >= o_.batch_reads) break;
    }
    if (b->parts.empty()) return nullptr;
    b->seq = batch_seq_++;
    return b;
  }

  // gathers the batch into page-locked memory, runs it on GPU g, copies the results out of the handle's buffers
  bool compute(int g, Batch* b, PinnedBuf* pin_packed, PinnedBuf* pin_off) {
    size_t pbytes = 0;
    for (auto& part : b->parts) pbytes += part->packed.size();
    const auto tb0 = std::chrono::steady_clock::now();
    auto since = [](std::chrono::steady_clock::time_point t) {
      return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t).count();
    };
    const uint64_t n = b->n_reads;
    if (!pin_packed->fit(pbytes + 64, pbytes + pbytes / 4 + 4096) ||
        !pin_off->fit((n + 1) * 8, (n + 1) * 8 + (n / 4) * 8 + 4096)) {
      fail(2, std::string("Error running query: ") + mtsvgpu_last_error());
      return false;
    }
    uint8_t* packed = (uint8_t*)pin_packed->p.get();
    uint64_t* off = (uint64_t*)pin_off->p.get();
    size_t at = 0;
    uint64_t r = 0, bases = 0;
    off[0] = 0;
    for (auto& part : b->parts) {
      memcpy(packed + at, part->packed.data(), part->packed.size());
      at += part->packed.size();
      for (uint32_t i = 0; i < part->n; ++i) off[++r] = (bases += part->len[i]);
      std::vector<uint8_t>().swap(part->packed);
    }
    // default format: the library merges each read's hits into its TaxID=edit list; long: the Hit records
    mtsvgpu_index* ix = ix_[(size_t)g].get();
    const mtsvgpu_hit* hits = nullptr;
    const mtsvgpu_taxhit* taxhits = nullptr;
    const uint64_t* hit_off = nullptr;
    uint64_t n_hits = 0;
    const double ms_gather = since(tb0);
    const auto tc0 = std::chrono::steady_clock::now();
    const int rc = o_.long_fmt ? mtsvgpu_bin_batch_packed(ix, packed, pbytes, off, n, &o_.p, &hits, &hit_off, &n_hits)
                               : mtsvgpu_assign_batch_packed(ix, packed, pbytes, off, n, &o_.p, &taxhits, &hit_off,
                                                             &n_hits);
    if (rc != 0) {
      fail(2, std::string("Error running query: ") + mtsvgpu_last_error());
      return false;
    }
    const double ms_call = since(tc0);
    mtsvgpu_batch_stats bst;
    if (mtsvgpu_last_batch_stats(ix, &bst) == 0) {
      over_len += bst.n_reads_over_limit;
      over_hits += bst.n_strands_over_hits;
    }
    if (o_.long_fmt)
      b->hits.assign(hits, hits + n_hits);
    else
      b->taxhits.assign(taxhits, taxhits + n_hits);
    b->hit_off.assign(hit_off, hit_off + n + 1);
    logf("DEBUG", "gpu %d batch %llu: %llu reads, %llu %s; waited+gathered %.1f ms, library call %.1f ms, results copied %.1f ms",
         g, (unsigned long long)b->seq, (unsigned long long)n, (unsigned long long)n_hits,
         o_.long_fmt ? "hits" : "assignments", ms_gather, ms_call, since(tc0) - ms_call);
    return true;
  }

  // one format task per parsed block of the batch; the last one to finish hands the batch to the writer
  void queue_format(const std::shared_ptr<Batch>& b) {
    b->text.resize(b->parts.size());
    b->pending.store((uint32_t)b->parts.size());
    uint64_t r0 = 0;  // the part's first read in the batch
    for (size_t k = 0; k < b->parts.size(); ++k) {
      submit([this, b, k, r0] {
        const ParsedBlock& part = *b->parts[k];
        std::string& text = b->text[k];
        uint64_t lines = 0;
        uint32_t id0 = 0;
        for (uint32_t i = 0; i < part.n; ++i) {
          const uint32_t id1 = part.id_end[i];
          if (o_.dump_mt) {
            text.append(part.ids, id0, id1 - id0);
            text.push_back('\t');
            put_u64(&text, part.len[i]);
            text.push_back('\n');
          } else {
            const uint64_t h0 = b->hit_off[r0 + i], h1 = b->hit_off[r0 + i + 1];
            const size_t before = text.size();
            if (o_.long_fmt)
              format_hits_long(part.ids.data() + id0, id1 - id0, b->hits.data() + h0, h1 - h0, &text);
            else
              format_taxhits(part.ids.data() + id0, id1 - id0, b->taxhits.data() + h0, h1 - h0, &text);
            lines += text.size() != before;
          }
          id0 = id1;
        }
        total_lines += lines;
        if (b->pending.fetch_sub(1) == 1) {
          std::lock_guard<std::mutex> lk(mu_);
          done_[b->seq] = b;
          done_cv_.notify_all();
        }
      });
      r0 += b->parts[k]->n;
    }
    total_reads += b->n_reads;
  }

  void write_batches() {
    for (uint64_t next = 0;; ++next) {
      std::shared_ptr<Batch> b;
      {
        std::unique_lock<std::mutex> lk(mu_);
        done_cv_.wait(lk, [&] { return done_.count(next) || next == batches_total_ || code_; });
        auto it = done_.find(next);
        if (it == done_.end()) return;
        b = std::move(it->second);
        done_.erase(it);
      }
      for (const std::string& t : b->text)
        if (!t.empty() && fwrite(t.data(), 1, t.size(), out_) != t.size()) {
          fail(11, std::string("Error writing to result file (") + strerror(errno) + ")");  // src/binner.rs:136-139
          return;
        }
    }
  }

  const Options& o_;
  FastxBlocks& blocks_;
  FILE* out_;
  const std::vector<Index>& ix_;
  std::mutex mu_;
  std::atomic<int> code_{0};  // exit code of the first failure (set under mu_), and its message
  std::string error_;
  std::condition_variable task_cv_;          // the workers' queue of parse and format tasks
  std::deque<std::function<void()>> tasks_;
  bool stop_ = false;
  std::condition_variable parsed_cv_;                        // a block was parsed or taken, or the reader is done
  std::map<uint64_t, std::unique_ptr<ParsedBlock>> parsed_;  // parsed blocks waiting for their turn, by sequence
  uint64_t issued_ = 0, taken_ = 0;                          // blocks handed to the parser / taken into batches
  bool reader_done_ = false;
  std::mutex take_mu_;  // serialises take_batch, so that batches are consecutive runs of blocks
  uint64_t batch_seq_ = 0;
  std::condition_variable done_cv_;                  // a batch was formatted, or the number of batches is known
  std::map<uint64_t, std::shared_ptr<Batch>> done_;  // formatted (or empty) batches by sequence number
  uint64_t batches_total_ = ~0ull;                   // known once the GPU threads are done
};

}  // namespace

int main(int argc, char** argv) {
  Options o;
  int code = parse_args(argc, argv, &o);
  if (code != kGoOn) return code;
  if (o.dump_reads && !o.dump_mt && o.input()) return dump_reads(o);
  if ((code = check_options(&o)) != kGoOn) return code;
  FILE* out;  // (on an early return, exit() closes it)
  if ((code = open_results(&o, &out)) != kGoOn) return code;
  FastxBlocks blocks(o.input(), o.is_fastq());  // src/binner.rs:21-33
  if (!blocks.ok()) {
    logf("ERROR", "Error running query: cannot open %s", o.input());
    return 2;
  }
  std::vector<Index> ix = open_indexes(o);
  if (ix.empty()) return 2;
  logf("INFO", "Beginning queries.");
  const auto t0 = std::chrono::steady_clock::now();
  Pipeline pipe(o, blocks, out, ix);
  code = pipe.run();
  ix.clear();
  if (!o.dump_mt && fclose(out) != 0 && code == 0) {
    logf("ERROR", "Error writing to result file (%s)", strerror(errno));
    code = 11;
  }
  if (code) return code;
  if (pipe.over_len.load() || pipe.over_hits.load()) {
    // the reference has no such limits: say so loudly (README "Limits"); --strict-limits turns it into a failure
    logf("WARN", "%llu read(s) longer than %d bases and %llu read strand(s) with more than 2^26 seed hits were reported "
                 "without assignments (limits of this implementation)",
         (unsigned long long)pipe.over_len.load(), MTSVGPU_MAX_READ_LEN, (unsigned long long)pipe.over_hits.load());
    if (o.strict_limits) return 2;
  }
  double secs = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
  logf("INFO", "All reads binned: %llu reads, %llu result lines. Took %.3f seconds.",
       (unsigned long long)pipe.total_reads.load(), (unsigned long long)pipe.total_lines.load(), secs);
  return 0;
}
