// mtsv-build (B200) — the reference's index builder command line above the C ABI.
//
// Mirrors src/bin/mtsv-build.rs:17-123 (flags, defaults, exit codes) and the host part of
// builder::build_and_write_index (src/builder.rs:14-36): FASTA records -> (GI, TaxID) from the `ACCESSION-TAXID`
// header (parse_read_header, src/util.rs:26-55) or from a mapping file with header / taxid / seqid columns
// (parse_header_mapping, src/io.rs:35-112; --skip-missing as parse_fasta_db_with_mapping :153-184).  The index
// itself (MGIndex::new, src/index.rs:491-582) is built on the GPU by mtsvgpu_index_build and written as the
// bincode `.index` by mtsvgpu_index_write.  Exit codes: 0 ok, 1 any error (as the reference).
#include <ctype.h>
#include <errno.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <chrono>
#include <string>
#include <unordered_map>
#include <utility>
#include <vector>

#include "../../include/mtsv_b200.h"
#include "fastx.h"

namespace {

bool g_verbose = false;
void logf(const char* level, const char* fmt, ...) {
  if (!g_verbose && strcmp(level, "DEBUG") == 0) return;
  va_list ap;
  va_start(ap, fmt);
  fprintf(stderr, "[%s mtsv_build] ", level);
  vfprintf(stderr, fmt, ap);
  fputc('\n', stderr);
  va_end(ap);
}

bool parse_u32(const std::string& t, uint32_t* v) {
  if (t.empty()) return false;
  uint64_t x = 0;
  for (char c : t) {
    if (c < '0' || c > '9') return false;
    x = x * 10 + (uint64_t)(c - '0');
    if (x > 0xffffffffull) return false;
  }
  *v = (uint32_t)x;
  return true;
}

// `ACCESSION-TAXID` with exactly one dash (src/util.rs:26-55)
bool parse_read_header(const std::string& h, uint32_t* gi, uint32_t* tax, std::string* err) {
  const size_t d = h.find('-');
  if (d == std::string::npos || h.find('-', d + 1) != std::string::npos) {
    *err = "Invalid header: " + h;
    return false;
  }
  if (!parse_u32(h.substr(0, d), gi)) {
    *err = "Invalid integer: " + h.substr(0, d);
    return false;
  }
  if (!parse_u32(h.substr(d + 1), tax)) {
    *err = "Invalid integer: " + h.substr(d + 1);
    return false;
  }
  return true;
}

std::string trim(const std::string& s) {
  size_t b = 0, e = s.size();
  while (b < e && isspace((unsigned char)s[b])) ++b;
  while (e > b && isspace((unsigned char)s[e - 1])) --e;
  return s.substr(b, e - b);
}

std::vector<std::string> split_fields(const std::string& line, char delim) {  // delim 0: whitespace
  std::vector<std::string> out;
  if (delim) {
    size_t b = 0;
    for (;;) {
      size_t e = line.find(delim, b);
      out.push_back(trim(line.substr(b, e == std::string::npos ? std::string::npos : e - b)));
      if (e == std::string::npos) break;
      b = e + 1;
    }
  } else {
    size_t i = 0;
    while (i < line.size()) {
      while (i < line.size() && isspace((unsigned char)line[i])) ++i;
      size_t b = i;
      while (i < line.size() && !isspace((unsigned char)line[i])) ++i;
      if (i > b) out.push_back(line.substr(b, i - b));
    }
  }
  return out;
}

// header -> (seqid, taxid); src/io.rs:35-112
bool parse_header_mapping(const char* path, std::unordered_map<std::string, std::pair<uint32_t, uint32_t>>* map,
                          std::string* err) {
  FILE* f = fopen(path, "r");
  if (!f) {
    *err = strerror(errno);
    return false;
  }
  char* buf = nullptr;
  size_t cap = 0;
  ssize_t n;
  bool have_header = false;
  char delim = 0;
  size_t hi = 0, ti = 0, si = 0;
  bool ok = true;
  while (ok && (n = getline(&buf, &cap, f)) >= 0) {
    std::string line = trim(std::string(buf, (size_t)n));
    if (line.empty()) continue;
    if (!have_header) {
      for (char c : {',', '\t', ';', '|'})
        if (std::string(buf, (size_t)n).find(c) != std::string::npos) {
          delim = c;
          break;
        }
      std::vector<std::string> h = split_fields(line, delim);
      int fh = -1, ft = -1, fs = -1;
      for (size_t i = 0; i < h.size(); ++i) {
        std::string x = h[i];
        for (char& c : x) c = (char)tolower((unsigned char)c);
        if (x == "header" && fh < 0) fh = (int)i;
        if (x == "taxid" && ft < 0) ft = (int)i;
        if ((x == "seqid" || x == "gi") && fs < 0) fs = (int)i;
      }
      if (fh < 0 || ft < 0 || fs < 0) {
        *err = std::string("Missing '") + (fh < 0 ? "header" : ft < 0 ? "taxid" : "seqid") + "' column in mapping file";
        ok = false;
        break;
      }
      hi = (size_t)fh;
      ti = (size_t)ft;
      si = (size_t)fs;
      have_header = true;
      continue;
    }
    std::vector<std::string> fld = split_fields(line, delim);
    const size_t mx = std::max(hi, std::max(ti, si));
    if (fld.size() <= mx) {
      *err = "Invalid mapping row: " + line;
      ok = false;
      break;
    }
    uint32_t tax = 0, seq = 0;
    if (fld[hi].empty()) {
      *err = "Empty header in mapping file";
      ok = false;
    } else if (!parse_u32(fld[ti], &tax)) {
      *err = "Invalid integer: " + fld[ti];
      ok = false;
    } else if (!parse_u32(fld[si], &seq)) {
      *err = "Invalid integer: " + fld[si];
      ok = false;
    } else if (!map->emplace(fld[hi], std::make_pair(seq, tax)).second) {
      *err = "Duplicate header mapping for " + fld[hi];
      ok = false;
    }
  }
  free(buf);
  fclose(f);
  if (ok && !have_header) {
    *err = "Empty mapping file";
    ok = false;
  }
  return ok;
}

void usage() {
  fprintf(stderr,
          "mtsv-build (B200)\n"
          "USAGE: mtsv-build --fasta <FASTA> --index <INDEX> [FLAGS]\n"
          "  -f, --fasta <FASTA>            Path to FASTA database file (gz detected automatically).\n"
          "  -i, --index <INDEX>            Path to mtsv index file to write.\n"
          "      --sa-sample <n>            Suffix array sampling rate [default: 32]\n"
          "      --sample-interval <n>      BWT occurrence sampling rate [default: 64]\n"
          "      --mapping <PATH>           header -> taxid / seqid mapping file (columns: header, taxid, seqid)\n"
          "      --skip-missing             Skip FASTA records missing from the mapping file\n"
          "      --gpu <id>                 CUDA device [default: 0]\n"
          "  -v                             debug-level logging\n");
}

}  // namespace

int main(int argc, char** argv) {
  const char *fasta = nullptr, *index = nullptr, *mapping = nullptr;
  uint32_t sa_sample = 32, sample_interval = 64;
  bool skip_missing = false;
  int device = 0;
  auto need = [&](int& i) -> const char* {
    if (i + 1 >= argc) {
      fprintf(stderr, "error: %s requires a value\n", argv[i]);
      exit(1);
    }
    return argv[++i];
  };
  for (int i = 1; i < argc; ++i) {
    std::string a = argv[i];
    if (a == "--fasta" || a == "-f") fasta = need(i);
    else if (a == "--index" || a == "-i") index = need(i);
    else if (a == "--sa-sample") sa_sample = (uint32_t)strtoul(need(i), nullptr, 10);
    else if (a == "--sample-interval") sample_interval = (uint32_t)strtoul(need(i), nullptr, 10);
    else if (a == "--mapping") mapping = need(i);
    else if (a == "--skip-missing") skip_missing = true;
    else if (a == "--gpu") device = atoi(need(i));
    else if (a == "-v") g_verbose = true;
    else if (a == "-h" || a == "--help") {
      usage();
      return 0;
    } else {
      fprintf(stderr, "error: unknown argument %s\n", a.c_str());
      usage();
      return 1;
    }
  }
  if (!fasta || !index) {
    usage();
    return 1;
  }
  if (sa_sample == 0 || sample_interval == 0) {
    logf("ERROR", "Invalid sample interval entered!");
    return 1;
  }
  if (skip_missing && !mapping) logf("WARN", "--skip-missing has no effect without --mapping.");
  std::unordered_map<std::string, std::pair<uint32_t, uint32_t>> map;
  if (mapping) {
    std::string err;
    if (!parse_header_mapping(mapping, &map, &err)) {
      logf("ERROR", "Error parsing mapping file: %s", err.c_str());
      return 1;
    }
  }
  const auto t0 = std::chrono::steady_clock::now();
  logf("DEBUG", "Opening FASTA database file...");
  FastxBlocks in(fasta, false);
  if (!in.ok()) {
    logf("ERROR", "Unable to open FASTA database for parsing.");
    return 1;
  }
  std::vector<uint8_t> seqs;
  std::vector<uint64_t> off(1, 0);
  std::vector<uint32_t> gis, taxs;
  std::string text;
  uint64_t n;
  int rc;
  while ((rc = in.next(&text, &n)) == 1) {
    if (seqs.size() + text.size() > seqs.capacity())  // (one reallocation for a block of one long record)
      seqs.reserve(std::max(2 * seqs.capacity(), seqs.size() + text.size()));
    Lines ln{text.data(), text.data() + text.size()};
    FastxRecord r;
    while (next_record(ln, false, true, &r) == 1) {
      const std::string id(r.id, r.id_end);
      uint32_t gi = 0, tax = 0;
      if (mapping) {
        auto it = map.find(id);
        if (it == map.end()) {
          if (!skip_missing) {
            logf("ERROR", "Error building index: Missing mapping for header %s", id.c_str());
            return 1;
          }
          logf("WARN", "Missing mapping for header %s, skipping.", id.c_str());
          continue;
        }
        gi = it->second.first;
        tax = it->second.second;
      } else {
        std::string err;
        if (!parse_read_header(id, &gi, &tax, &err)) {
          logf("ERROR", "Error building index: %s", err.c_str());
          return 1;
        }
      }
      gis.push_back(gi);
      taxs.push_back(tax);
      Lines sl{r.seq, r.seq_end};
      const char *b, *e;
      while (sl.next(&b, &e)) seqs.insert(seqs.end(), b, e);
      off.push_back(seqs.size());
    }
  }
  if (rc < 0) {  // (a FASTA record can only be malformed by not starting with '>')
    logf("ERROR", rc == -1 ? "Error building index: FASTA record does not start with '>'"
                           : "Unable to read FASTA database.");
    return 1;
  }
  if (gis.empty()) {
    logf("ERROR", "Error building index: no sequences to index");
    return 1;
  }
  logf("INFO", "File parsed, building index...");
  mtsvgpu_index* ix = nullptr;
  mtsvgpu_index_opts opts;
  memset(&opts, 0, sizeof opts);
  opts.ktab_k = 0xFFFFFFFFu;  // no query acceleration structures: the handle is only written out
  if (mtsvgpu_index_build(seqs.data(), off.data(), gis.data(), taxs.data(), gis.size(), device, &opts, &ix) != 0) {
    logf("ERROR", "Error building index: %s", mtsvgpu_last_error());
    return 1;
  }
  logf("INFO", "Writing index to file...");
  if (mtsvgpu_index_write(ix, index, sample_interval, sa_sample) != 0) {
    logf("ERROR", "Error building index: %s", mtsvgpu_last_error());
    mtsvgpu_index_close(ix);
    return 1;
  }
  mtsvgpu_index_info info;
  mtsvgpu_index_get_info(ix, &info);
  mtsvgpu_index_close(ix);
  logf("INFO", "Done building and writing index! (%llu symbols, %llu bins; suffix array + BWT %.2f s on the GPU, %.2f s in all)",
       (unsigned long long)info.text_len, (unsigned long long)info.n_bins, info.build_seconds,
       std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count());
  return 0;
}
