/*
 * mtsv_b200.h — C ABI of the B200 (sm_100a) implementation of mtsv-binner's
 * read-assignment hot path.
 *
 * Boundary replaced (reference = FofanovLab/mtsv_tools v2.1.0):
 *   MGIndex::matching_tax_ids                       src/index.rs:258-432
 *   the per-read worker closure that calls it 2x    src/binner.rs:77-131
 *   from_file::<MGIndex>                            src/io.rs:115-122
 * FFI precedent this header follows (callee allocates, paired free function,
 * plain pointers and sizes, reentrant per handle): ssw/src/lib.rs:132-154,
 * ssw/build.rs:3-7.  INTEGRATION.md shows the Rust `extern "C"` block a
 * maintainer would add.
 *
 * Conventions
 *   - every function returns 0 on success or a negative MTSVGPU_E* code;
 *     mtsvgpu_last_error() gives a thread-local message for the last failure;
 *   - one mtsvgpu_index per GPU; calls on one handle must be serialised by the
 *     caller, distinct handles are independent;
 *   - buffers returned through `**` are allocated by the library and released
 *     with mtsvgpu_free();
 *   - there is NO CPU fallback: without a CUDA device every entry point that
 *     computes fails with MTSVGPU_ENODEVICE.
 */
#ifndef MTSV_B200_H
#define MTSV_B200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define MTSVGPU_API __attribute__((visibility("default")))
#else
#define MTSVGPU_API
#endif

#define MTSVGPU_OK 0
#define MTSVGPU_EINVAL -1    /* bad argument */
#define MTSVGPU_EIO -2       /* cannot open / short read */
#define MTSVGPU_EFORMAT -3   /* .index does not parse as a bincode MGIndex or fails validation */
#define MTSVGPU_ENODEVICE -4 /* no usable CUDA device */
#define MTSVGPU_ECUDA -5     /* CUDA runtime error */
#define MTSVGPU_ENOMEM -6    /* host or device allocation failed */
#define MTSVGPU_ELIMIT -7    /* input exceeds a documented limit (index >= 2^32 - 64 symbols, exchange slot too small) */

/* Limits that apply PER READ (the batch goes on, the read is reported without hits and counted in
 * mtsvgpu_batch_stats; the reference has no such limits):
 *   - reads longer than MTSVGPU_MAX_READ_LEN bases          -> stats.n_reads_over_limit
 *   - a read strand whose seeds produce more than 2^26 hits -> stats.n_strands_over_hits */
#define MTSVGPU_MAX_READ_LEN 4096

typedef struct mtsvgpu_index mtsvgpu_index;

/* `Hit` — src/index.rs:30-40.  offset = window start - bin start (src/index.rs:416). */
typedef struct {
  uint32_t tax_id;
  uint32_t gi;
  uint64_t offset;
  uint32_t edit;
  uint32_t reserved;
} mtsvgpu_hit;

/* One read's assignment to a TaxID with the minimum edit of its hits there: what the default results format
 * prints as `TaxID=edit` (write_assignments, src/binner.rs:330-352) and what mtsv-collapse mode TaxId keeps. */
typedef struct {
  uint32_t tax_id;
  uint32_t edit;
} mtsvgpu_taxhit;

/* `Bin` — src/index.rs:44-54 (same field order as the bincode record). */
typedef struct {
  uint32_t gi;
  uint32_t tax_id;
  uint64_t start;
  uint64_t end;
} mtsvgpu_bin;

/* Arguments of matching_tax_ids — src/index.rs:258-269; CLI defaults src/bin/mtsv-binner.rs:68-94. */
typedef struct {
  double edit_rate;        /* edit_freq            (--edit-rate, 0.13)   */
  uint32_t seed_size;      /* seed_length          (--seed-size, 18)     */
  uint32_t seed_gap;       /* seed_gap             (--seed-interval, 15) */
  double min_seed;         /* min_seeds_percent    (--min-seed, 0.015)   */
  uint64_t max_hits;       /* max_hits             (--max-hits, 2000)    */
  uint64_t tune_max_hits;  /* tune_max_hits        (--tune-max-hits, 200)*/
  int64_t max_candidates;  /* max_candidates_checked, -1 = None          */
  int64_t max_assignments; /* max_hits_found,         -1 = None          */
  uint32_t strands;        /* 2 (or 0) = forward then reverse complement, as src/binner.rs:102-128;
                              1 = the given strand only, i.e. one matching_tax_ids call */
  uint32_t reserved;
} mtsvgpu_params;

/* Device-side re-layout options (all optional; pass NULL for defaults). */
typedef struct {
  uint32_t sa_rate;       /* suffix-array sample rate kept on the device: 0 = auto (1 = full SA when it
                             fits the memory budget), otherwise a divisor of the file's rate          */
  uint32_t ktab_k;        /* k-mer interval table order: 0 = auto, 1..16; 0xFFFFFFFF = none           */
  uint64_t max_batch_hits;/* cap on seed hits in flight per device sub-batch (0 = default 1<<27)      */
  uint32_t batch_reads;   /* reads per device sub-batch (0 = default: 1<<22 for device-resident input,
                             1<<20 with ramped first/last slices for host input)                       */
  uint32_t reserved;
} mtsvgpu_index_opts;

typedef struct {
  uint64_t text_len;       /* n, including the '$' terminator */
  uint64_t n_bins;
  uint64_t file_sa_rate;   /* s of the .index file */
  uint32_t device_sa_rate; /* s' kept on the device */
  uint32_t ktab_k;
  uint64_t device_bytes;   /* bytes of HBM held by the index */
  uint64_t dollar_row;
  double load_seconds;     /* parse + upload + re-layout */
  double relayout_seconds; /* device re-layout only */
  double build_seconds;    /* mtsvgpu_index_build only: text assembly + suffix array + BWT */
} mtsvgpu_index_info;

/* Per-stage device time of the last mtsvgpu_bin_batch*() or mtsvgpu_assign_batch*(), CUDA events on the launch stream (ms). */
#define MTSVGPU_N_STAGES 12
typedef struct {
  float ms[MTSVGPU_N_STAGES];
  uint64_t launches[MTSVGPU_N_STAGES];
  /* work actually performed, for the roofline (DESIGN.md §4) */
  uint64_t n_queries;      /* read-strands */
  uint64_t n_seed_slots;   /* seeds searched */
  uint64_t n_seed_hits;    /* SA rows located */
  uint64_t n_candidates;   /* windows verified */
  uint64_t n_hits;         /* hits returned */
  uint64_t window_bytes;   /* reference bytes read by the verifier */
  uint64_t rank_queries;   /* 32-byte index sectors touched by seed search: FM blocks + k-mer table (0 unless profiling) */
  uint64_t n_sub_batches;  /* device sub-batches the call was processed in (= launches of every stage kernel) */
  uint64_t h2d_bytes;      /* host API: bytes actually uploaded (offsets of equal-length slices are generated
                              on the device instead) */
  uint64_t n_reads_over_limit;   /* reads longer than MTSVGPU_MAX_READ_LEN: given no hits */
  uint64_t n_strands_over_hits;  /* read strands with more than 2^26 seed hits: given no hits */
} mtsvgpu_batch_stats;

/* ---- index lifetime: replaces from_file::<MGIndex> (src/io.rs:115-122, src/binner.rs:63-67) ---- */
MTSVGPU_API int mtsvgpu_index_open(const char* index_path, int device, const mtsvgpu_index_opts* opts,
                       mtsvgpu_index** out);
/* Same, from the in-memory fields of an MGIndex (src/index.rs:60-68): text incl. '$', bins, the
 * byte BWT and the row-sampled suffix array (rows 0,s,2s,..). */
MTSVGPU_API int mtsvgpu_index_from_parts(const uint8_t* text, uint64_t n, const mtsvgpu_bin* bins,
                             uint64_t n_bins, const uint8_t* bwt, const uint64_t* sa_sample,
                             uint64_t sa_sample_len, uint64_t sa_rate, int device,
                             const mtsvgpu_index_opts* opts, mtsvgpu_index** out);
/* ---- mtsv-build on the device: MGIndex::new (src/index.rs:491-582; called from src/bin/mtsv-build.rs) ----
 * n_seqs reference sequences, raw bytes concatenated in `seqs` (host OR device memory) with n_seqs+1 offsets (host),
 * their GI and TaxID (host; what parse_read_header extracts from `>seqid-taxid`, src/util.rs:26-55).  Bins are laid
 * out in TaxID order, file order within a TaxID (parse_fasta_db's BTreeMap, src/io.rs:135-150); the text is folded
 * to ACGTN and terminated by '$' (src/index.rs:543-556); suffix array and BWT are built on the device and go
 * straight into the device layout: the returned handle is ready for mtsvgpu_bin_batch*.  Peak device memory of
 * the construction is about 29 bytes per reference base. */
MTSVGPU_API int mtsvgpu_index_build(const uint8_t* seqs, const uint64_t* seq_off, const uint32_t* gi,
                        const uint32_t* tax_id, uint64_t n_seqs, int device, const mtsvgpu_index_opts* opts,
                        mtsvgpu_index** out);
/* write_to_file(&index, path) (src/io.rs:125-132): the bincode MGIndex a reference mtsv-binner / mtsv-collapse
 * reads, with Occ checkpoints every `sample_interval` BWT rows (mtsv-build --sample-interval, default 64) and the
 * suffix array sampled every `sa_sample` rows (--sa-sample, default 32).  Works for any loaded handle. */
MTSVGPU_API int mtsvgpu_index_write(mtsvgpu_index* ix, const char* path, uint32_t sample_interval, uint32_t sa_sample);
/* The same fields into caller-allocated host buffers instead of a file (each may be NULL): sequences [text_len],
 * the byte BWT [text_len], the suffix array rows 0, s, 2s, ... [ceil(text_len / sa_sample)]. */
MTSVGPU_API int mtsvgpu_index_export(mtsvgpu_index* ix, uint8_t* text_out, uint8_t* bwt_out, uint64_t* sa_sample_out,
                         uint32_t sa_sample);
MTSVGPU_API void mtsvgpu_index_close(mtsvgpu_index* ix);
MTSVGPU_API int mtsvgpu_index_get_info(const mtsvgpu_index* ix, mtsvgpu_index_info* info);

/* ---- the hot path: replaces the worker closure of run_fastx_pipeline (src/binner.rs:77-131) ----
 * seqs: concatenated raw read bytes exactly as parsed from FASTA/FASTQ (normalisation of
 * src/binner.rs:88-100 happens on the device); seq_off: n_reads+1 offsets into seqs.
 * Output is CSR by read: hits of read i are (*hits)[(*hit_off)[i] .. (*hit_off)[i+1]), forward-strand
 * hits first then reverse-complement hits, each in the reference's acceptance order. */
MTSVGPU_API int mtsvgpu_bin_batch(mtsvgpu_index* ix, const uint8_t* seqs, const uint64_t* seq_off,
                      uint64_t n_reads, const mtsvgpu_params* params, mtsvgpu_hit** hits,
                      uint64_t** hit_off);
/* Same, but the results are left in page-locked buffers owned by the handle (no allocation, no extra
 * copy): valid until the next batch call on this handle or its close; do not free them. */
MTSVGPU_API int mtsvgpu_bin_batch_pinned(mtsvgpu_index* ix, const uint8_t* seqs, const uint64_t* seq_off,
                             uint64_t n_reads, const mtsvgpu_params* params,
                             const mtsvgpu_hit** hits, const uint64_t** hit_off, uint64_t* n_hits);
/* Same with inputs already resident in device memory and results left there.  The returned device
 * pointers are owned by the handle and stay valid until its next batch call or close. */
MTSVGPU_API int mtsvgpu_bin_batch_device(mtsvgpu_index* ix, const uint8_t* d_seqs, const uint64_t* d_seq_off,
                             uint64_t n_reads, const mtsvgpu_params* params,
                             const mtsvgpu_hit** d_hits, const uint64_t** d_hit_off,
                             uint64_t* n_hits);
/* Same as mtsvgpu_bin_batch_pinned for reads the host parser has already PACKED: per read three bit planes of
 * ceil(L/8) bytes each — lo, hi (the two bits of the base code: A 0, C 1, G 2, T 3) and nn (1 = not a base after
 * the folding of src/binner.rs:88-100, lo = hi = 0 there), base j at bit j%8 of byte j/8 — records back to back
 * in read order (57 bytes instead of 150 for a 150-base read, and the upload is what bounds the host API).
 * seq_off still counts BASES (n_reads+1 entries): it gives every read's length.  A parser fills the planes while
 * it scans the record; mtsvgpu_pack_reads does it for bytes already in memory. */
MTSVGPU_API int mtsvgpu_bin_batch_packed(mtsvgpu_index* ix, const uint8_t* packed, uint64_t packed_bytes,
                             const uint64_t* seq_off, uint64_t n_reads, const mtsvgpu_params* params,
                             const mtsvgpu_hit** hits, const uint64_t** hit_off, uint64_t* n_hits);
/* ---- the default results format computed on the device ----
 * The same batches as the three calls above with a smaller output: per read each TaxID that the matching
 * mtsvgpu_bin_batch_* call returns a hit for (on either strand) appears once, with the minimum edit of those hits,
 * by ascending TaxID — exactly the `TaxID=edit` list write_assignments prints (src/binner.rs:330-352); a read
 * without hits gets an empty range.  8 bytes per record instead of 24 per hit, and fewer records where both
 * strands hit a TaxID.  Output is CSR by read: records of read i are (*out)[(*out_off)[i] .. (*out_off)[i+1]),
 * *n_out records in all.  Inputs, ownership and lifetimes are those of the matching mtsvgpu_bin_batch_* call: the
 * pinned and packed results live in the handle's page-locked buffers and the device results in its device
 * buffers, until the next batch call of either kind on the handle.  mtsvgpu_last_batch_stats reports the call as
 * for a bin call (n_hits counts the Hit records before the merge). */
MTSVGPU_API int mtsvgpu_assign_batch_device(mtsvgpu_index* ix, const uint8_t* d_seqs, const uint64_t* d_seq_off,
                                uint64_t n_reads, const mtsvgpu_params* params,
                                const mtsvgpu_taxhit** d_out, const uint64_t** d_out_off, uint64_t* n_out);
MTSVGPU_API int mtsvgpu_assign_batch_pinned(mtsvgpu_index* ix, const uint8_t* seqs, const uint64_t* seq_off,
                                uint64_t n_reads, const mtsvgpu_params* params,
                                const mtsvgpu_taxhit** out, const uint64_t** out_off, uint64_t* n_out);
MTSVGPU_API int mtsvgpu_assign_batch_packed(mtsvgpu_index* ix, const uint8_t* packed, uint64_t packed_bytes,
                                const uint64_t* seq_off, uint64_t n_reads, const mtsvgpu_params* params,
                                const mtsvgpu_taxhit** out, const uint64_t** out_off, uint64_t* n_out);
/* Host helpers of the packed format (no GPU involved).  mtsvgpu_packed_size: bytes of the records of n_reads reads.
 * mtsvgpu_pack_reads: raw read bytes -> records, on `threads` host threads (0 = all); *packed_bytes gets the size. */
MTSVGPU_API uint64_t mtsvgpu_packed_size(const uint64_t* seq_off, uint64_t n_reads);
MTSVGPU_API int mtsvgpu_pack_reads(const uint8_t* seqs, const uint64_t* seq_off, uint64_t n_reads, uint8_t* packed,
                       uint64_t packed_cap, uint64_t* packed_bytes, int threads);
/* One read -> its record (3 * ceil(len / 8) bytes at `record`): what a parser thread calls per sequence. */
MTSVGPU_API void mtsvgpu_pack_read(const uint8_t* seq, uint32_t len, uint8_t* record);
/* Page-locked host memory for batch inputs (uploads from pageable memory are staged by the driver and do not
 * overlap with compute).  NULL on failure. */
MTSVGPU_API void* mtsvgpu_host_alloc(uint64_t bytes);
MTSVGPU_API void mtsvgpu_host_free(void* p);
MTSVGPU_API int mtsvgpu_last_batch_stats(const mtsvgpu_index* ix, mtsvgpu_batch_stats* stats);
/* Launch on a caller-provided cudaStream_t (e.g. torch's current stream); NULL = the handle's own
 * non-blocking stream.  To use the legacy default stream pass cudaStreamLegacy ((cudaStream_t)0x1).
 * Inputs produced on another stream must be complete (or ordered by the caller) before a batch call. */
MTSVGPU_API int mtsvgpu_set_stream(mtsvgpu_index* ix, void* cuda_stream);
/* Collect per-stage CUDA-event timings (costs a few event records per stage); 0 = off (default). */
MTSVGPU_API int mtsvgpu_set_profiling(mtsvgpu_index* ix, int on);

/* ---- stage-level entry points (parity tests of the individual kernels) ---- */
/* FMIndex::backward_search (bio 3.0.0; call site src/index.rs:305) for n_pats patterns of equal
 * length over {A,C,G,T,N}: lower/upper = half-open SA interval when the result is Complete, else 0,0. */
MTSVGPU_API int mtsvgpu_backward_search(mtsvgpu_index* ix, const uint8_t* pats, uint32_t pat_len,
                            uint64_t n_pats, uint64_t* lower, uint64_t* upper);
/* suffix_array(&seq) and bwt(&seq, &sa) of MGIndex::new (src/index.rs:560-567) for a '$'-terminated text in host
 * memory: sa_out[n] (and bwt_out[n] unless NULL). */
MTSVGPU_API int mtsvgpu_suffix_array(int device, const uint8_t* text, uint64_t n, uint32_t* sa_out, uint8_t* bwt_out);
/* SampledSuffixArray::get (bio 3.0.0; call site src/index.rs:347): text position of each SA row. */
MTSVGPU_API int mtsvgpu_locate(mtsvgpu_index* ix, const uint64_t* rows, uint64_t n_rows, uint64_t* pos);
/* Aligner::min_edit_distance (src/align.rs:28-85) for n pairs; pattern i = pats[pat_off[i]..pat_off[i+1]),
 * text i likewise.  Bytes are compared as-is except that, as at src/index.rs:272-279, callers wanting
 * the binner's rule replace 'N' by '.' in the pattern beforehand; any byte outside ACGT never matches. */
MTSVGPU_API int mtsvgpu_edit_distance(int device, const uint8_t* pats, const uint64_t* pat_off,
                          const uint8_t* texts, const uint64_t* text_off, uint64_t n_pairs,
                          uint32_t* edits);

/* ---- chunk-sharded operation: the mtsv-collapse reduction (src/collapse.rs:543-654, mode TaxId) on
 * the device.  Every part holds, for the SAME n_reads reads, a device array of hits and a device array
 * of per-read counts (u32); the result lists, per read, each TaxID once with its minimum edit, by
 * ascending TaxID (write_collapsed_taxid, src/collapse.rs:278-279).  *d_out / *d_out_off are device
 * allocations released with mtsvgpu_device_free().  stream: a cudaStream_t or NULL. */
MTSVGPU_API int mtsvgpu_collapse_device(int device, void* stream, uint32_t n_parts,
                            const mtsvgpu_hit* const* d_hits, const uint32_t* const* d_counts,
                            uint64_t n_reads, mtsvgpu_taxhit** d_out, uint64_t** d_out_off, uint64_t* n_out);
/* Same merge in mtsv-collapse's mode TaxIdGi (src/collapse.rs:603-625): per read and per (TaxID, GI) the hit with
 * the smallest edit, ties to the smallest offset; listed by (TaxID, GI) as write_collapsed_taxid_gi does (:311-318).
 * Output records are whole hits (tax_id, gi, offset, edit). */
MTSVGPU_API int mtsvgpu_collapse_device_taxid_gi(int device, void* stream, uint32_t n_parts,
                            const mtsvgpu_hit* const* d_hits, const uint32_t* const* d_counts,
                            uint64_t n_reads, mtsvgpu_hit** d_out, uint64_t** d_out_off, uint64_t* n_out);
MTSVGPU_API void mtsvgpu_device_free(void* d_ptr);

/* ---- chunk-sharded batches (BASELINE config 3): GPU g holds MG-index chunk g, every read visits every chunk, the
 * per-read TaxID sets are gathered over NVLink into the collapse step.  One process per GPU on one NVSwitch box.
 * The exchange is done by this library's own kernels through peer memory: each rank's communicator owns one device
 * buffer that its peers map (CUDA IPC).  Setup is mediated by the host, which only has to move `world` opaque
 * 128-byte handles between the ranks (any channel: MPI, a pipe, torch.distributed ...):
 *     mtsvgpu_comm_create(...)  on every rank  -> its handle
 *     (host: all-gather the handles, in rank order)
 *     mtsvgpu_comm_connect(comm, all_handles)
 * max_local_reads: upper bound on ceil(n_reads / world) of any batch; max_hits_per_source: upper bound on the hits
 * one chunk produces for one rank's range of reads in one batch (a batch that exceeds it fails on every rank with
 * MTSVGPU_ELIMIT; nothing is truncated).  Destroy only after every rank has finished its last batch. */
#define MTSVGPU_COMM_HANDLE_BYTES 128
typedef struct mtsvgpu_comm mtsvgpu_comm;
MTSVGPU_API int mtsvgpu_comm_create(int device, uint32_t rank, uint32_t world, uint64_t max_local_reads,
                        uint64_t max_hits_per_source, mtsvgpu_comm** out, uint8_t* handle_out);
MTSVGPU_API int mtsvgpu_comm_connect(mtsvgpu_comm* comm, const uint8_t* all_handles);
MTSVGPU_API void mtsvgpu_comm_destroy(mtsvgpu_comm* comm);
/* One batch.  Every rank passes the SAME n_reads reads (device memory, as for mtsvgpu_bin_batch_device) and its own
 * chunk's index.  On return this rank holds, for the reads [*first_read, *first_read + *n_local_reads) (the rank-th
 * of `world` contiguous ranges), what mtsv-collapse leaves of the per-chunk results (src/collapse.rs:597-602,
 * :278-279): each TaxID once with its minimum edit, by ascending TaxID, CSR by read.  The device pointers are owned
 * by the communicator and stay valid until its next batch.  Every rank of the communicator must make the call: a
 * rank that fails before the exchange (or never calls) makes its peers give up after 30 s with MTSVGPU_ECUDA. */
MTSVGPU_API int mtsvgpu_bin_batch_chunked(mtsvgpu_index* ix, mtsvgpu_comm* comm, const uint8_t* d_seqs,
                              const uint64_t* d_seq_off, uint64_t n_reads, const mtsvgpu_params* params,
                              uint64_t* first_read, uint64_t* n_local_reads, const mtsvgpu_taxhit** d_out,
                              const uint64_t** d_out_off, uint64_t* n_out);

MTSVGPU_API void mtsvgpu_free(void* p);
MTSVGPU_API const char* mtsvgpu_last_error(void);
/* Number of kernels this library has launched in this process (all handles). */
MTSVGPU_API uint64_t mtsvgpu_launch_count(void);
MTSVGPU_API const char* mtsvgpu_version(void);

#ifdef __cplusplus
}
#endif
#endif /* MTSV_B200_H */
