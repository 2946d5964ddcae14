"""Host mirror of the reference's MGIndex for the read-assignment path (src/index.rs)."""
import ctypes as C
import os
from collections import namedtuple

import numpy as np

from . import _lib
from ._lib import HitStruct, BinStruct, InfoStruct, OptsStruct, ParamsStruct, StatsStruct, TaxHitStruct, check

#: `Hit` — src/index.rs:30-40
Hit = namedtuple("Hit", ["tax_id", "gi", "offset", "edit"])

HIT_DTYPE = np.dtype([("tax_id", "<u4"), ("gi", "<u4"), ("offset", "<u8"), ("edit", "<u4"),
                      ("reserved", "<u4")])

#: mtsvgpu_taxhit: one `TaxID=edit` entry of the default results format (src/binner.rs:330-352)
TAXHIT_DTYPE = np.dtype([("tax_id", "<u4"), ("edit", "<u4")])


class Params:
    """Arguments of ``matching_tax_ids`` (src/index.rs:258-269); defaults of the mtsv-binner CLI
    (src/bin/mtsv-binner.rs:68-94)."""

    def __init__(self, edit_rate=0.13, seed_size=18, seed_gap=15, min_seed=0.015, max_hits=2000,
                 tune_max_hits=200, max_candidates=None, max_assignments=None):
        self.edit_rate = edit_rate
        self.seed_size = seed_size
        self.seed_gap = seed_gap
        self.min_seed = min_seed
        self.max_hits = max_hits
        self.tune_max_hits = tune_max_hits
        self.max_candidates = max_candidates
        self.max_assignments = max_assignments

    def c_struct(self, strands=2):
        return ParamsStruct(self.edit_rate, self.seed_size, self.seed_gap, self.min_seed, self.max_hits,
                            self.tune_max_hits,
                            -1 if self.max_candidates is None else self.max_candidates,
                            -1 if self.max_assignments is None else self.max_assignments, strands, 0)


def _ptr(a):
    return C.c_void_p(a.ctypes.data)


def pack_reads(reads):
    """list of bytes -> (uint8 concat, uint64 offsets[n+1])"""
    off = np.zeros(len(reads) + 1, dtype=np.uint64)
    if len(reads):
        off[1:] = np.cumsum([len(s) for s in reads], dtype=np.uint64)
    cat = np.frombuffer(b"".join(reads), dtype=np.uint8).copy() if len(reads) else np.zeros(0, np.uint8)
    return cat, off


def pack_reads_planes(reads, threads=0, out=None):
    """Raw reads -> the packed records mtsvgpu_bin_batch_packed takes (include/mtsv_b200.h): returns
    (uint8 records, uint64 base offsets).  `out`: a preallocated (e.g. page-locked) uint8 array to fill."""
    L = _lib.load_library()
    cat, off = reads if isinstance(reads, tuple) else pack_reads(reads)
    cat = np.ascontiguousarray(cat, dtype=np.uint8)
    off = np.ascontiguousarray(off, dtype=np.uint64)
    n = len(off) - 1
    if out is None:
        out = np.empty(int(L.mtsvgpu_packed_size(_ptr(off), n)), dtype=np.uint8)
    nb = C.c_uint64()
    check(L.mtsvgpu_pack_reads(_ptr(cat) if len(cat) else None, _ptr(off), n, _ptr(out) if len(out) else None,
                               len(out), C.byref(nb), threads))
    return out[: nb.value], off


class MGIndex:
    """Device-resident MG-index.  ``MGIndex.from_file`` replaces ``from_file::<MGIndex>``
    (src/io.rs:115-122, called at src/binner.rs:63): the `.index` written by mtsv-build is parsed,
    re-laid out on the GPU (not rebuilt) and kept in HBM."""

    def __init__(self, handle):
        self._h = C.c_void_p(handle)

    # ---- construction ----
    @staticmethod
    def _opts(sa_rate=0, ktab_k=0, max_batch_hits=0, batch_reads=0):
        return OptsStruct(sa_rate, ktab_k, max_batch_hits, batch_reads, 0)

    @classmethod
    def from_file(cls, path, device=0, **opts):
        L = _lib.load_library()
        h = C.c_void_p()
        o = cls._opts(**opts)
        check(L.mtsvgpu_index_open(os.fsencode(path), device, C.byref(o), C.byref(h)))
        return cls(h.value)

    @classmethod
    def from_parts(cls, text, bins, bwt, sa_sample, file_sa_rate, device=0, **opts):
        """text/bwt: uint8 arrays incl. '$'; bins: (gi, tax, start, end) arrays; sa_sample: uint64."""
        L = _lib.load_library()
        text = np.ascontiguousarray(text, dtype=np.uint8)
        bwt = np.ascontiguousarray(bwt, dtype=np.uint8)
        sa_sample = np.ascontiguousarray(sa_sample, dtype=np.uint64)
        gi, tax, st, en = bins
        barr = (BinStruct * len(gi))()
        for i in range(len(gi)):
            barr[i] = BinStruct(int(gi[i]), int(tax[i]), int(st[i]), int(en[i]))
        h = C.c_void_p()
        o = cls._opts(**opts)
        check(L.mtsvgpu_index_from_parts(_ptr(text), len(text), barr, len(gi), _ptr(bwt), _ptr(sa_sample),
                                         len(sa_sample), file_sa_rate, device, C.byref(o), C.byref(h)))
        return cls(h.value)

    @classmethod
    def build(cls, cat, off, gi, taxid, device=0, **opts):
        """``MGIndex::new`` (src/index.rs:491-582) on the GPU: reference sequences (uint8 concat + uint64
        offsets[n+1], GI and TaxID per sequence) -> device-resident index, ready to bin.  `cat` may be a numpy
        array (host) or an int device pointer to the concatenated bytes (e.g. a torch tensor's data_ptr())."""
        L = _lib.load_library()
        off = np.ascontiguousarray(off, dtype=np.uint64)
        gi = np.ascontiguousarray(gi, dtype=np.uint32)
        taxid = np.ascontiguousarray(taxid, dtype=np.uint32)
        if isinstance(cat, int):
            cat_ptr = C.c_void_p(cat)
        else:
            cat = np.ascontiguousarray(cat, dtype=np.uint8)
            cat_ptr = _ptr(cat)
        h = C.c_void_p()
        o = cls._opts(**opts)
        check(L.mtsvgpu_index_build(cat_ptr, _ptr(off), _ptr(gi), _ptr(taxid), len(gi), device, C.byref(o),
                                    C.byref(h)))
        return cls(h.value)

    def write(self, path, sample_interval=64, sa_sample=32):
        """``write_to_file(&index, path)`` (src/io.rs:125-132): the bincode `.index` of this index, with the
        defaults of mtsv-build's --sample-interval / --sa-sample."""
        check(_lib.load_library().mtsvgpu_index_write(self._h, os.fsencode(path), sample_interval, sa_sample))

    def export_parts(self, sa_sample=32):
        """The MGIndex fields back on the host: dict(text, bins, bwt, sa_sample, sa_rate) — what
        ``from_parts`` (here and in the oracle) takes."""
        info = self.info()
        n = info["text_len"]
        text = np.empty(n, np.uint8)
        bwt = np.empty(n, np.uint8)
        sample = np.empty((n + sa_sample - 1) // sa_sample, np.uint64)
        check(_lib.load_library().mtsvgpu_index_export(self._h, _ptr(text), _ptr(bwt), _ptr(sample), sa_sample))
        return dict(text=text, bwt=bwt, sa_sample=sample, sa_rate=sa_sample)

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            _lib.load_library().mtsvgpu_index_close(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # ---- introspection ----
    def info(self):
        i = InfoStruct()
        check(_lib.load_library().mtsvgpu_index_get_info(self._h, C.byref(i)))
        return {n: getattr(i, n) for n, _ in i._fields_}

    def set_stream(self, cuda_stream_handle):
        """Launch on the given cudaStream_t.  None = the handle's own (non-blocking) stream.  torch reports
        its default stream as handle 0; that is passed as cudaStreamLegacy (1) so that the library's work is
        ordered with torch's kernels and bracketed by torch.cuda.Event on the current stream."""
        if cuda_stream_handle is None:
            h = 0
        else:
            h = int(cuda_stream_handle) or 1
        check(_lib.load_library().mtsvgpu_set_stream(self._h, C.c_void_p(h)))

    def set_profiling(self, on):
        check(_lib.load_library().mtsvgpu_set_profiling(self._h, int(bool(on))))

    def last_batch_stats(self):
        s = StatsStruct()
        check(_lib.load_library().mtsvgpu_last_batch_stats(self._h, C.byref(s)))
        d = {n: int(getattr(s, n)) for n in ("n_queries", "n_seed_slots", "n_seed_hits", "n_candidates",
                                            "n_hits", "window_bytes", "rank_queries", "n_sub_batches", "h2d_bytes",
                                            "n_reads_over_limit", "n_strands_over_hits")}
        d["ms"] = {name: float(s.ms[i]) for i, name in enumerate(_lib.STAGE_NAMES)}
        return d

    # ---- the hot path ----
    def bin_reads(self, reads, params=None, strands=2):
        """Worker closure of run_fastx_pipeline (src/binner.rs:77-131) for a batch of raw reads.
        reads: list of bytes, or (uint8 concat, uint64 offsets).  Returns (hits, hit_off): a
        structured array (HIT_DTYPE) and CSR offsets per read; forward hits first, then
        reverse-complement hits, each in the reference's acceptance order."""
        L = _lib.load_library()
        params = params or Params()
        cat, off = reads if isinstance(reads, tuple) else pack_reads(reads)
        cat = np.ascontiguousarray(cat, dtype=np.uint8)
        off = np.ascontiguousarray(off, dtype=np.uint64)
        n = len(off) - 1
        ps = params.c_struct(strands)
        hp = C.POINTER(HitStruct)()
        op = C.POINTER(C.c_uint64)()
        check(L.mtsvgpu_bin_batch(self._h, _ptr(cat), _ptr(off), n, C.byref(ps), C.byref(hp), C.byref(op)))
        offs = np.ctypeslib.as_array(op, shape=(n + 1,)).copy()
        total = int(offs[-1])
        if total:
            buf = (C.c_uint8 * (total * C.sizeof(HitStruct))).from_address(C.addressof(hp.contents))
            hits = np.frombuffer(buf, dtype=HIT_DTYPE).copy()
        else:
            hits = np.zeros(0, dtype=HIT_DTYPE)
        L.mtsvgpu_free(hp)
        L.mtsvgpu_free(op)
        return hits, offs

    def bin_reads_pinned(self, reads, params=None, strands=2):
        """Like bin_reads but zero-copy on the way out: returns numpy views of the handle's page-locked
        result buffers, valid until the next batch call on this index."""
        L = _lib.load_library()
        params = params or Params()
        cat, off = reads if isinstance(reads, tuple) else pack_reads(reads)
        assert cat.dtype == np.uint8 and off.dtype == np.uint64 and cat.flags.c_contiguous
        n = len(off) - 1
        ps = params.c_struct(strands)
        hp, op, nh = C.c_void_p(), C.c_void_p(), C.c_uint64()
        check(L.mtsvgpu_bin_batch_pinned(self._h, _ptr(cat), _ptr(off), n, C.byref(ps), C.byref(hp),
                                         C.byref(op), C.byref(nh)))
        offs = np.frombuffer((C.c_uint8 * ((n + 1) * 8)).from_address(op.value), dtype=np.uint64)
        total = int(nh.value)
        hits = np.frombuffer((C.c_uint8 * (max(total, 1) * 24)).from_address(hp.value), dtype=HIT_DTYPE)[:total]
        return hits, offs

    def bin_reads_packed(self, packed, off, params=None, strands=2):
        """mtsvgpu_bin_batch_packed: reads as packed records (pack_reads_planes) + their base offsets; results as
        bin_reads_pinned (views of the handle's page-locked buffers)."""
        L = _lib.load_library()
        params = params or Params()
        assert packed.dtype == np.uint8 and off.dtype == np.uint64 and packed.flags.c_contiguous
        n = len(off) - 1
        ps = params.c_struct(strands)
        hp, op, nh = C.c_void_p(), C.c_void_p(), C.c_uint64()
        check(L.mtsvgpu_bin_batch_packed(self._h, _ptr(packed) if len(packed) else None, len(packed), _ptr(off), n,
                                         C.byref(ps), C.byref(hp), C.byref(op), C.byref(nh)))
        offs = np.frombuffer((C.c_uint8 * ((n + 1) * 8)).from_address(op.value), dtype=np.uint64)
        total = int(nh.value)
        hits = np.frombuffer((C.c_uint8 * (max(total, 1) * 24)).from_address(hp.value), dtype=HIT_DTYPE)[:total]
        return hits, offs

    def bin_reads_device(self, d_seqs_ptr, d_seq_off_ptr, n_reads, params=None, strands=2):
        """Device-resident variant: inputs are device pointers (e.g. torch tensors' data_ptr());
        returns (d_hits_ptr, d_hit_off_ptr, n_hits) valid until the next batch call."""
        L = _lib.load_library()
        params = params or Params()
        ps = params.c_struct(strands)
        dh, do, nh = C.c_void_p(), C.c_void_p(), C.c_uint64()
        check(L.mtsvgpu_bin_batch_device(self._h, C.c_void_p(d_seqs_ptr), C.c_void_p(d_seq_off_ptr), n_reads,
                                         C.byref(ps), C.byref(dh), C.byref(do), C.byref(nh)))
        return dh.value, do.value, nh.value

    @staticmethod
    def _pinned_taxhits(tp, op, n_out, n):
        offs = np.frombuffer((C.c_uint8 * ((n + 1) * 8)).from_address(op.value), dtype=np.uint64)
        size = C.sizeof(TaxHitStruct)
        recs = np.frombuffer((C.c_uint8 * (max(n_out, 1) * size)).from_address(tp.value), dtype=TAXHIT_DTYPE)[:n_out]
        return recs, offs

    def assign_reads(self, reads, params=None, strands=2):
        """mtsvgpu_assign_batch_pinned: the default results format computed on the device.  reads as for bin_reads.
        Returns (taxhits, off): a structured array (TAXHIT_DTYPE) and CSR offsets per read.  Read i's records are
        each TaxID it hits on either strand, once, with the minimum edit of those hits, by ascending TaxID.  Copies."""
        L = _lib.load_library()
        params = params or Params()
        cat, off = reads if isinstance(reads, tuple) else pack_reads(reads)
        cat = np.ascontiguousarray(cat, dtype=np.uint8)
        off = np.ascontiguousarray(off, dtype=np.uint64)
        n = len(off) - 1
        ps = params.c_struct(strands)
        tp, op, nt = C.c_void_p(), C.c_void_p(), C.c_uint64()
        check(L.mtsvgpu_assign_batch_pinned(self._h, _ptr(cat), _ptr(off), n, C.byref(ps), C.byref(tp), C.byref(op),
                                            C.byref(nt)))
        recs, offs = self._pinned_taxhits(tp, op, int(nt.value), n)
        return recs.copy(), offs.copy()

    def assign_reads_packed(self, packed, off, params=None, strands=2):
        """mtsvgpu_assign_batch_packed: packed records (pack_reads_planes) + their base offsets in; results as
        assign_reads, but views of the handle's page-locked buffers, valid until the next batch call on this index."""
        L = _lib.load_library()
        params = params or Params()
        assert packed.dtype == np.uint8 and off.dtype == np.uint64 and packed.flags.c_contiguous
        n = len(off) - 1
        ps = params.c_struct(strands)
        tp, op, nt = C.c_void_p(), C.c_void_p(), C.c_uint64()
        check(L.mtsvgpu_assign_batch_packed(self._h, _ptr(packed) if len(packed) else None, len(packed), _ptr(off), n,
                                            C.byref(ps), C.byref(tp), C.byref(op), C.byref(nt)))
        return self._pinned_taxhits(tp, op, int(nt.value), n)

    def assign_reads_device(self, d_seqs_ptr, d_seq_off_ptr, n_reads, params=None, strands=2):
        """mtsvgpu_assign_batch_device: device pointers in, as for bin_reads_device.  Returns (d_taxhits_ptr,
        d_off_ptr, n_taxhits): 8-byte (tax_id, edit) records and n_reads + 1 uint64 offsets, valid until the next
        batch call."""
        L = _lib.load_library()
        params = params or Params()
        ps = params.c_struct(strands)
        dt, do, nt = C.c_void_p(), C.c_void_p(), C.c_uint64()
        check(L.mtsvgpu_assign_batch_device(self._h, C.c_void_p(d_seqs_ptr), C.c_void_p(d_seq_off_ptr), n_reads,
                                            C.byref(ps), C.byref(dt), C.byref(do), C.byref(nt)))
        return dt.value, do.value, nt.value

    def matching_tax_ids(self, sequence, edit_freq=0.13, seed_length=18, seed_gap=15,
                         min_seeds_percent=0.015, max_hits=2000, tune_max_hits=200,
                         max_candidates_checked=None, max_hits_found=None):
        """``MGIndex::matching_tax_ids`` (src/index.rs:258-432): one strand of one read, same argument
        names and meaning (the FM-index view argument of the reference is implicit here)."""
        p = Params(edit_freq, seed_length, seed_gap, min_seeds_percent, max_hits, tune_max_hits,
                   max_candidates_checked, max_hits_found)
        hits, _ = self.bin_reads([bytes(sequence)], p, strands=1)
        return [Hit(int(h["tax_id"]), int(h["gi"]), int(h["offset"]), int(h["edit"])) for h in hits]

    # ---- stage-level entry points (parity tests) ----
    def backward_search(self, patterns):
        """FMIndex::backward_search for equal-length patterns; returns (lower, upper) arrays, 0/0 when
        the result is not Complete."""
        L = _lib.load_library()
        n = len(patterns)
        plen = len(patterns[0]) if n else 1
        assert all(len(p) == plen for p in patterns)
        cat = np.frombuffer(b"".join(bytes(p) for p in patterns), dtype=np.uint8).copy()
        lo = np.zeros(n, np.uint64)
        up = np.zeros(n, np.uint64)
        check(L.mtsvgpu_backward_search(self._h, _ptr(cat), plen, n, _ptr(lo), _ptr(up)))
        return lo, up

    def locate(self, rows):
        L = _lib.load_library()
        rows = np.ascontiguousarray(rows, dtype=np.uint64)
        pos = np.zeros(len(rows), np.uint64)
        check(L.mtsvgpu_locate(self._h, _ptr(rows), len(rows), _ptr(pos)))
        return pos


def edit_distance(patterns, texts, device=0):
    """Aligner::min_edit_distance (src/align.rs:28-85) for a batch of (pattern, text) pairs."""
    L = _lib.load_library()
    pc, po = pack_reads([bytes(p) for p in patterns])
    tc, to = pack_reads([bytes(t) for t in texts])
    out = np.zeros(len(patterns), np.uint32)
    if len(pc) == 0:
        pc = np.zeros(1, np.uint8)
    if len(tc) == 0:
        tc = np.zeros(1, np.uint8)
    check(L.mtsvgpu_edit_distance(device, _ptr(pc), _ptr(po), _ptr(tc), _ptr(to), len(patterns), _ptr(out)))
    return out
