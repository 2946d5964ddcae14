"""ctypes binding of tests/emul/libemul.so: the device per-item logic (csrc/core.cuh) compiled with
g++ and run serially on the CPU.  TEST-ONLY: lets the CPU suite diff the kernels' arithmetic against
the oracle; the product library never uses it."""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "emul", "libemul.so")
_SRC = os.path.join(_HERE, "emul", "emul.cpp")
_CORE = os.path.join(_HERE, "..", "mtsv_tools_b200", "csrc", "core.cuh")
_LIB = None

HIT_DTYPE = np.dtype([("tax_id", "<u4"), ("gi", "<u4"), ("offset", "<u8"), ("edit", "<u4"),
                      ("reserved", "<u4")])


class Bin(C.Structure):
    _fields_ = [("gi", C.c_uint32), ("tax_id", C.c_uint32), ("start", C.c_uint64), ("end", C.c_uint64)]


class Params(C.Structure):
    _fields_ = [("edit_rate", C.c_double), ("seed_size", C.c_uint32), ("seed_gap", C.c_uint32),
                ("min_seed", C.c_double), ("max_hits", C.c_uint64), ("tune_max_hits", C.c_uint64),
                ("max_candidates", C.c_int64), ("max_assignments", C.c_int64),
                ("strands", C.c_uint32), ("reserved", C.c_uint32)]


def lib():
    global _LIB
    if _LIB is not None:
        return _LIB
    stale = not os.path.exists(_SO) or any(os.path.getmtime(s) > os.path.getmtime(_SO)
                                           for s in (_SRC, _CORE))
    if stale:
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wno-unknown-pragmas",
                               "-o", _SO, _SRC])
    L = C.CDLL(_SO)
    vp = C.c_void_p
    L.emul_index_build.restype = vp
    L.emul_index_build.argtypes = [vp, C.c_uint64, vp, C.c_uint64, vp, vp, C.c_uint64, C.c_uint64,
                                   C.c_uint32, C.c_uint32]
    L.emul_index_free.argtypes = [vp]
    L.emul_occ.restype = C.c_uint32
    L.emul_occ.argtypes = [vp, C.c_uint32, C.c_uint32]
    L.emul_locate.restype = C.c_uint32
    L.emul_locate.argtypes = [vp, C.c_uint32]
    L.emul_backward_search.argtypes = [vp, C.c_char_p, C.c_uint32, C.POINTER(C.c_uint32),
                                       C.POINTER(C.c_uint32)]
    L.emul_edit_distance.restype = C.c_uint32
    L.emul_edit_distance.argtypes = [C.c_char_p, C.c_uint32, C.c_uint32, C.c_char_p, C.c_uint32, C.c_int]
    L.emul_edit_distance_k.restype = C.c_uint32
    L.emul_edit_distance_k.argtypes = [C.c_char_p, C.c_uint32, C.c_uint32, C.c_char_p, C.c_uint32, C.c_int,
                                       C.c_uint32]
    L.emul_edit_distance_warp.restype = C.c_uint32
    L.emul_edit_distance_warp.argtypes = [C.c_char_p, C.c_uint32, C.c_uint32, C.c_char_p, C.c_uint32, C.c_uint32,
                                          C.c_int, C.c_uint32, C.c_uint64, C.c_uint32]
    L.emul_edit_distance_warp_wide.restype = C.c_uint32
    L.emul_edit_distance_warp_wide.argtypes = [C.c_char_p, C.c_uint32, C.c_char_p, C.c_uint32, C.c_uint32,
                                               C.c_uint32, C.c_uint64, C.c_uint32]
    L.emul_ssw_scores.argtypes = [C.c_char_p, C.c_uint32, C.c_char_p, C.c_uint32, C.POINTER(C.c_uint32),
                                  C.POINTER(C.c_uint32)]
    L.emul_edit_distance_end.restype = C.c_uint32
    L.emul_edit_distance_end.argtypes = [C.c_char_p, C.c_uint32, C.c_char_p, C.c_uint32, C.c_uint32,
                                         C.POINTER(C.c_uint32)]
    L.emul_sub_batch_bounds.restype = C.c_uint32
    L.emul_sub_batch_bounds.argtypes = [C.c_uint64, C.c_uint64, C.c_int, C.POINTER(C.c_uint64), C.c_uint32]
    L.emul_slice_bounds.restype = C.c_uint32
    L.emul_slice_bounds.argtypes = [C.c_uint64, C.c_uint64, C.c_int, C.c_int, C.POINTER(C.c_uint64), C.c_uint32]
    L.emul_ssw_accepts.restype = C.c_uint32
    L.emul_ssw_accepts.argtypes = [C.c_char_p, C.c_uint32, C.c_char_p, C.c_uint32, C.c_uint32, C.c_uint32,
                                   C.c_uint32, C.c_int]
    L.emul_bin_reads.argtypes = [vp, vp, vp, C.c_uint64, C.POINTER(Params), C.POINTER(vp), C.POINTER(vp)]
    L.emul_free.argtypes = [vp]
    L.emul_packed_words.restype = C.c_uint32
    L.emul_packed_words.argtypes = [C.c_char_p, C.c_uint32, vp, vp, vp]
    _LIB = L
    return L


class EmulIndex:
    def __init__(self, orc_index, sa_rate=1, ktab_k=0):
        """orc_index: oracle.pyoracle.Index (source of text/bins/bwt/samples)."""
        L = lib()
        self.text = np.ascontiguousarray(orc_index.text)
        self.bwt = np.ascontiguousarray(orc_index.bwt)
        self.sample = np.ascontiguousarray(orc_index.sa_sample)
        gi, tax, st, en = orc_index.bins()
        bins = (Bin * len(gi))()
        for i in range(len(gi)):
            bins[i] = Bin(int(gi[i]), int(tax[i]), int(st[i]), int(en[i]))
        self.h = L.emul_index_build(self.text.ctypes.data, len(self.text), bins, len(gi),
                                    self.bwt.ctypes.data, self.sample.ctypes.data, len(self.sample),
                                    orc_index.sa_sample_rate, sa_rate, ktab_k)

    def __del__(self):
        if getattr(self, "h", None):
            lib().emul_index_free(self.h)
            self.h = None

    def occ(self, a, i):
        return lib().emul_occ(self.h, a, i)

    def locate(self, row):
        return lib().emul_locate(self.h, row)

    def backward_search(self, pat):
        lo, cnt = C.c_uint32(), C.c_uint32()
        lib().emul_backward_search(self.h, bytes(pat), len(pat), C.byref(lo), C.byref(cnt))
        return lo.value, cnt.value

    def bin_reads(self, cat, off, params, strands=2):
        L = lib()
        cat = np.ascontiguousarray(cat, dtype=np.uint8)
        off = np.ascontiguousarray(off, dtype=np.uint64)
        n = len(off) - 1
        p = Params(params.edit_rate, params.seed_size, params.seed_gap, params.min_seed, params.max_hits,
                   params.tune_max_hits, params.max_candidates, params.max_assignments, strands, 0)
        hp, op = C.c_void_p(), C.c_void_p()
        rc = L.emul_bin_reads(self.h, cat.ctypes.data, off.ctypes.data, n, C.byref(p), C.byref(hp),
                              C.byref(op))
        assert rc == 0, rc
        offs = np.frombuffer((C.c_uint64 * (n + 1)).from_address(op.value), dtype=np.uint64).copy()
        total = int(offs[-1])
        if total:
            hits = np.frombuffer((C.c_uint8 * (total * 24)).from_address(hp.value), dtype=HIT_DTYPE).copy()
        else:
            hits = np.zeros(0, dtype=HIT_DTYPE)
        L.emul_free(hp)
        L.emul_free(op)
        return hits, offs


def edit_distance(pat, txt, rc=0, ncls=5, k=None):
    """k=None: exact value; otherwise the bounded variant (exact when <= k, anything > k otherwise)."""
    if k is None:
        return int(lib().emul_edit_distance(bytes(pat), len(pat), rc, bytes(txt), len(txt), ncls))
    return int(lib().emul_edit_distance_k(bytes(pat), len(pat), rc, bytes(txt), len(txt), ncls, k))


def edit_distance_warp(pat, txt, k, rc=0, uniform=True, noise=0, seed=1, other_T=0, wide=False):
    """core.cuh::myers_warp (the verifier's fast path, reads <= 256 bases, binner match rule) as one lane
    whose warp votes are perturbed with probability noise/256; exact when the result is <= k."""
    if wide:
        return int(lib().emul_edit_distance_warp_wide(bytes(pat), len(pat), bytes(txt), len(txt), k, noise, seed,
                                                      other_T))
    return int(lib().emul_edit_distance_warp(bytes(pat), len(pat), rc, bytes(txt), len(txt), k, int(uniform),
                                             noise, seed, other_T))


def ssw_accepts(read, txt, k, edit, end_col, which=0):
    """src/index.rs:406 for reads >= 254 bases as the device decides it (core.cuh ssw_word_band /
    ssw_accepts_full).  which: 0 = band then full, 1 = full only, 2 = the band's lower-bound score."""
    return int(lib().emul_ssw_accepts(bytes(read), len(read), bytes(txt), len(txt), k, edit, end_col, which))


def ssw_scores(read, txt):
    """(emulated sw_sse2_word score, textbook SW score) over the full matrices."""
    w, e = C.c_uint32(), C.c_uint32()
    lib().emul_ssw_scores(bytes(read), len(read), bytes(txt), len(txt), C.byref(w), C.byref(e))
    return w.value, e.value


def edit_distance_end(pat, txt, k):
    """(bounded edit distance, number of text columns consumed by the first best alignment)."""
    ec = C.c_uint32()
    e = lib().emul_edit_distance_end(bytes(pat), len(pat), bytes(txt), len(txt), k, C.byref(ec))
    return int(e), ec.value


def sub_batch_bounds(n_reads, step, ramp):
    """Read boundaries of the device slices of one batch call (core.cuh::sub_batch_bounds)."""
    buf = (C.c_uint64 * 4096)()
    n = lib().emul_sub_batch_bounds(n_reads, step, int(ramp), buf, 4096)
    return [int(buf[i]) for i in range(min(n, 4096))]


def slice_bounds(n_reads, step, host_input, two_lanes):
    """Read boundaries of the slices one batch call computes (core.cuh::slice_bounds); step 0 = the default."""
    buf = (C.c_uint64 * 4096)()
    n = lib().emul_slice_bounds(n_reads, step, int(host_input), int(two_lanes), buf, 4096)
    return [int(buf[i]) for i in range(min(n, 4096))]


def packed_words(seq, record=None):
    """(planes unpacked from the read's packed record, planes encoded from its raw bytes): two uint64 arrays of
    3 words per 64 bases.  record: bytes of a record made by another packer (None: core.cuh::pack_read)."""
    import numpy as np
    seq = bytes(seq)
    W = (len(seq) + 63) // 64
    a = np.zeros(3 * max(W, 1), np.uint64)
    b = np.zeros(3 * max(W, 1), np.uint64)
    rec = None
    if record is not None:
        rec = np.frombuffer(bytes(record), dtype=np.uint8).copy()
    lib().emul_packed_words(seq, len(seq), rec.ctypes.data if rec is not None and len(rec) else None,
                            a.ctypes.data, b.ctypes.data)
    return a[:3 * W], b[:3 * W]
