"""Generates tests/golden/ssw_scores.npz: what the reference's own ssw.c answers for the inputs of the tests that
pin the 16-bit SW kernel (reads of 254 bases and more).  Run from the repo root:
    python -m tests.golden.make_ssw_golden

ssw.c is not part of this repository, so the tests that compared with it now compare with these stored answers
(and still with ssw.c itself when oracle/_ref/libssw_ref.so has been built from a reference tree).  The answers
are computed by tests/emul, the CPU build of core.cuh, whose cell-for-cell emulation of ssw.c's sw_sse2_word was
held equal to ssw.c by these same tests; the generator refuses to write them unless the oracle's independent
textbook SW agrees wherever ssw.c is textbook SW (scores below 254) and the GPU suite checks the device against
them.  Contents:
  short_scores      ssw.c score of each short_sw_pairs() pair (reads <= 253 bases: the 8-bit kernel)
  long_scores       ssw.c score of each long_sw_pairs() pair (reads >= 254 bases)
  emul<i>_*, gpu<i>_*  hit_off / tax_id / gi / offset / edit of bin_reads with ssw.c as the SW of the oracle, for
                    long_read_batch(EMUL_CASES[i]) and long_read_batch(GPU_CASES[i])"""
import os
import random

import numpy as np

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "ssw_scores.npz")

# (read_len, edit_rate, edit_frac, reads): tests/test_emul_parity.py and tests/test_gpu_parity.py
EMUL_CASES = ((254, 0.13, 0.11, 150), (300, 0.13, 0.12, 150), (300, 0.05, 0.045, 150), (420, 0.10, 0.09, 150))
GPU_CASES = ((254, 0.13, 0.11, 300), (300, 0.13, 0.12, 400), (300, 0.05, 0.045, 300), (420, 0.10, 0.09, 300),
             (700, 0.13, 0.10, 200), (1500, 0.13, 0.08, 100), (3000, 0.13, 0.05, 60))
FIELDS = ("tax_id", "gi", "offset", "edit")


def small_ref():
    from mtsv_tools_b200 import synth
    return synth.make_reference(8, 20000, seed=1, n_frac=0.002, shared_frac=0.1, seqs_per_taxid=2)


def short_sw_pairs():
    """(read, reference window) pairs of 15-253 bases, edited copies of each other."""
    rng = random.Random(4)
    out = []
    for _ in range(400):
        L = rng.randint(15, 253)
        read = bytes(rng.choice(b"ACGTN" if rng.random() < 0.2 else b"ACGT") for _ in range(L))
        s = list(read)
        for _ in range(rng.randint(0, L // 4)):
            i = rng.randrange(len(s))
            r = rng.random()
            if r < 0.5:
                s[i] = rng.choice(b"ACGTN")
            elif r < 0.75:
                s.insert(i, rng.choice(b"ACGT"))
            elif len(s) > 1:
                del s[i]
        ref = bytes(rng.choice(b"ACGT") for _ in range(rng.randint(0, 20))) + bytes(s) + \
            bytes(rng.choice(b"ACGT") for _ in range(rng.randint(0, 20)))
        out.append((read, ref))
    return out


def long_sw_pairs():
    from tests.test_emul_parity import _long_pair
    rng = random.Random(7)
    return [_long_pair(rng) for _ in range(1200)]


def long_read_batch(oracle, ref_cat, case, ragged):
    """Packed reads of one case: edited long reads, reads on the SW threshold and (ragged) 50 short reads."""
    from tests.test_emul_parity import _borderline_long_reads, _long_reads
    read_len, rate, frac, n = case
    rl = _long_reads(ref_cat, n, read_len, seed=read_len + int(rate * 100), edit_frac=frac)
    k = int(np.ceil(read_len * rate))
    rl += _borderline_long_reads(ref_cat, n, read_len, k, seed=read_len)
    if ragged:
        rl += [r[:rng_len] for r, rng_len in zip(rl[:50], range(100, 150))]  # ragged: short reads in the batch
    return oracle.pack_seqs(rl)


def expected_hits(golden, prefix):
    """(hit offsets, hits with the fields FIELDS) stored under `prefix`."""
    cols = [golden[prefix + "_" + f] for f in FIELDS]
    hits = np.zeros(len(cols[0]), dtype=[(f, c.dtype) for f, c in zip(FIELDS, cols)])
    for f, c in zip(FIELDS, cols):
        hits[f] = c
    return golden[prefix + "_hit_off"], hits


def _ssw_c_score(emul, read, ref):
    w, e = emul.ssw_scores(read, ref)
    return w if e >= 254 else e  # ssw_align re-runs sw_sse2_word once the 8-bit score reaches 255 - bias


def main():
    from oracle import pyoracle
    from tests import emul_api
    pyoracle.lib()
    out = {}
    short = []
    for read, ref in short_sw_pairs():
        s = _ssw_c_score(emul_api, read, ref)
        assert s == pyoracle.ssw_score(read, ref, 2), (read, ref)
        short.append(s)
    out["short_scores"] = np.array(short, dtype=np.uint16)
    out["long_scores"] = np.array([_ssw_c_score(emul_api, r, t) for r, t in long_sw_pairs()], dtype=np.uint16)
    cat, off, gi, tax = small_ref()
    ix = pyoracle.Index.build((cat, off), gi, tax, 64, 32)
    e = emul_api.EmulIndex(ix, sa_rate=1, ktab_k=6)
    n_changed = 0
    for prefix, cases, ragged in (("emul", EMUL_CASES, False), ("gpu", GPU_CASES, True)):
        for i, case in enumerate(cases):
            reads = long_read_batch(pyoracle, cat, case, ragged)
            p = pyoracle.default_params(edit_rate=case[1])
            hits, offs = e.bin_reads(reads[0], reads[1], p)
            h_sw, o_sw = ix.bin_reads(reads, p, threads=8)  # textbook SW: differs only on reads of 254 bases and more
            short_reads = np.nonzero(np.diff(reads[1]) < 254)[0]
            assert np.array_equal(np.diff(offs)[short_reads], np.diff(o_sw)[short_reads])
            n_changed += int(np.sum(np.diff(offs) != np.diff(o_sw)))
            out["%s%d_hit_off" % (prefix, i)] = offs
            for f in FIELDS:
                out["%s%d_%s" % (prefix, i, f)] = hits[f]
    assert n_changed > 0
    np.savez_compressed(PATH, **out)
    print("wrote", PATH, "reads whose hits differ from textbook SW:", n_changed)


if __name__ == "__main__":
    main()
