"""Pins the oracle (CPU restatement, oracle/) against every known-answer vector the reference's own
tests hold for this path, plus self-consistency checks for the pieces the reference never tests
(SURVEY.md §4 / §8c).  No GPU needed."""
import os
import random

import numpy as np
import pytest

HAY = b"ACGACTAGTTATAAAAATTCNACTCCANTTAGCTCCCTACTTTCCGAGAG"

# src/align.rs:100-170 — the nine exact edit distances
ALIGN_KATS = [
    (b"TACGTCAGC", b"AACCCTATGTCATGCCTTGGA", 2),
    (HAY, HAY, 0),
    (b"AAAAAT", HAY, 0),
    (b"", HAY, 0),
    (b"*********", HAY, 9),
    (b"ACGT", b"ACGA", 1),
    (b"ANNGTTCNGNT", HAY, 5),
    (b"***GTTATAA", HAY, 3),
    (b"GTTATAA***", HAY, 3),
]


@pytest.mark.parametrize("needle,hay,want", ALIGN_KATS)
def test_edit_distance_kats(oracle, needle, hay, want):
    assert oracle.min_edit_distance(needle, hay) == want


def test_candidate_indices_kats(oracle):
    # src/index.rs:794-839 seed_hits_success
    s, e = oracle.candidate_indices(110, 1, 100, 200, 50, 3)
    assert s < e and s >= 100 and e <= 200 and e - s >= 50 + 2 * 3
    assert (s, e) == (106, 162)
    s, e = oracle.candidate_indices(180, 25, 100, 200, 50, 3)
    assert s < e and s >= 100 and e <= 200 and e - s >= 50 - 3
    assert (s, e) == (152, 200)
    # src/index.rs:841-857 seed_hits_fail (unwrap on None panics)
    assert oracle.candidate_indices(90, 1, 100, 200, 50, 3) is None


def test_reference_candidate_merge(oracle):
    # src/index.rs:721-769: second hit (115, 3) merges, start unchanged, end = second window's end
    s1, e1 = oracle.candidate_indices(110, 1, 100, 300, 50, 3)
    s2, e2 = oracle.candidate_indices(115, 3, 100, 300, 50, 3)
    assert (s1 <= s2 < e1) or (s1 < e2 <= e1)
    assert min(s1, s2) == s1 and max(e1, e2) == e2


def test_write_assignments_kats(oracle):
    # src/binner.rs:439-472
    hits = [(2, 10, 3, 7), (2, 11, 8, 4), (5, 12, 1, 9)]
    assert oracle.format_assignments("R1_1_0_0", hits, False) == "R1_1_0_0:2=4,5=9\n"
    hits = [(2, 10, 3, 7), (2, 10, 3, 4), (2, 11, 8, 6), (5, 12, 1, 9)]
    assert oracle.format_assignments("R1_1_0_0", hits, True) == "R1_1_0_0:2-10-3=4,2-11-8=6,5-12-1=9\n"
    assert oracle.format_assignments("R1_1_0_0", [], False) == ""


def test_python_writer_matches_oracle(oracle):
    from mtsv_tools_b200 import Hit, format_assignments
    rng = random.Random(0)
    for _ in range(200):
        hits = [(rng.randint(1, 5), rng.randint(1, 3), rng.randint(0, 4), rng.randint(0, 9))
                for _ in range(rng.randint(0, 8))]
        for long in (False, True):
            assert format_assignments("r", [Hit(*h) for h in hits], long) == \
                oracle.format_assignments("r", hits, long)


def test_suffix_array_vs_naive(oracle):
    rng = random.Random(1)
    L = oracle.lib()
    for _ in range(150):
        n = rng.randint(1, 200)
        alpha = rng.choice([b"ACGT", b"ACGTN", b"AC", b"A"])
        t = bytes(rng.choice(alpha) for _ in range(n)) + b"$"
        arr = np.frombuffer(t, dtype=np.uint8).copy()
        sa = np.zeros(len(t), np.uint64)
        assert L.orc_suffix_array(arr.ctypes.data, len(t), sa.ctypes.data) == 0
        assert list(sa) == sorted(range(len(t)), key=lambda i: t[i:])


def test_fm_index_vs_bruteforce(oracle):
    """backward_search + locate == naive substring search (5-letter alphabet incl. N, as the
    reference's random_database, src/index.rs:604-642)."""
    rng = random.Random(2)
    for _ in range(40):
        nseq = rng.randint(1, 4)
        seqs = [bytes(rng.choice(b"ACGTN") for _ in range(rng.randint(1, 300))) for _ in range(nseq)]
        k, s = rng.choice([1, 3, 8, 64]), rng.choice([1, 2, 5, 32])
        ix = oracle.Index.build(seqs, list(range(nseq)), [rng.randint(1, 5) for _ in range(nseq)], k, s)
        text = bytes(ix.text)
        for _ in range(60):
            m = rng.randint(1, 8)
            if rng.random() < 0.5:
                st = rng.randrange(0, len(text) - 1)
                pat = text[st:st + m].rstrip(b"$")
                if not pat:
                    continue
            else:
                pat = bytes(rng.choice(b"ACGTN") for _ in range(m))
            r, lo, up, _ = ix.backward_search(pat)
            want = sorted(i for i in range(len(text)) if text.startswith(pat, i))
            if r == 2:
                assert sorted(ix.locate(row)[0] for row in range(lo, up)) == want
            else:
                assert not want


def test_index_bincode_roundtrip(oracle, tmp_path):
    rng = random.Random(3)
    seqs = [bytes(rng.choice(b"ACGT" * 12 + b"Nacgtx") for _ in range(rng.randint(200, 400))) for _ in range(5)]
    ix = oracle.Index.build(seqs, [7, 8, 9, 10, 11], [30, 10, 20, 10, 30], 16, 8)
    gi, tax, st, en = ix.bins()
    # BTreeMap order: TaxID ascending, file order within a TaxID (src/io.rs:135-150)
    assert list(tax) == [10, 10, 20, 30, 30] and list(gi) == [8, 10, 9, 7, 11]
    text = bytes(ix.text)
    assert text.endswith(b"$") and set(text[:-1]) <= set(b"ACGTN")  # src/index.rs:543-555
    p = str(tmp_path / "t.index")
    ix.write(p)
    # layout check: u64 n, text, u64 nbins, 24-byte bins ... (SURVEY §8b)
    raw = open(p, "rb").read()
    n = int.from_bytes(raw[:8], "little")
    assert n == len(text) and raw[8:8 + n] == text
    nb = int.from_bytes(raw[8 + n:16 + n], "little")
    assert nb == 5
    ix2 = oracle.Index.read(p)
    assert bytes(ix2.text) == text and bytes(ix2.bwt) == bytes(ix.bwt)
    assert np.array_equal(ix2.sa_sample, ix.sa_sample) and ix2.sa_sample_rate == 8
    reads = [text[40:120], text[300:380], text[500:580]]
    h1, o1 = ix.bin_reads(reads, oracle.default_params(seed_size=10, seed_gap=5))
    h2, o2 = ix2.bin_reads(reads, oracle.default_params(seed_size=10, seed_gap=5))
    assert np.array_equal(h1, h2) and np.array_equal(o1, o2) and len(h1) >= 2


def test_ssw_reference_equals_restated_sw(oracle):
    """The reference's ssw.c (its scores stored in tests/golden/ssw_scores.npz, and oracle/_ref/libssw_ref.so itself
    when it is built) vs the textbook restatement, reads <= 253 bp (SURVEY fact 3), and the theorem
    ed <= k  =>  SW >= L - 2k that lets the GPU drop the SW stage."""
    from tests.golden.make_ssw_golden import PATH, short_sw_pairs
    scores = np.load(PATH)["short_scores"]
    have_ref = oracle.ssw_ref_available()
    for i, (read, ref) in enumerate(short_sw_pairs()):
        L = len(read)
        a = int(scores[i])
        if have_ref:
            assert oracle.ssw_score(read, ref, 1) == a
        b = oracle.ssw_score(read, ref, 2)
        assert a == b
        ed = oracle.min_edit_distance(read.replace(b"N", b"."), ref)
        assert a >= L - 2 * ed


# SURVEY.md appendix E: vectors from an independent Python restatement (naive substring search,
# textbook SW, full DP).  Flags: seed-size 10, seed-interval 5 unless stated; headers GI-TAXID.
V1 = [(11, 7, b"TAGGCGTCGATGCCGATCCCACGGATGATAACCGATACTCGACATCCGTCACGACCGGCTGAAATATCAGCATAATGTCGACATCGCCCCGCAACATCAGTATTCCCAGGCTCCCTTGAA"),
      (12, 9, b"TCCCCGGCAGTAGAACGAGTGTGTGGTTAGTACGCAAAACTTCGGCGGTAGGATCCACGCGTCACAAGTGACATCCGGCGAAACTACGCTTTAGATGAGTTAGGTGCTAATAACAAGCATTTATCCGCTCTCCCCTACAA")]
V2 = [(21, 5, b"AACCGCCGGACTTTTGGATTCTAAAGGTTTCAGCCGCTGTTCTAAGCTTATTAGCTGTACCTGCAGATGCGATGCGCACTATATCATCAGCGCTCGGGTAGCTAGTTCGG"),
      (22, 5, b"CTTATGCTTCGTGCTGACCAATCGACCAAGAAGCCGCTGTTCTAAGCTTATTAGCAGTACCTGCAGATGCGATGCGCACGGCGGGGTAATTGCGACGACCCGCGGAACCA")]
V3 = [(31, 3, b"CAACTTTACCCTAGACAAGCGGCGCGTAGCGTCCTATCGCCGGGAGTCTAACTCAAATCATATGGCCCATCGCAGTGCGTGAGTTTTATTCAGCCCACCC"),
      (32, 4, b"CAACAAGAGATCGAAATAGTAATCTGTCTCTCTGCTATGATGAGACAATGTCCGTACACTCACTACTTGTTGTACAGTAGATATTCAACCTTAGTGGTTG")]
V4 = [(41, 8, b"GTACCTTAGGGTGGGCGAATTTTCTCCGTGAAGCCGCTGTTCTAAGCTTANTAGCTGTACCTGCAGATGCGATGCGCACGTTAAGTACACGACAGTCCGGGTCCTACCCT")]
V5 = [(51, 2, b"ACCAAGTGGCTATCTCACCGCATCCTGCGACATCCTGCGACATCCTGCGACATCCTGCGACATCCTGCGACATCCTGCGAAAGCGCTAGGTGAGAGCAAC")]
APPENDIX_E = [
    ("V1a", V1, b"TACGCAAAACTTCGGCGGTAGGATCCACGCGTCACAAGTGACATCCGGCG", {}, "r:9=0", "r:9-12-23=0"),
    ("V1b", V1, b"AGCCGGTCGTGACGGATGTCGAGTATCGGTTATCATCCGTGGGATCGGCA", {}, "r:7=0", "r:7-11-3=0"),
    ("V2", V2, b"AAGCCGCTGTTCTAAGCTTATTAGCTGTACCTGCAGATGCGATGCGCACG", {}, "r:5=2", "r:5-21-23=2"),
    ("V3", V3, b"CAACAAGAGATCGAAATAGTAATCTGTCTCTCTGCTATGATGAGACAATG", {}, "r:4=0", "r:4-32-0=0"),
    ("V4", V4, b"AAGCCGCTGTTCTAAGCTTANTAGCTGTACCTGCAGATGCGATGCGCACG", {}, "r:8=1", "r:8-41-23=1"),
    ("V5", V5, b"CGGTTCATCCTGCGACATCCTGCGACATCCTGCGACATCCTGCGAAAAAG", dict(tune_max_hits=2, max_hits=5),
     "r:2=5", "r:2-51-0=5"),
]


@pytest.mark.parametrize("name,refs,read,flags,want,want_long", APPENDIX_E, ids=[v[0] for v in APPENDIX_E])
def test_appendix_e_vectors(oracle, name, refs, read, flags, want, want_long):
    ix = oracle.Index.build([r[2] for r in refs], [r[0] for r in refs], [r[1] for r in refs])
    p = oracle.default_params(seed_size=10, seed_gap=5, **flags)
    hits, offs = ix.bin_reads([read], p)
    assert "".join(oracle.results_lines(["r"], hits, offs, False)).strip() == want
    assert "".join(oracle.results_lines(["r"], hits, offs, True)).strip() == want_long


def test_golden_fixture_matches_oracle(oracle):
    """tests/golden/cfg1_small.npz was produced by tests/golden/make_golden.py with this oracle; it
    pins the oracle against silent drift and is what the GPU tests compare with at run time."""
    path = os.path.join(os.path.dirname(__file__), "golden", "cfg1_small.npz")
    g = np.load(path)
    from tests.golden.make_golden import build_case
    ix, reads, params = build_case(oracle)
    hits, offs = ix.bin_reads(reads, params, threads=4)
    assert np.array_equal(offs, g["hit_off"])
    for f in ("tax_id", "gi", "offset", "edit"):
        assert np.array_equal(hits[f], g[f])
