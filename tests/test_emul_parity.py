"""CPU differential tests: the per-item device logic (csrc/core.cuh compiled with g++, run serially by
tests/emul/) against the oracle.  Covers the arithmetic of every stage — packed-BWT rank, k-mer
table, backward search, LF locate / dense SA, seed rule replay, windows + coalesce, ranking,
Myers bit-vector edit distance, per-TaxID selection — without a GPU.  The GPU suite
(test_gpu_parity.py) repeats the same comparisons through the C ABI on the real kernels."""
import random

import numpy as np
import pytest

from mtsv_tools_b200 import synth


def _same(h1, o1, h2, o2):
    assert np.array_equal(o1, o2)
    for f in ("tax_id", "gi", "offset", "edit"):
        assert np.array_equal(h1[f], h2[f]), f


@pytest.fixture(scope="module")
def small_ref():
    return synth.make_reference(8, 20000, seed=1, n_frac=0.002, shared_frac=0.1, seqs_per_taxid=2)


@pytest.fixture(scope="module")
def small_index(oracle, small_ref):
    cat, off, gi, tax = small_ref
    return oracle.Index.build((cat, off), gi, tax, 64, 32)


def test_rank_symbol_locate(oracle, emul, small_index):
    ix = small_index
    rng = random.Random(0)
    n = len(ix)
    codes = {0: ord("A"), 1: ord("C"), 2: ord("G"), 3: ord("T"), 4: ord("N")}
    for sa_rate in (1, 4, 32):
        e = emul.EmulIndex(ix, sa_rate=sa_rate, ktab_k=0)
        for _ in range(3000):
            i = rng.randint(1, n)
            a = rng.randint(0, 4)
            assert e.occ(a, i) == ix.occ(i - 1, codes[a])
        for _ in range(2000):
            row = rng.randrange(n)
            assert e.locate(row) == ix.locate(row)[0]


@pytest.mark.parametrize("ktab_k", [0, 1, 4, 7, 10])
def test_backward_search(oracle, emul, small_index, ktab_k):
    ix = small_index
    e = emul.EmulIndex(ix, sa_rate=1, ktab_k=ktab_k)
    text = bytes(ix.text)
    rng = random.Random(ktab_k)
    n_direct = 0
    for _ in range(1500):
        m = rng.randint(max(1, ktab_k), 40 if ktab_k == 10 else 24)  # > k + 8: the comparison continues in the text
        if rng.random() < 0.6:
            st = rng.randrange(0, len(text) - m - 1)
            pat = bytearray(text[st:st + m])
            if rng.random() < 0.3:
                pat[rng.randrange(m)] = rng.choice(b"ACGTN")
            pat = bytes(pat)
        else:
            pat = bytes(rng.choice(b"ACGTN") for _ in range(m))
        r, lo, up, _ = ix.backward_search(pat)
        elo, ecnt = e.backward_search(pat)
        if r == 2 and ecnt & 0x80000000:
            # direct entry of the k-mer table (core.cuh): a seed that ends in a unique k-mer comes back as its
            # text position, without rank queries
            n_direct += 1
            assert up - lo == 1 and ecnt == 0x80000001 and ix.locate(lo)[0] == elo, pat
        elif r == 2:
            assert (elo, ecnt) == (lo, up - lo), pat
        else:
            assert ecnt == 0
    assert n_direct > 100 or ktab_k < 10  # (a 160 kbp text: its 10-mers are mostly unique, shorter ones are not)


def test_edit_distance_fuzz(oracle, emul):
    rng = random.Random(5)
    for _ in range(1500):
        L = rng.randint(1, 300)
        alpha = b"ACGTN" if rng.random() < 0.5 else b"ACGT"
        p = bytes(rng.choice(alpha) for _ in range(L))
        if rng.random() < 0.6:
            s = list(p)
            for _ in range(rng.randint(0, 20)):
                i = rng.randrange(len(s))
                r = rng.random()
                if r < 0.4:
                    s[i] = rng.choice(b"ACGT")
                elif r < 0.7:
                    s.insert(i, rng.choice(b"ACGT"))
                elif len(s) > 1:
                    del s[i]
            tx = bytes(rng.choice(b"ACGT") for _ in range(rng.randint(0, 30))) + bytes(s) + \
                bytes(rng.choice(b"ACGT") for _ in range(rng.randint(0, 30)))
        else:
            tx = bytes(rng.choice(alpha) for _ in range(rng.randint(1, 400)))
        assert oracle.min_edit_distance(p, tx) == emul.edit_distance(p, tx, 0, 5)
        assert oracle.min_edit_distance(p.replace(b"N", b"."), tx) == emul.edit_distance(p, tx, 0, 4)


def test_edit_distance_warp_fuzz(oracle, emul):
    """The warp-uniform verifier recurrence (core.cuh::myers_warp) against the full DP: exact whenever the
    distance is within the budget, above the budget otherwise — with the votes of the other lanes perturbed
    (early activation, late drops, a longer window elsewhere in the warp) and for ragged lengths."""
    rng = random.Random(11)
    n_within = 0
    for it in range(4000):
        L = rng.randint(1, 256)
        alpha = b"ACGTN" if rng.random() < 0.3 else b"ACGT"
        p = bytes(rng.choice(alpha) for _ in range(L))
        mode = rng.random()
        if mode < 0.7:
            s = list(p)
            for _ in range(rng.randint(0, 30)):
                i = rng.randrange(len(s))
                r = rng.random()
                if r < 0.4:
                    s[i] = rng.choice(b"ACGTN")
                elif r < 0.7:
                    s.insert(i, rng.choice(b"ACGT"))
                elif len(s) > 1:
                    del s[i]
            tx = bytes(rng.choice(b"ACGT") for _ in range(rng.randint(0, 60))) + bytes(s) + \
                bytes(rng.choice(b"ACGT") for _ in range(rng.randint(0, 60)))
        else:
            tx = bytes(rng.choice(alpha) for _ in range(rng.randint(0, 500)))
        k = rng.choice([0, 1, 3, 10, 20, 33, 50, 64, 65, 100, 128, 129, 255, 400])
        want = oracle.min_edit_distance(p.replace(b"N", b"."), tx) if tx else L
        n_within += want <= k
        for uniform in (True, False):
            noise = rng.choice([0, 0, 8, 64, 200])
            other_T = rng.choice([0, 0, len(tx) + rng.randint(1, 100)])
            got = emul.edit_distance_warp(p, tx, k, 0, uniform, noise, rng.getrandbits(60), other_T)
            assert (got == want) if want <= k else (got > k), (it, L, len(tx), k, uniform, noise, other_T, got, want)
        got = emul.edit_distance_warp(p, tx, k, wide=True, noise=rng.choice([0, 16, 128]), seed=rng.getrandbits(60),
                                      other_T=rng.choice([0, len(tx) + 37]))
        assert (got == want) if want <= k else (got > k), (it, "wide", L, len(tx), k, got, want)
    assert n_within > 1000


def _long_pair(rng, max_edits=40):
    L = rng.randint(254, 520)
    read = [rng.choice(b"ACGT") for _ in range(L)]
    if rng.random() < 0.2:
        for _ in range(rng.randint(1, 5)):
            read[rng.randrange(L)] = ord("N")
    s = list(read)
    for _ in range(rng.randint(0, max_edits)):
        i = rng.randrange(len(s))
        r = rng.random()
        if r < 0.3:
            s[i] = rng.choice(b"ACGTN")
        elif r < 0.65:  # runs of inserted reference bases / deleted read bases: gaps that cross SIMD lane rows
            for _ in range(rng.randint(1, 4)):
                s.insert(i, rng.choice(b"ACGT"))
        else:
            for _ in range(rng.randint(1, 4)):
                if len(s) > 1 and i < len(s):
                    del s[i]
    tx = bytes(rng.choice(b"ACGT") for _ in range(rng.randint(0, 50))) + bytes(s) + \
        bytes(rng.choice(b"ACGT") for _ in range(rng.randint(0, 50)))
    return bytes(read), tx


def test_ssw_word_kernel_emulation(oracle, emul):
    """Reads >= 254 bases: ssw_align falls to sw_sse2_word once SW reaches 254, and that kernel is not textbook
    SW (core.cuh).  The cell-for-cell emulation must reproduce the reference's own ssw.c score (stored in
    tests/golden/ssw_scores.npz, and ssw.c itself when oracle/_ref is built); the banded lower bound must never exceed
    it; the device's accept decision must equal `score >= L - 2k`."""
    from tests.golden.make_ssw_golden import PATH, long_sw_pairs
    scores = np.load(PATH)["long_scores"]
    have_ref = oracle.ssw_ref_available()
    n_word = n_diff = n_band_ok = n_band_short = 0
    for it, (read, tx) in enumerate(long_sw_pairs()):
        L = len(read)
        ref_score = int(scores[it])
        if have_ref:
            assert oracle.ssw_score(read, tx, 1) == ref_score, it
        w, e = emul.ssw_scores(read, tx)
        assert (w if e >= 254 else e) == ref_score, (it, L, len(tx), ref_score, w, e)
        assert w <= e
        n_word += e >= 254
        n_diff += w != e
        # decision as the device takes it, for budgets around the candidate's own edit distance
        ed, end_col = emul.edit_distance_end(read, tx, L)
        for k in {ed, ed + 1, ed + 3, (L - ref_score) // 2, (L - ref_score + 1) // 2, int(L * 0.13) + 1}:
            if ed > k or 2 * k > L:
                continue
            want = ref_score >= L - 2 * k
            assert bool(emul.ssw_accepts(read, tx, k, ed, end_col, 0)) == want, (it, L, k, ed, ref_score)
            assert bool(emul.ssw_accepts(read, tx, k, ed, end_col, 1)) == want
            if ed + 1 <= 127:
                b = emul.ssw_accepts(read, tx, 0, ed, end_col, 2)  # k = 0: threshold L, never reached early
                assert b <= w, (it, b, w)
                n_band_ok += b >= L - 2 * ed
                n_band_short += b < L - 2 * ed
    assert n_word > 500 and n_diff > 20
    assert n_band_ok > 10 * max(1, n_band_short)  # the band settles nearly every case without the full matrices


def _long_reads(ref_cat, n, read_len, seed, edit_frac):
    """Reads of `read_len` bases sampled from the reference and edited at about edit_frac per base with
    substitutions and RUNS of inserted / deleted bases (what trips sw_sse2_word), half reverse-complemented."""
    rng = random.Random(seed)
    out = []
    text = bytes(ref_cat)
    for _ in range(n):
        st = rng.randrange(0, len(text) - 2 * read_len)
        s = list(text[st:st + read_len + 60])
        n_ed = max(0, int(rng.gauss(edit_frac * read_len, 0.25 * edit_frac * read_len)))
        done = 0
        while done < n_ed:
            i = rng.randrange(5, read_len - 5)
            r = rng.random()
            if r < 0.4:
                s[i] = rng.choice(b"ACGT")
                done += 1
            elif r < 0.7:
                run = rng.randint(1, 4)
                for _ in range(run):
                    s.insert(i, rng.choice(b"ACGT"))
                done += run
            else:
                run = rng.randint(1, 4)
                del s[i:i + run]
                done += run
        read = bytes(s[:read_len])
        if rng.random() < 0.5:
            read = synth.revcomp(read)
        out.append(read)
    return out


def _borderline_long_reads(ref_cat, n, read_len, k, seed):
    """Reads built to sit on the SW threshold: exactly k or k-1 edits, none of them a deleted reference base
    (SW = L - 2*edits then), with a run of 2-4 inserted bases laid across a SIMD lane boundary row of
    sw_sse2_word (row l * ceil(L/8)) — the alignments its truncated lazy-F loop under-scores."""
    rng = random.Random(seed)
    text = bytes(ref_cat)
    seg = (read_len + 7) // 8
    out = []
    other = {65: b"CGT", 67: b"AGT", 71: b"ACT", 84: b"ACG"}
    while len(out) < n:
        a = rng.randint(2, 4)
        st = rng.randrange(0, len(text) - 2 * read_len)
        base = list(text[st:st + read_len - a])
        if any(c not in other for c in base):
            continue
        lane = rng.randint(1, 7)
        pos = lane * seg - rng.randint(1, a - 1)  # the run covers rows pos .. pos+a-1, crossing row lane*seg
        ins = [rng.choice(b"ACGT") for _ in range(a)]
        s = base[:pos] + ins + base[pos:]
        assert len(s) == read_len
        n_sub = k - a - rng.randint(0, 1)
        for i in rng.sample([i for i in range(3, read_len - 3) if not pos - 2 <= i < pos + a + 2], max(0, n_sub)):
            s[i] = rng.choice(other[s[i]])
        read = bytes(s)
        if rng.random() < 0.5:
            read = synth.revcomp(read)
        out.append(read)
    return out


def test_pipeline_reads_of_254_bases_and_more(oracle, emul, small_ref, small_index):
    """What the oracle answers with the reference's own ssw.c (16-bit kernel for these reads; stored in
    tests/golden/ssw_scores.npz, and ssw.c itself when oracle/_ref is built): the per-item device logic must reject
    exactly the candidates it rejects (edit distance within budget but SSW score below L - 2k)."""
    from tests.golden.make_ssw_golden import EMUL_CASES, PATH, expected_hits, long_read_batch
    golden = np.load(PATH)
    L = oracle.lib()
    n_changed = 0
    for i, case in enumerate(EMUL_CASES):
        reads = long_read_batch(oracle, small_ref[0], case, ragged=False)
        p = oracle.default_params(edit_rate=case[1])
        o1, h1 = expected_hits(golden, "emul%d" % i)
        if oracle.ssw_ref_available():
            _same(h1, o1, *small_index.bin_reads(reads, p, threads=4))  # real ssw.c
        e = emul.EmulIndex(small_index, sa_rate=1, ktab_k=6)
        h2, o2 = e.bin_reads(reads[0], reads[1], p)
        _same(h1, o1, h2, o2)
        assert len(h1) > 40
        L.orc_set_ssw_kind(2)  # textbook SW: "edit <= k" alone
        try:
            h3, o3 = small_index.bin_reads(reads, p, threads=4)
        finally:
            L.orc_set_ssw_kind(0)
        n_changed += int(np.sum((o3[1:] - o3[:-1]) != (o1[1:] - o1[:-1])))
    assert n_changed > 0, "no read exercised the 16-bit kernel's deviation; make the cases harder"


def test_slice_schedule(emul):
    """The slices of one batch call: cover the reads exactly once, in order, never longer than the step;
    with host input short first and last slices (the call lasts upload + first upload + last compute)."""
    rng = random.Random(3)
    for _ in range(2000):
        n = rng.choice([0, 1, 2, rng.randint(0, 5000), rng.randint(0, 3 << 20), rng.randint(0, 40 << 20)])
        step = rng.choice([1, 7, 97, 1 << 10, 1 << 16, 1 << 20, 1 << 22, rng.randint(1, 1 << 22)])
        if n // step > 3000:
            continue
        for ramp in (False, True):
            b = emul.sub_batch_bounds(n, step, ramp)
            assert b[0] == 0 and b[-1] == n
            sizes = [y - x for x, y in zip(b, b[1:])]
            assert all(0 < s <= step for s in sizes), (n, step, ramp, sizes[:8])
            if not ramp:
                assert all(s == step for s in sizes[:-1])
    b = emul.sub_batch_bounds(10_000_000, 1 << 20, True)
    sizes = [y - x for x, y in zip(b, b[1:])]
    assert sizes[0] == 1 << 16 and sizes[-1] == 1 << 17 and max(sizes) <= 1 << 20


CASES = [
    ("defaults dense+ktab", {}, 1, 8),
    ("direct k-mer entries", {}, 1, 10),
    ("direct entries, seeds longer than k + 8", dict(seed_size=24, seed_gap=9), 1, 10),
    ("sa_rate 4, no table", {}, 4, 0),
    ("file-rate SA, ktab 5", {}, 32, 5),
    ("max_candidates 1", dict(max_candidates=1), 1, 6),
    ("max_assignments 1", dict(max_assignments=1), 1, 6),
    ("edit 0.2 gap 3", dict(edit_rate=0.2, seed_gap=3), 1, 6),
    ("2k > L", dict(edit_rate=0.6), 1, 6),
    ("edit 0", dict(edit_rate=0.0), 1, 6),
    ("min_seed 0.5", dict(min_seed=0.5), 1, 6),
]


@pytest.mark.parametrize("name,flags,sa_rate,ktab_k", CASES, ids=[c[0] for c in CASES])
def test_pipeline_small(oracle, emul, small_ref, small_index, name, flags, sa_rate, ktab_k):
    reads = synth.make_reads(small_ref[0], small_ref[1], 1500, 150, seed=2)
    p = oracle.default_params(**flags)
    h1, o1 = small_index.bin_reads(reads, p, threads=4)
    e = emul.EmulIndex(small_index, sa_rate=sa_rate, ktab_k=ktab_k)
    h2, o2 = e.bin_reads(reads[0], reads[1], p)
    _same(h1, o1, h2, o2)
    if name.startswith("defaults"):
        assert len(h1) > 1000


def test_pipeline_redundant_reference(oracle, emul):
    """BASELINE config 4 in miniature: near-identical strains, 75 bp reads -> large SA intervals,
    tune-max-hits doubling, max-hits drops, hundreds of candidates per read."""
    ref = synth.make_reference(40, 3000, seed=6, n_frac=0.0, shared_frac=0.9, divergence=0.003)
    ix = oracle.Index.build((ref[0], ref[1]), ref[2], ref[3], 64, 32)
    reads = synth.make_reads(ref[0], ref[1], 800, 75, seed=7)
    for flags in ({}, dict(tune_max_hits=5, max_hits=30), dict(tune_max_hits=5, max_hits=30, seed_size=10,
                                                              seed_gap=4)):
        p = oracle.default_params(**flags)
        h1, o1 = ix.bin_reads(reads, p, threads=4)
        e = emul.EmulIndex(ix, sa_rate=2, ktab_k=5)
        h2, o2 = e.bin_reads(reads[0], reads[1], p)
        _same(h1, o1, h2, o2)
        assert len(h1) > 3000


def _n_rich_case(seed=41):
    """Reference with 3 % of its bases in N runs of 10-50 and reads sampled across them: N-rich seeds match
    other N runs (many spurious candidates), reads with more N than the edit budget can never be accepted
    (core.cuh::query_hopeless), reads with fewer still can."""
    ref = synth.make_reference(6, 30000, seed=seed, n_frac=0.03, shared_frac=0.1)
    reads = synth.make_reads(ref[0], ref[1], 1500, 150, seed=seed + 1, frac_n_reads=0.2)
    return ref, reads


def test_pipeline_n_rich_reference(oracle, emul):
    ref, reads = _n_rich_case()
    ix = oracle.Index.build((ref[0], ref[1]), ref[2], ref[3], 64, 32)
    cat = reads[0].reshape(-1, 150)
    n_per_read = (cat == ord("N")).sum(axis=1)
    assert (n_per_read > 20).sum() > 50 and ((n_per_read > 0) & (n_per_read <= 20)).sum() > 100
    for flags in ({}, dict(edit_rate=0.05), dict(edit_rate=0.3, max_hits=100000, tune_max_hits=100000)):
        p = oracle.default_params(**flags)
        h1, o1 = ix.bin_reads(reads, p, threads=4)
        e = emul.EmulIndex(ix, sa_rate=1, ktab_k=6)
        h2, o2 = e.bin_reads(reads[0], reads[1], p)
        _same(h1, o1, h2, o2)
        assert len(h1) > 500


def test_pipeline_checklist_cases(oracle, emul):
    """SURVEY appendix C, constructed (tests/checklist_cases.py): bin junctions, bins shorter than reads, equal seed
    counts, the same TaxID on both strands, tandem repeats, min_seeds >= 2, degenerate read lengths."""
    from tests.checklist_cases import build
    ix, reads, flag_sets = build()
    packed = oracle.pack_seqs(reads)
    for sa_rate, ktab_k in ((1, 8), (32, 0)):
        e = emul.EmulIndex(ix, sa_rate=sa_rate, ktab_k=ktab_k)
        for flags in flag_sets:
            p = oracle.default_params(**flags)
            h1, o1 = ix.bin_reads(reads, p, threads=4)
            h2, o2 = e.bin_reads(packed[0], packed[1], p)
            _same(h1, o1, h2, o2)


def test_pipeline_long_reads_high_edit(oracle, emul, small_ref, small_index):
    """BASELINE config 5 in miniature: 250 bp, edit-rate 0.2, dense seeding."""
    reads = synth.make_reads(small_ref[0], small_ref[1], 500, 250, seed=8, sub=0.10)
    p = oracle.default_params(edit_rate=0.2, seed_gap=3)
    h1, o1 = small_index.bin_reads(reads, p, threads=4)
    e = emul.EmulIndex(small_index, sa_rate=1, ktab_k=6)
    h2, o2 = e.bin_reads(reads[0], reads[1], p)
    _same(h1, o1, h2, o2)


def test_pipeline_ragged_and_garbage(oracle, emul, small_ref, small_index):
    """Empty reads, reads shorter than the seed (the reference panics; defined as no hits), lower case,
    IUPAC / garbage bytes (all map to N, src/binner.rs:88-100)."""
    rng = np.random.default_rng(3)
    ref = small_ref[0]
    rl = []
    for _ in range(400):
        L = int(rng.integers(0, 200))
        st = int(rng.integers(0, len(ref) - 220))
        s = bytes(ref[st:st + L])
        if rng.random() < 0.3:
            s = s.lower()
        rl.append(s)
    rl += [b"", b"A", b"ACGTNNNNacgtnnxx" * 3, b"RYKMSW" * 10]
    reads = oracle.pack_seqs(rl)
    p = oracle.default_params()
    h1, o1 = small_index.bin_reads(reads, p)
    e = emul.EmulIndex(small_index, sa_rate=1, ktab_k=6)
    h2, o2 = e.bin_reads(reads[0], reads[1], p)
    _same(h1, o1, h2, o2)


def test_appendix_e_through_emulation(oracle, emul):
    from tests.test_oracle import APPENDIX_E
    from mtsv_tools_b200 import results_lines
    for name, refs, read, flags, want, want_long in APPENDIX_E:
        ix = oracle.Index.build([r[2] for r in refs], [r[0] for r in refs], [r[1] for r in refs])
        e = emul.EmulIndex(ix, sa_rate=1, ktab_k=3)
        p = oracle.default_params(seed_size=10, seed_gap=5, **flags)
        cat, off = oracle.pack_seqs([read])
        hits, offs = e.bin_reads(cat, off, p)
        assert "".join(results_lines(["r"], hits, offs, False)).strip() == want, name
        assert "".join(results_lines(["r"], hits, offs, True)).strip() == want_long, name


def test_randomized_adversarial_cases(oracle, emul):
    import random
    from tests.fuzz_cases import rand_case
    rng = random.Random(20261018)
    for t in range(120):
        ix, reads, p = rand_case(rng)
        h1, o1 = ix.bin_reads(reads, p)
        cat, off = oracle.pack_seqs(reads)
        for sa_rate, kk in ((1, rng.randint(0, 6)), (rng.choice([2, 5, 32]), rng.randint(0, 6))):
            e = emul.EmulIndex(ix, sa_rate=sa_rate, ktab_k=kk)
            h2, o2 = e.bin_reads(cat, off, p)
            _same(h1, o1, h2, o2)
