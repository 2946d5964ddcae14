"""GPU parity tests: the CUDA hot path, called through the C ABI (libmtsv_b200.so), against the oracle
on the same seeded inputs, against the committed golden fixture, and — at larger sizes — through
size-independent properties.  Bit-exact comparisons throughout (integer work)."""
import os
import random

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from mtsv_tools_b200 import MGIndex, Params, results_lines, synth  # noqa: E402
from mtsv_tools_b200.index import edit_distance  # noqa: E402


def _params(oracle, **flags):
    return oracle.default_params(**flags), Params(**{
        "edit_rate": flags.get("edit_rate", 0.13), "seed_size": flags.get("seed_size", 18),
        "seed_gap": flags.get("seed_gap", 15), "min_seed": flags.get("min_seed", 0.015),
        "max_hits": flags.get("max_hits", 2000), "tune_max_hits": flags.get("tune_max_hits", 200),
        "max_candidates": flags.get("max_candidates"), "max_assignments": flags.get("max_assignments")})


def _gpu_index(orc_ix, **opts):
    return MGIndex.from_parts(orc_ix.text, orc_ix.bins(), orc_ix.bwt, orc_ix.sa_sample,
                              orc_ix.sa_sample_rate, **opts)


def _same(h1, o1, h2, o2):
    assert np.array_equal(o1, o2), "hit offsets differ at reads %s" % np.nonzero(o1 != o2)[0][:8]
    for f in ("tax_id", "gi", "offset", "edit"):
        assert np.array_equal(h1[f], h2[f]), f


@pytest.fixture(scope="module")
def small_ref():
    return synth.make_reference(8, 20000, seed=1, n_frac=0.002, shared_frac=0.1, seqs_per_taxid=2)


@pytest.fixture(scope="module")
def small_index(oracle, small_ref):
    cat, off, gi, tax = small_ref
    return oracle.Index.build((cat, off), gi, tax, 64, 32)


# ------------------------------------------------------------------ stage level
@pytest.mark.parametrize("ktab_k", [0xFFFFFFFF, 1, 4, 7, 0])
def test_backward_search_kernel(oracle, small_index, ktab_k):
    ix = small_index
    text = bytes(ix.text)
    rng = random.Random(11)
    with _gpu_index(ix, ktab_k=ktab_k) as g:
        for m in (7, 12, 18, 24):
            pats = []
            for _ in range(2000):
                if rng.random() < 0.6:
                    st = rng.randrange(0, len(text) - m - 1)
                    pat = bytearray(text[st:st + m])
                    if rng.random() < 0.3:
                        pat[rng.randrange(m)] = rng.choice(b"ACGTN")
                    pats.append(bytes(pat))
                else:
                    pats.append(bytes(rng.choice(b"ACGTN") for _ in range(m)))
            lo, up = g.backward_search(pats)
            for i, pat in enumerate(pats):
                r, olo, oup, _ = ix.backward_search(pat)
                want = (olo, oup) if r == 2 else (0, 0)
                assert (int(lo[i]), int(up[i])) == want, pat


@pytest.mark.parametrize("sa_rate", [1, 2, 8, 32])
def test_locate_kernel(oracle, small_index, sa_rate):
    ix = small_index
    n = len(ix)
    rng = np.random.default_rng(12)
    rows = np.concatenate([rng.integers(0, n, size=20000, dtype=np.uint64),
                           np.arange(0, 200, dtype=np.uint64), np.arange(n - 200, n, dtype=np.uint64)])
    with _gpu_index(ix, sa_rate=sa_rate) as g:
        assert g.info()["device_sa_rate"] == sa_rate
        pos = g.locate(rows)
    want = np.array([ix.locate(int(r))[0] for r in rows], dtype=np.uint64)
    assert np.array_equal(pos, want)
    # a full suffix array is a permutation of the text positions
    if sa_rate == 1:
        with _gpu_index(ix, sa_rate=1) as g:
            allpos = g.locate(np.arange(n, dtype=np.uint64))
        assert np.array_equal(np.sort(allpos), np.arange(n, dtype=np.uint64))


def test_edit_distance_kernel_kats_and_fuzz(oracle):
    from tests.test_oracle import ALIGN_KATS
    got = edit_distance([k[0] for k in ALIGN_KATS], [k[1] for k in ALIGN_KATS])
    assert list(got) == [k[2] for k in ALIGN_KATS]
    rng = random.Random(5)
    pats, txts = [], []
    for _ in range(4000):
        L = rng.choice([rng.randint(1, 64), rng.randint(65, 300), rng.randint(300, 1024), rng.randint(1025, 4096)])
        alpha = b"ACGTN" if rng.random() < 0.5 else b"ACGT"
        p = bytes(rng.choice(alpha) for _ in range(L))
        if rng.random() < 0.6:
            s = list(p)
            for _ in range(rng.randint(0, 30)):
                i = rng.randrange(len(s))
                r = rng.random()
                if r < 0.4:
                    s[i] = rng.choice(b"ACGT")
                elif r < 0.7:
                    s.insert(i, rng.choice(b"ACGT"))
                elif len(s) > 1:
                    del s[i]
            t = bytes(rng.choice(b"ACGT") for _ in range(rng.randint(0, 30))) + bytes(s) + \
                bytes(rng.choice(b"ACGT") for _ in range(rng.randint(0, 30)))
        else:
            t = bytes(rng.choice(alpha) for _ in range(rng.randint(1, 500)))
        pats.append(p)
        txts.append(t)
    got = edit_distance(pats, txts)
    want = [oracle.min_edit_distance(p, t) for p, t in zip(pats, txts)]
    assert list(got) == want


# ------------------------------------------------------------------ whole path
def test_golden_fixture(oracle):
    """The committed fixture (tests/golden/cfg1_small.npz, made by make_golden.py) — no oracle call."""
    from tests.golden.make_golden import build_case
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "cfg1_small.npz"))
    ix, reads, _ = build_case(oracle)
    with _gpu_index(ix) as gi:
        hits, offs = gi.bin_reads(reads, Params())
    assert np.array_equal(offs, g["hit_off"])
    for f in ("tax_id", "gi", "offset", "edit"):
        assert np.array_equal(hits[f], g[f])


CASES = [
    ("defaults", {}, {}),
    ("sa_rate 4, no table", {}, dict(sa_rate=4, ktab_k=0xFFFFFFFF)),
    ("file-rate SA, ktab 5", {}, dict(sa_rate=32, ktab_k=5)),
    ("max_candidates 1", dict(max_candidates=1), {}),
    ("max_assignments 1", dict(max_assignments=1), {}),
    ("edit 0.2 gap 3", dict(edit_rate=0.2, seed_gap=3), {}),
    ("2k > L", dict(edit_rate=0.6), {}),
    ("edit 0", dict(edit_rate=0.0), {}),
    ("min_seed 0.5", dict(min_seed=0.5), {}),
    ("seeds longer than k + 8 (direct k-mer entries continue in the text)", dict(seed_size=24, seed_gap=9), {}),
    ("file-rate SA, auto table (direct entries located by LF walks)", {}, dict(sa_rate=32)),
    ("tiny sub-batches", {}, dict(batch_reads=97)),
    ("hit cap forces splitting", {}, dict(max_batch_hits=5000)),
]


@pytest.mark.parametrize("name,flags,opts", CASES, ids=[c[0] for c in CASES])
def test_pipeline_small(oracle, small_ref, small_index, name, flags, opts):
    reads = synth.make_reads(small_ref[0], small_ref[1], 3000, 150, seed=2)
    po, pg = _params(oracle, **flags)
    h1, o1 = small_index.bin_reads(reads, po, threads=8)
    with _gpu_index(small_index, **opts) as g:
        h2, o2 = g.bin_reads(reads, pg)
        _same(h1, o1, h2, o2)
        # idempotence: the same batch again on the same handle, through the pinned-result entry point
        h3, o3 = g.bin_reads_pinned(reads, pg)
        _same(h2, o2, h3, o3)


def test_pipeline_redundant_reference(oracle):
    """BASELINE config 4 in miniature (locate / max-hits / tune-max-hits / many candidates; exercises
    the shared-memory and global-memory segmented sorts)."""
    ref = synth.make_reference(40, 3000, seed=6, n_frac=0.0, shared_frac=0.9, divergence=0.003)
    ix = oracle.Index.build((ref[0], ref[1]), ref[2], ref[3], 64, 32)
    reads = synth.make_reads(ref[0], ref[1], 1500, 75, seed=7)
    with _gpu_index(ix, sa_rate=2) as g:
        for flags in ({}, dict(tune_max_hits=5, max_hits=30),
                      dict(tune_max_hits=5, max_hits=30, seed_size=10, seed_gap=4),
                      dict(tune_max_hits=100000, max_hits=100000, seed_size=8, seed_gap=2)):
            po, pg = _params(oracle, **flags)
            h1, o1 = ix.bin_reads(reads, po, threads=8)
            h2, o2 = g.bin_reads(reads, pg)
            _same(h1, o1, h2, o2)


def test_pipeline_many_strains_sharing_taxids(oracle):
    """Heavy strands (hundreds of candidates) where several strains carry the SAME TaxID: only the first passing
    candidate of a TaxID in rank order may be reported (src/index.rs:393-396), with and without the
    max-candidates / max-assignments limits (:385-389, :421-425) — the warp-level selection with its hash set of
    accepted TaxIDs, and the scan fall-back beyond 512 candidates."""
    for n_strains, per_tax in ((200, 7), (200, 1), (700, 3)):
        taxids = 500 + (np.arange(n_strains, dtype=np.uint32) // np.uint32(per_tax))
        rng = np.random.default_rng(n_strains)
        taxids = taxids[rng.permutation(n_strains)]  # strains of one TaxID are not neighbours in the text
        ref = synth.make_reference(n_strains, 2000, seed=16, n_frac=0.0, shared_frac=0.95, divergence=0.004, taxids=taxids)
        ix = oracle.Index.build((ref[0], ref[1]), ref[2], ref[3], 64, 32)
        reads = synth.make_reads(ref[0], ref[1], 600, 75, seed=17)
        with _gpu_index(ix) as g:
            for flags in ({}, dict(max_assignments=3), dict(max_assignments=0), dict(max_candidates=40),
                          dict(max_candidates=100, max_assignments=33), dict(tune_max_hits=100000, max_hits=100000)):
                po, pg = _params(oracle, **flags)
                h1, o1 = ix.bin_reads(reads, po, threads=8)
                h2, o2 = g.bin_reads(reads, pg)
                _same(h1, o1, h2, o2)
            # (heavy strands indeed: about n_strains candidates per strand, one hit per TaxID among them)
            assert int((o1[1:] - o1[:-1]).max()) >= min(100, n_strains // per_tax)


def test_two_round_verification_is_result_preserving(oracle, small_ref, small_index, monkeypatch):
    """Verifying the leaders of the (strand, TaxID) groups first and the other members only when their leader
    failed (binner.cu, cand_leader_kernel) must give the results of verifying everything: forced on and forced off,
    on strands with one, a few and hundreds of candidates."""
    cat, off, gi, tax = small_ref
    reads_small = synth.make_reads(cat, off, 3000, 150, seed=41)
    taxids = 500 + (np.arange(150, dtype=np.uint32) // np.uint32(6))
    ref = synth.make_reference(150, 2000, seed=26, n_frac=0.0, shared_frac=0.95, divergence=0.01, taxids=taxids)
    heavy_ix = oracle.Index.build((ref[0], ref[1]), ref[2], ref[3], 64, 32)
    reads_heavy = synth.make_reads(ref[0], ref[1], 800, 75, seed=27, sub=0.06)  # some leaders fail, members pass
    for ix, reads, flags in ((small_index, reads_small, {}), (small_index, reads_small, dict(seed_gap=3, edit_rate=0.2)),
                             (heavy_ix, reads_heavy, {}), (heavy_ix, reads_heavy, dict(edit_rate=0.08)),
                             (heavy_ix, reads_heavy, dict(max_candidates=60, max_assignments=4))):
        po, pg = _params(oracle, **flags)
        h1, o1 = ix.bin_reads(reads, po, threads=8)
        with _gpu_index(ix) as g:
            verified = {}
            for mode in ("1", "0"):
                monkeypatch.setenv("MTSV_B200_GROUP_VERIFY", mode)
                h2, o2 = g.bin_reads(reads, pg)
                _same(h1, o1, h2, o2)
                verified[mode] = g.last_batch_stats()["n_candidates"]
            assert verified["1"] <= verified["0"]
            if ix is heavy_ix and not flags:
                assert verified["1"] < 0.5 * verified["0"]  # six strains per TaxID: most members are never aligned
    monkeypatch.delenv("MTSV_B200_GROUP_VERIFY")


def test_pipeline_long_reads_high_edit(oracle, small_ref, small_index):
    """BASELINE config 5 in miniature: 250 bp, edit-rate 0.2, --seed-interval 3."""
    reads = synth.make_reads(small_ref[0], small_ref[1], 1000, 250, seed=8, sub=0.10)
    po, pg = _params(oracle, edit_rate=0.2, seed_gap=3)
    h1, o1 = small_index.bin_reads(reads, po, threads=8)
    with _gpu_index(small_index) as g:
        h2, o2 = g.bin_reads(reads, pg)
    _same(h1, o1, h2, o2)


def test_pipeline_ragged_and_garbage(oracle, small_ref, small_index):
    rng = np.random.default_rng(3)
    ref = small_ref[0]
    rl = []
    for _ in range(600):
        L = int(rng.integers(0, 200))
        st = int(rng.integers(0, len(ref) - 220))
        s = bytes(ref[st:st + L])
        if rng.random() < 0.3:
            s = s.lower()
        rl.append(s)
    rl += [b"", b"A", b"ACGTNNNNacgtnnxx" * 3, b"RYKMSW" * 10]
    po, pg = _params(oracle)
    h1, o1 = small_index.bin_reads(oracle.pack_seqs(rl), po)
    with _gpu_index(small_index) as g:
        h2, o2 = g.bin_reads(rl, pg)
        _same(h1, o1, h2, o2)
        # empty batch
        h0, o0 = g.bin_reads([], pg)
        assert len(h0) == 0 and list(o0) == [0]
        # single-strand call == matching_tax_ids of the reference
        text = bytes(small_index.text)
        for st in (100, 5000, 33333):
            seq = text[st:st + 150]
            want = small_index.matching_tax_ids(seq, po)
            got = g.matching_tax_ids(seq)
            assert [tuple(h) for h in got] == want


def test_reads_over_the_length_limit_do_not_fail_the_batch(oracle, small_ref, small_index):
    """A read longer than MTSVGPU_MAX_READ_LEN is reported without hits and counted; every other read of the batch
    gets exactly the oracle's result (the reference itself has no such limit: README "Limits")."""
    cat, off, gi, tax = small_ref
    reads = synth.make_reads(cat, off, 2000, 150, seed=71)
    lst = [reads[0][int(reads[1][i]):int(reads[1][i + 1])].tobytes() for i in range(2000)]
    big1, big2 = bytes(cat[100:5100]), bytes(cat[20000:140000])
    lst.insert(700, big1)
    lst.insert(1500, big2)
    lst.append(bytes(cat[5:4101]))  # 4096 bases: the longest read that is still processed
    po, pg = _params(oracle)
    keep = [i for i in range(len(lst)) if i not in (700, 1500)]
    for opts in ({}, {"batch_reads": 300}):
        with _gpu_index(small_index, **opts) as g:
            for entry in ("bin_reads", "packed"):
                if entry == "packed":
                    from mtsv_tools_b200.index import pack_reads_planes
                    pk, po_ = pack_reads_planes(lst)
                    h2, o2 = g.bin_reads_packed(pk, po_, pg)
                    h2, o2 = h2.copy(), o2.copy()
                else:
                    h2, o2 = g.bin_reads(lst, pg)
                st = g.last_batch_stats()
                assert st["n_reads_over_limit"] == 2 and st["n_strands_over_hits"] == 0
                cnt = o2[1:] - o2[:-1]
                assert cnt[700] == 0 and cnt[1500] == 0
                h1, o1 = small_index.bin_reads([lst[i] for i in keep], po, threads=8)
                assert np.array_equal(cnt[keep], o1[1:] - o1[:-1])
                for f in ("tax_id", "gi", "offset", "edit"):
                    assert np.array_equal(h2[f], h1[f]), (opts, entry, f)
                assert (o1[-1] - o1[-2]) >= 1  # the 4096-base read maps


def test_pipeline_n_rich_reference(oracle):
    """N runs in the reference and reads sampled across them (see tests/test_emul_parity.py::_n_rich_case)."""
    from tests.test_emul_parity import _n_rich_case
    ref, reads = _n_rich_case()
    ix = oracle.Index.build((ref[0], ref[1]), ref[2], ref[3], 64, 32)
    with _gpu_index(ix) as g:
        for flags in ({}, dict(edit_rate=0.05), dict(edit_rate=0.3, max_hits=100000, tune_max_hits=100000)):
            po, pg = _params(oracle, **flags)
            h1, o1 = ix.bin_reads(reads, po, threads=8)
            h2, o2 = g.bin_reads(reads, pg)
            _same(h1, o1, h2, o2)
            assert len(h1) > 500


def test_warp_and_per_lane_verifiers_match_the_oracle(oracle, small_ref, small_index):
    """Batches whose reads all have at most 253 bases go through verify_warp_kernel (warp-uniform block range, 4-bit
    text); the per-lane verify_kernel (+ SW re-check) takes the others.  Both must give the oracle's hits: the warp
    verifier on uniform batches (1, 3 and 4 words) and on a ragged one (mutated reads of 1..253 bases so that the
    edit budget is actually used), the per-lane one on a uniform batch of 256 bases."""
    rng = np.random.default_rng(21)
    ref = small_ref[0]
    batches = {"uniform_150": synth.make_reads(small_ref[0], small_ref[1], 4000, 150, seed=31, sub=0.05),
               "uniform_64": synth.make_reads(small_ref[0], small_ref[1], 3000, 64, seed=32, sub=0.04),
               "uniform_253": synth.make_reads(small_ref[0], small_ref[1], 2000, 253, seed=34, sub=0.06),
               "uniform_256": synth.make_reads(small_ref[0], small_ref[1], 2000, 256, seed=33, sub=0.06)}
    rl = []
    for _ in range(4000):
        L = int(rng.integers(1, 254))  # <= 253: the whole batch stays on verify_warp_kernel (W = 4, ragged)
        st = int(rng.integers(0, len(ref) - 300))
        s = bytearray(ref[st:st + L])
        for _ in range(int(rng.integers(0, max(1, L // 12)))):
            s[int(rng.integers(0, L))] = b"ACGTN"[int(rng.integers(0, 5))]
        rl.append(bytes(s))
    batches["ragged"] = oracle.pack_seqs(rl)
    with _gpu_index(small_index) as g:
        for name, reads in batches.items():
            for flags in ({}, dict(edit_rate=0.2, seed_gap=5), dict(edit_rate=0.05)):
                po, pg = _params(oracle, **flags)
                h1, o1 = small_index.bin_reads(reads, po, threads=8)
                assert len(h1) > 100, name
                h2, o2 = g.bin_reads(reads, pg)
                _same(h1, o1, h2, o2)


def test_pipeline_reads_longer_than_253(oracle, small_ref, small_index):
    """Reads of 254-3000 bp (per-lane verifier with 4-64 words + the SW re-check) against what the oracle answers
    with the reference's own ssw.c (tests/golden/ssw_scores.npz; and ssw.c itself when oracle/_ref is built), whose
    16-bit kernel (used once SW reaches 254) is not textbook SW: candidates with edit <= k can still fail
    `score >= L - 2k`.  ssw_band_kernel / ssw_full_kernel must reject exactly those.
    Includes reads built to sit on that threshold (tests/test_emul_parity.py::_borderline_long_reads)."""
    from tests.golden.make_ssw_golden import GPU_CASES, PATH, expected_hits, long_read_batch
    golden = np.load(PATH)
    L = oracle.lib()
    have_ref = oracle.ssw_ref_available()
    n_changed = 0
    with _gpu_index(small_index) as g:
        for i, case in enumerate(GPU_CASES):
            reads = long_read_batch(oracle, small_ref[0], case, ragged=True)
            po, pg = _params(oracle, edit_rate=case[1])
            o1, h1 = expected_hits(golden, "gpu%d" % i)
            if have_ref:
                _same(h1, o1, *small_index.bin_reads(reads, po, threads=8))
            h2, o2 = g.bin_reads(reads, pg)
            _same(h1, o1, h2, o2)
            assert len(h1) > case[3] // 4
            L.orc_set_ssw_kind(2)  # textbook SW: "edit <= k" would be the whole rule
            try:
                h3, o3 = small_index.bin_reads(reads, po, threads=8)
            finally:
                L.orc_set_ssw_kind(0)
            n_changed += int(np.sum((o3[1:] - o3[:-1]) != (o1[1:] - o1[:-1])))
    assert n_changed > 0, "no read exercised the 16-bit kernel's deviation"


def test_randomized_adversarial_cases(oracle):
    """tests/fuzz_cases.py through the C ABI: 150 random tiny indexes x up to 40 reads with extreme flags."""
    from tests.fuzz_cases import rand_case
    rng = random.Random(20261018)
    for t in range(150):
        ix, reads, p = rand_case(rng)
        h1, o1 = ix.bin_reads(reads, p)
        pg = Params(edit_rate=p.edit_rate, seed_size=p.seed_size, seed_gap=p.seed_gap, min_seed=p.min_seed,
                    max_hits=p.max_hits, tune_max_hits=p.tune_max_hits,
                    max_candidates=None if p.max_candidates < 0 else p.max_candidates,
                    max_assignments=None if p.max_assignments < 0 else p.max_assignments)
        opts = dict(sa_rate=rng.choice([1, 2, 32]), ktab_k=rng.choice([0, 0xFFFFFFFF, 2, 5]))
        if opts["sa_rate"] > ix.sa_sample_rate:
            opts["sa_rate"] = 1
        with _gpu_index(ix, **opts) as g:
            h2, o2 = g.bin_reads(reads, pg)
        _same(h1, o1, h2, o2)


def test_pipeline_checklist_cases(oracle):
    """SURVEY appendix C, constructed (tests/checklist_cases.py), through both host entry points."""
    from tests.checklist_cases import build
    ix, reads, flag_sets = build()
    packed = oracle.pack_seqs(reads)
    for opts in ({}, dict(sa_rate=32, ktab_k=0xFFFFFFFF), dict(batch_reads=64)):
        with _gpu_index(ix, **opts) as g:
            for flags in flag_sets:
                po, pg = _params(oracle, **flags)
                h1, o1 = ix.bin_reads(reads, po, threads=8)
                h2, o2 = g.bin_reads(reads, pg)
                _same(h1, o1, h2, o2)
                h3, o3 = g.bin_reads_pinned(packed, pg)
                _same(h1, o1, h3, o3)


def test_randomized_long_and_ragged_cases(oracle):
    """tests/fuzz_cases.py::long_case through both host entry points: read lengths 0..420 (every verifier width,
    uniform and ragged batches, the SW re-check of reads >= 254 bases), tiny sub-batches (many slices on both
    lanes, adaptive launch groups).  tools/fuzz_gpu.py runs the same generator for minutes."""
    from tests.fuzz_cases import long_case
    rng = random.Random(4242)
    for t in range(120):
        ix, reads, p = long_case(rng)
        h1, o1 = ix.bin_reads(reads, p)
        pg = Params(edit_rate=p.edit_rate, seed_size=p.seed_size, seed_gap=p.seed_gap, min_seed=p.min_seed,
                    max_hits=p.max_hits, tune_max_hits=p.tune_max_hits,
                    max_candidates=None if p.max_candidates < 0 else p.max_candidates,
                    max_assignments=None if p.max_assignments < 0 else p.max_assignments)
        opts = dict(sa_rate=rng.choice([1, 2, 32]), ktab_k=rng.choice([0, 0xFFFFFFFF, 2, 5]),
                    batch_reads=rng.choice([0, 0, 1, 3, 7, 16]), max_batch_hits=rng.choice([0, 0, 50]))
        if opts["sa_rate"] > ix.sa_sample_rate:
            opts["sa_rate"] = 1
        with _gpu_index(ix, **opts) as g:
            try:
                h2, o2 = g.bin_reads(reads, pg)
                h3, o3 = g.bin_reads_pinned(oracle.pack_seqs(reads), pg)
                h3, o3 = h3.copy(), o3.copy()  # views of the handle's page-locked buffers: gone when it closes
            except Exception as e:  # a refused case (seed-hit cap of 50 on one read) must say so
                assert "cap" in str(e) or "limit" in str(e).lower(), e
                continue
        _same(h1, o1, h2, o2)
        _same(h1, o1, h3, o3)


def test_appendix_e_vectors_on_gpu(oracle):
    from tests.test_oracle import APPENDIX_E
    for name, refs, read, flags, want, want_long in APPENDIX_E:
        ix = oracle.Index.build([r[2] for r in refs], [r[0] for r in refs], [r[1] for r in refs])
        po, pg = _params(oracle, seed_size=10, seed_gap=5, **flags)
        with _gpu_index(ix) as g:
            hits, offs = g.bin_reads([read], pg)
        assert "".join(results_lines(["r"], hits, offs, False)).strip() == want, name
        assert "".join(results_lines(["r"], hits, offs, True)).strip() == want_long, name


def test_index_file_roundtrip_on_gpu(oracle, small_index, small_ref, tmp_path):
    """mtsvgpu_index_open on a bincode .index written by the restated mtsv-build."""
    p = str(tmp_path / "small.index")
    small_index.write(p)
    reads = synth.make_reads(small_ref[0], small_ref[1], 500, 150, seed=21)
    po, pg = _params(oracle)
    h1, o1 = small_index.bin_reads(reads, po, threads=4)
    with MGIndex.from_file(p) as g:
        info = g.info()
        assert info["text_len"] == len(small_index) and info["file_sa_rate"] == 32
        h2, o2 = g.bin_reads(reads, pg)
    _same(h1, o1, h2, o2)
    # corrupt files are rejected, not mis-read
    raw = bytearray(open(p, "rb").read())
    bad = str(tmp_path / "bad.index")
    open(bad, "wb").write(raw[:-5])
    from mtsv_tools_b200 import LibraryError
    with pytest.raises(LibraryError):
        MGIndex.from_file(bad)
    raw2 = bytearray(raw)
    n = int.from_bytes(raw2[:8], "little")
    bwt_off = 8 + n + 8 + 24 * len(small_index.bins()[0]) + 8
    for i in range(0, 4000, 7):  # scramble BWT symbols: LF walks no longer agree with the samples
        raw2[bwt_off + 1000 + i] = ord("A") if raw2[bwt_off + 1000 + i] != ord("A") else ord("C")
    open(bad, "wb").write(raw2)
    with pytest.raises(LibraryError):
        MGIndex.from_file(bad)


def test_medium_scale_properties(oracle):
    """10 Mbp reference (BASELINE config 1 shape), 100k reads: compare a 5k-read sample with the oracle and
    check size-independent properties on the whole batch."""
    cat, off, gi, tax = synth.make_reference(52, 192308, seed=1, n_frac=0.001)
    ix = oracle.Index.build((cat, off), gi, tax, 64, 32)
    reads = synth.make_reads(cat, off, 100000, 150, seed=2)
    po, pg = _params(oracle)
    with _gpu_index(ix) as g:
        hits, offs = g.bin_reads(reads, pg)
        # (1) sample vs oracle
        sub = (reads[0][:5000 * 150], reads[1][:5001])
        h1, o1 = ix.bin_reads(sub, po, threads=8)
        assert np.array_equal(offs[:5001], o1)
        for f in ("tax_id", "gi", "offset", "edit"):
            assert np.array_equal(hits[f][:int(o1[-1])], h1[f])
        # (2) strand symmetry: reverse-complemented reads give the same TaxID/edit sets
        rc = synth._COMP[reads[0].reshape(-1, 150)[:, ::-1]].reshape(-1)
        hits_rc, offs_rc = g.bin_reads((rc, reads[1]), pg)
    names = [str(i) for i in range(100000)]
    a = results_lines(names, hits, offs)
    b = results_lines(names, hits_rc, offs_rc)
    assert a == b
    # (3) ~90% of reads come from the reference and must be assigned; edits within budget
    assert 0.85 < len(a) / 100000 < 0.95
    assert hits["edit"].max() <= 20
