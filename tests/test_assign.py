"""mtsvgpu_assign_batch_{pinned,packed,device}: the default results format computed on the device.  Every comparison
is bit-exact against two references: the oracle's default-format lines, and the host reduction (each TaxID once with
its minimum edit, by TaxID) of the same handle's bin_reads* output."""
import gzip
import os
import subprocess

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from mtsv_tools_b200 import assignment_lines, results_lines, synth  # noqa: E402
from mtsv_tools_b200.chunked import _DevArray  # noqa: E402
from mtsv_tools_b200.index import HIT_DTYPE, TAXHIT_DTYPE, pack_reads, pack_reads_planes  # noqa: E402
from tests.test_gpu_parity import CASES, _gpu_index, _params  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _reduce(hits, off):
    """Host reduction of Hit records: per read each TaxID once with its minimum edit, by TaxID."""
    n = len(off) - 1
    read = np.repeat(np.arange(n), (off[1:] - off[:-1]).astype(np.int64))
    order = np.lexsort((hits["edit"], hits["tax_id"], read))
    r, t, e = read[order], hits["tax_id"][order], hits["edit"][order]
    first = np.ones(len(r), bool)
    first[1:] = (r[1:] != r[:-1]) | (t[1:] != t[:-1])
    out = np.zeros(int(first.sum()), TAXHIT_DTYPE)
    out["tax_id"], out["edit"] = t[first], e[first]
    roff = np.zeros(n + 1, np.uint64)
    roff[1:] = np.cumsum(np.bincount(r[first], minlength=n))
    return out, roff


def _same(got, want, what):
    (t1, o1), (t2, o2) = got, want
    assert np.array_equal(np.asarray(o1, np.uint64), o2), "%s: offsets differ at reads %s" % (
        what, np.nonzero(np.asarray(o1, np.uint64) != o2)[0][:8])
    assert np.array_equal(t1["tax_id"], t2["tax_id"]) and np.array_equal(t1["edit"], t2["edit"]), what


def _device_assign(g, reads, pg, strands=2):
    cat, off = reads if isinstance(reads, tuple) else pack_reads(reads)
    n = len(off) - 1
    d_seqs = torch.from_numpy(np.concatenate([cat, np.zeros(1, np.uint8)])).cuda()  # (never a null pointer)
    d_off = torch.from_numpy(np.asarray(off, np.uint64).astype(np.int64)).cuda()
    dt, do, nt = g.assign_reads_device(d_seqs.data_ptr(), d_off.data_ptr(), n, pg, strands)
    recs = torch.as_tensor(_DevArray(dt, max(nt, 1) * 8), device="cuda").cpu().numpy()
    offs = torch.as_tensor(_DevArray(do, (n + 1) * 8), device="cuda").cpu().numpy()
    return recs.view(TAXHIT_DTYPE)[:nt].copy(), offs.view(np.uint64).copy()


def _from_device(ptr, n, dtype):
    """n records of `dtype` at a device pointer the library returned, copied to the host."""
    raw = torch.as_tensor(_DevArray(ptr, max(n, 1) * dtype.itemsize), device="cuda").cpu().numpy()
    return raw.view(dtype)[:n].copy()


def _seq_off_with_tail(off, tail):
    """seq_off at the start of a longer device tensor whose `tail` further entries hold 1 << 62: a slice bound
    fetched from past seq_off[n] is then far beyond the batch (and the batch fails) instead of reading whatever
    follows the array."""
    t = np.full(len(off) + tail, 1 << 62, np.int64)
    t[:len(off)] = np.asarray(off, np.uint64).astype(np.int64)
    return torch.from_numpy(t).cuda()


# (reads, batch_reads) of device-resident batches whose slice count is raised to an even number, which leaves the
# last slice empty: 5 reads in steps of 2 are sliced 0 2 4 5 5
EMPTY_LAST_SLICE = [(5, 2), (3, 1), (9, 4), (1000, 16), (4097, 16), (20000, 97)]


def test_device_input_whose_last_slice_is_empty(oracle, emul, small_ref, small_index):
    """mtsvgpu_bin_batch_device and mtsvgpu_assign_batch_device on batches whose last slice is empty, against the
    oracle; with per-stage timing on (one lane: no empty slice) as the control.  Every slice bound, the empty slice's
    too, is seq_off[n] or an entry before it."""
    cat, off = small_ref[0], small_ref[1]
    po, pg = _params(oracle)
    for n, step in EMPTY_LAST_SLICE:
        b = emul.slice_bounds(n, step, False, True)
        assert b[-3] < b[-2] == b[-1] == n, (n, step, b[-3:])
        assert emul.slice_bounds(n, step, False, False)[-2] < n
        reads = synth.make_reads(cat, off, n, 150, seed=n)
        h1, o1 = small_index.bin_reads(reads, po, threads=8)
        want = _reduce(h1, o1)
        d_seqs = torch.from_numpy(np.concatenate([reads[0], np.zeros(1, np.uint8)])).cuda()
        d_off = _seq_off_with_tail(reads[1], b[1] + 1)
        with _gpu_index(small_index, batch_reads=step) as g:
            for profiling in (False, True):
                g.set_profiling(profiling)
                what = "%d reads, batch_reads %d, profiling %d" % (n, step, profiling)
                dh, do, nh = g.bin_reads_device(d_seqs.data_ptr(), d_off.data_ptr(), n, pg)
                hits, offs = _from_device(dh, nh, HIT_DTYPE), _from_device(do, n + 1, np.dtype(np.uint64))
                assert np.array_equal(offs, o1), what
                for f in ("tax_id", "gi", "offset", "edit"):
                    assert np.array_equal(hits[f], h1[f]), (what, f)
                dt, do, nt = g.assign_reads_device(d_seqs.data_ptr(), d_off.data_ptr(), n, pg)
                _same((_from_device(dt, nt, TAXHIT_DTYPE), _from_device(do, n + 1, np.dtype(np.uint64))), want, what)
                st = g.last_batch_stats()
                assert st["n_queries"] == 2 * n and st["n_hits"] == len(h1), what
                assert st["n_sub_batches"] >= (len(b) - 2 if not profiling else 1), what


def _check(g, reads, names, pg, want_lines, strands=2, entries=("pinned", "packed", "device")):
    """Each entry point against the oracle's lines and against the host reduction of this handle's bin output."""
    h, o = g.bin_reads(reads, pg, strands)
    want = _reduce(h, o)
    assert results_lines(names, h, o, False) == want_lines
    for entry in entries:
        if entry == "pinned":
            got = g.assign_reads(reads, pg, strands)
        elif entry == "packed":
            pk, poff = pack_reads_planes(reads)
            got = tuple(x.copy() for x in g.assign_reads_packed(pk, poff, pg, strands))
        else:
            got = _device_assign(g, reads, pg, strands)
        _same(got, want, entry)
        assert assignment_lines(names, *got) == want_lines, entry
        st = g.last_batch_stats()
        assert st["n_hits"] == len(h) and st["n_queries"] == len(names) * strands
    return want


@pytest.fixture(scope="module")
def small_ref():
    return synth.make_reference(8, 20000, seed=1, n_frac=0.002, shared_frac=0.1, seqs_per_taxid=2)


@pytest.fixture(scope="module")
def small_index(oracle, small_ref):
    cat, off, gi, tax = small_ref
    return oracle.Index.build((cat, off), gi, tax, 64, 32)


def _names(n):
    return ["r%d" % i for i in range(n)]


@pytest.mark.parametrize("name,flags,opts", CASES, ids=[c[0] for c in CASES])
def test_assign_pipeline_small(oracle, small_ref, small_index, name, flags, opts):
    reads = synth.make_reads(small_ref[0], small_ref[1], 3000, 150, seed=2)
    names = _names(3000)
    po, pg = _params(oracle, **flags)
    h1, o1 = small_index.bin_reads(reads, po, threads=8)
    with _gpu_index(small_index, **opts) as g:
        _check(g, reads, names, pg, oracle.results_lines(names, h1, o1, False))


def test_assign_packed_ragged(oracle, small_ref, small_index):
    rng = np.random.default_rng(5)
    cat = small_ref[0]
    rl = []
    for _ in range(2500):
        L = int(rng.integers(1, 300))
        st = int(rng.integers(0, len(cat) - 320))
        rl.append(bytes(cat[st:st + L]))
    names = _names(len(rl))
    po, pg = _params(oracle)
    h1, o1 = small_index.bin_reads(oracle.pack_seqs(rl), po, threads=8)
    with _gpu_index(small_index) as g:
        _check(g, rl, names, pg, oracle.results_lines(names, h1, o1, False))


def test_assign_many_taxids_per_read(oracle):
    """A redundant reference, and hundreds to thousands of strains under distinct or shared TaxIDs: hundreds of
    records per read, segments for the warp, medium (33-4096 keys) and large (> 4096 keys) sorts."""
    ref = synth.make_reference(40, 3000, seed=6, n_frac=0.0, shared_frac=0.9, divergence=0.003)
    ix = oracle.Index.build((ref[0], ref[1]), ref[2], ref[3], 64, 32)
    reads = synth.make_reads(ref[0], ref[1], 1500, 75, seed=7)
    names = _names(1500)
    with _gpu_index(ix, sa_rate=2) as g:
        for flags in ({}, dict(tune_max_hits=5, max_hits=30), dict(tune_max_hits=100000, max_hits=100000, seed_size=8,
                                                                   seed_gap=2)):
            po, pg = _params(oracle, **flags)
            h1, o1 = ix.bin_reads(reads, po, threads=8)
            _check(g, reads, names, pg, oracle.results_lines(names, h1, o1, False))
    big = dict(tune_max_hits=100000, max_hits=100000)
    for n_strains, per_tax, n_reads, flag_sets in (
            (700, 3, 600, ({}, dict(max_assignments=3), dict(max_assignments=0), dict(max_candidates=100,
                                                                                      max_assignments=33), big)),
            (8000, 1, 120, (big, dict(big, max_assignments=2500)))):
        taxids = 500 + (np.arange(n_strains, dtype=np.uint32) // np.uint32(per_tax))
        taxids = taxids[np.random.default_rng(n_strains).permutation(n_strains)]
        ref = synth.make_reference(n_strains, 200 if n_strains > 1000 else 2000, seed=16, n_frac=0.0,
                                   shared_frac=0.95, divergence=0.004, taxids=taxids)
        ix = oracle.Index.build((ref[0], ref[1]), ref[2], ref[3], 64, 32)
        reads = synth.make_reads(ref[0], ref[1], n_reads, 75, seed=17)
        names = _names(n_reads)
        with _gpu_index(ix) as g:
            for flags in flag_sets:
                po, pg = _params(oracle, **flags)
                h1, o1 = ix.bin_reads(reads, po, threads=8)
                t, to = _check(g, reads, names, pg, oracle.results_lines(names, h1, o1, False))
                if flags is big:
                    per_read = (to[1:] - to[:-1]).max()
                    assert per_read >= min(100, n_strains // per_tax), per_read
                    if n_strains > 1000:
                        assert int((o1[1:] - o1[:-1]).max()) > 4096  # a read's keys take the large sort


def _repeated_taxids(hits, off):
    """Reads of which several hits carry one TaxID, and how many of those hits carry different edits."""
    reads = same_edit = 0
    for i in range(len(off) - 1):
        h = hits[int(off[i]):int(off[i + 1])]
        edits = {}
        for t, e in zip(h["tax_id"].tolist(), h["edit"].tolist()):
            edits.setdefault(t, []).append(e)
        rep = [v for v in edits.values() if len(v) > 1]
        reads += bool(rep)
        same_edit += sum(len(set(v)) > 1 for v in rep)
    return reads, same_edit


def test_assign_merges_a_taxid_hit_on_both_strands(oracle):
    """The merge itself: reads whose TaxID is hit on both strands (tests/checklist_cases.py: a sequence and a mutated
    reverse-complement copy under one TaxID) become one record with the smaller edit.  Every flag set of the checklist,
    through all three entry points, with one slice and with many."""
    from tests.checklist_cases import build
    ix, reads, flag_sets = build()
    names = _names(len(reads))
    merged_sets = differing = 0
    for opts in ({}, dict(batch_reads=64)):
        with _gpu_index(ix, **opts) as g:
            for flags in flag_sets:
                po, pg = _params(oracle, **flags)
                h1, o1 = ix.bin_reads(reads, po, threads=8)
                t, to = _check(g, reads, names, pg, oracle.results_lines(names, h1, o1, False))
                if len(t) < len(h1):
                    merged_sets += 1
                    n_rep, n_diff = _repeated_taxids(h1, o1)
                    assert n_rep == int(np.sum((o1[1:] - o1[:-1]) != (to[1:] - to[:-1]).astype(o1.dtype)))
                    differing += n_diff
    assert merged_sets >= 2  # (at least one flag set per option set merges hits)
    assert differing > 0  # and some merged hits had different edits: the smaller one must win


def test_assign_merges_hundreds_of_taxids_on_both_strands(oracle):
    """Strains and mutated reverse-complement copies of them under the same TaxIDs: every read hits its TaxIDs on both
    strands, a few hundred keys per read with one duplicate per TaxID (the medium sort, then the merge)."""
    n_strains = 300
    taxids = 500 + (np.arange(n_strains, dtype=np.uint32) // np.uint32(2))
    cat, off, gi, tax = synth.make_reference(n_strains, 2000, seed=23, n_frac=0.0, shared_frac=0.95, divergence=0.004,
                                             taxids=taxids)
    rng = np.random.default_rng(24)
    seqs = [bytes(cat[int(off[i]):int(off[i + 1])]) for i in range(n_strains)]
    for i in range(n_strains):  # the copy of strain i: reverse complement, 1 % substitutions
        rc = bytearray(synth.revcomp(seqs[i]))
        for p in rng.integers(0, len(rc), size=len(rc) // 100):
            rc[int(p)] = b"ACGT"[int(rng.integers(0, 4))]
        seqs.append(bytes(rc))
    gi2 = np.arange(1, 2 * n_strains + 1, dtype=np.uint32)
    tax2 = np.concatenate([tax, tax])
    ix = oracle.Index.build(seqs, gi2, tax2, 64, 32)
    rcat = np.frombuffer(b"".join(seqs[:n_strains]), np.uint8).copy()
    reads = synth.make_reads(rcat, off, 800, 100, seed=25)
    names = _names(800)
    with _gpu_index(ix) as g:
        for flags in ({}, dict(tune_max_hits=100000, max_hits=100000), dict(max_assignments=40)):
            po, pg = _params(oracle, **flags)
            h1, o1 = ix.bin_reads(reads, po, threads=8)
            t, to = _check(g, reads, names, pg, oracle.results_lines(names, h1, o1, False))
            n_rep, n_diff = _repeated_taxids(h1, o1)
            assert len(t) < 0.75 * len(h1) and n_rep > 400 and n_diff > 0, (len(t), len(h1), n_rep, n_diff)
            if not flags:
                assert int((o1[1:] - o1[:-1]).max()) > 32  # segments beyond the warp sort


def test_assign_reads_longer_than_253(oracle, small_ref, small_index):
    """Reads of 254 bases and more (the per-lane verifier and the SW re-check), against the stored answers of the
    reference's ssw.c (tests/golden/ssw_scores.npz)."""
    from tests.golden.make_ssw_golden import GPU_CASES, PATH, expected_hits, long_read_batch
    golden = np.load(PATH)
    with _gpu_index(small_index) as g:
        for i, case in enumerate(GPU_CASES):
            reads = long_read_batch(oracle, small_ref[0], case, ragged=True)
            names = _names(len(reads[1]) - 1)
            _, pg = _params(oracle, edit_rate=case[1])
            o1, h1 = expected_hits(golden, "gpu%d" % i)
            _check(g, reads, names, pg, oracle.results_lines(names, h1, o1, False))


def test_assign_ragged_garbage_empty_and_single_strand(oracle, small_ref, small_index):
    rng = np.random.default_rng(3)
    cat = small_ref[0]
    rl = []
    for _ in range(600):
        L = int(rng.integers(0, 200))
        st = int(rng.integers(0, len(cat) - 220))
        s = bytes(cat[st:st + L])
        rl.append(s.lower() if rng.random() < 0.3 else s)
    rl += [b"", b"A", b"ACGTNNNNacgtnnxx" * 3, b"RYKMSW" * 10, b"", b""]
    names = _names(len(rl))
    po, pg = _params(oracle)
    h1, o1 = small_index.bin_reads(oracle.pack_seqs(rl), po)
    with _gpu_index(small_index) as g:
        _check(g, rl, names, pg, oracle.results_lines(names, h1, o1, False))
        # no reads at all
        empty = pack_reads_planes([])
        for got in (g.assign_reads([], pg), g.assign_reads_packed(*empty, pg), _device_assign(g, [], pg)):
            assert len(got[0]) == 0 and list(got[1]) == [0]
        # only reads without hits
        t, to = g.assign_reads([b"", b"NNNN", b""], pg)
        assert len(t) == 0 and list(to) == [0, 0, 0, 0]
        # one strand: matching_tax_ids of the reference, per read
        text = bytes(small_index.text)
        one = [text[st:st + 150] for st in range(100, 150000, 499)]
        names1 = _names(len(one))
        lines = [oracle.format_assignments(n, small_index.matching_tax_ids(s, po), False)
                 for n, s in zip(names1, one)]
        _check(g, one, names1, pg, [x for x in lines if x], strands=1)


def test_assign_reads_over_the_length_limit(oracle, small_ref, small_index):
    cat, off, gi, tax = small_ref
    reads = synth.make_reads(cat, off, 2000, 150, seed=71)
    lst = [reads[0][int(reads[1][i]):int(reads[1][i + 1])].tobytes() for i in range(2000)]
    lst.insert(700, bytes(cat[100:5100]))
    lst.insert(1500, bytes(cat[20000:140000]))
    names = _names(len(lst))
    po, pg = _params(oracle)
    keep = [i for i in range(len(lst)) if i not in (700, 1500)]
    h1, o1 = small_index.bin_reads([lst[i] for i in keep], po, threads=8)
    want_lines = oracle.results_lines([names[i] for i in keep], h1, o1, False)
    for opts in ({}, {"batch_reads": 300}):
        with _gpu_index(small_index, **opts) as g:
            _check(g, lst, names, pg, want_lines)
            assert g.last_batch_stats()["n_reads_over_limit"] == 2


def test_assign_slices_splits_regrowth_and_interleaving(oracle, small_ref, small_index):
    """Many slices on both lanes with the result copy overlapped (pinned buffers already large enough), the
    split-and-retry path of a small seed-hit cap, batches that grow (pinned buffers regrow), and bin and assign calls
    taking turns on one handle."""
    cat, off = small_ref[0], small_ref[1]
    po, pg = _params(oracle)
    batches = [synth.make_reads(cat, off, n, 150, seed=90 + i) for i, n in enumerate((100, 1200, 5000, 800, 9000))]
    want = []
    for reads in batches:
        h1, o1 = small_index.bin_reads(reads, po, threads=8)
        names = _names(len(reads[1]) - 1)
        want.append((names, oracle.results_lines(names, h1, o1, False)))
    for opts in ({"batch_reads": 97}, {"batch_reads": 1024}, {"max_batch_hits": 5000}, {}):
        with _gpu_index(small_index, **opts) as g:
            for reads, (names, lines) in zip(batches, want):
                _check(g, reads, names, pg, lines)
            # the same batches again: the pinned buffers now fit, the copy-out overlaps the compute
            for reads, (names, lines) in zip(batches, want):
                t, to = g.assign_reads(reads, pg)
                assert assignment_lines(names, t, to) == lines
                h, o = g.bin_reads_pinned(reads, pg)
                assert results_lines(names, h, o, False) == lines
            if opts.get("batch_reads") == 97:
                assert g.last_batch_stats()["n_sub_batches"] > 50


def test_cli_many_taxids_both_formats(oracle, tmp_path):
    """mtsv-binner on a reference of hundreds of strains sharing TaxIDs: the default format (merged on the device)
    and the long format, against the oracle's lines."""
    binary = os.path.join(ROOT, "mtsv_tools_b200", "bin", "mtsv-binner")
    taxids = 500 + (np.arange(300, dtype=np.uint32) // np.uint32(3))
    taxids = taxids[np.random.default_rng(9).permutation(300)]
    cat, off, gi, tax = synth.make_reference(300, 2000, seed=19, n_frac=0.0, shared_frac=0.95, divergence=0.004,
                                             taxids=taxids)
    ix = oracle.Index.build((cat, off), gi, tax, 64, 32)
    index_path = str(tmp_path / "ref.index")
    ix.write(index_path)
    rc, ro = synth.make_reads(cat, off, 4000, 75, seed=20)
    names = ["read_%d" % i for i in range(4000)]
    fq = tmp_path / "reads.fq.gz"
    with gzip.open(fq, "wt") as f:
        for i, n in enumerate(names):
            s = bytes(rc[int(ro[i]):int(ro[i + 1])]).decode()
            f.write("@%s x\n%s\n+\n%s\n" % (n, s, "I" * len(s)))
    hits, offs = ix.bin_reads((rc, ro), oracle.default_params(), threads=8)
    assert int((offs[1:] - offs[:-1]).max()) >= 50
    for long in (False, True):
        res = tmp_path / ("res_%d.txt" % long)
        args = [binary, "--fastq", str(fq), "--index", index_path, "--results", str(res), "--batch-reads", "1000"]
        r = subprocess.run(args + (["--output-format", "long"] if long else []), capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        assert res.read_text() == "".join(oracle.results_lines(names, hits, offs, long))
