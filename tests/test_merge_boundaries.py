"""The per-read sort, merge and scan kernels at the sizes where the library switches kernels, against exact
references.

* mtsvgpu_collapse_device (mode TaxId) takes arbitrary per-read hit lists, which makes it a direct harness for the
  segmented sorts (segsort.cu::run_segmented_sort: warp <= 32 keys, shared-memory bitonic <= 4096, in place in global
  memory above), the merge (core.cuh::taxid_count / taxid_write) and the scan (util.cu::exclusive_scan_u32: 2048-entry
  tiles, a carry loop above 1024 tiles).  The reference is plain numpy.
* mtsvgpu_collapse_device_taxid_gi against a numpy statement of its rule.
* The binning pipeline on references built so that every strand's seed-hit count is known exactly (m copies of one
  segment, one seed per strand), at the per-strand boundaries of the sort, coalesce, rank, select and leader kernels,
  through every bin and assign entry point, against the oracle; and a read-length sweep across the verifier's
  word widths and the switch to the SW route."""
import numpy as np
import pytest

from mtsv_tools_b200 import synth
from mtsv_tools_b200.index import HIT_DTYPE
from tests.test_assign import small_index, small_ref  # noqa: F401  (fixtures)

U32 = 0xFFFFFFFF


# ------------------------------------------------------------------------------------------------
# numpy references
# ------------------------------------------------------------------------------------------------
def ref_taxid(read, tax, edit, n_reads):
    """mtsv-collapse mode TaxId: per read each TaxID once with its minimum edit, by TaxID.  Returns (pairs uint32
    [n, 2], offsets uint64 [n_reads + 1])."""
    order = np.lexsort((edit, tax, read))
    r, t, e = read[order], tax[order], edit[order]
    first = np.ones(len(r), bool)
    first[1:] = (r[1:] != r[:-1]) | (t[1:] != t[:-1])
    pairs = np.stack([t[first], e[first]], axis=1).astype(np.uint32).reshape(-1, 2)
    offs = np.zeros(n_reads + 1, np.uint64)
    offs[1:] = np.cumsum(np.bincount(r[first], minlength=n_reads))
    return pairs, offs


def ref_taxid_gi(read, hits, n_reads):
    """mtsv-collapse mode TaxIdGi: per read and (TaxID, GI) the hit with the smallest edit, ties to the smallest
    offset, by (TaxID, GI).  Returns (hits HIT_DTYPE, offsets uint64 [n_reads + 1])."""
    order = np.lexsort((hits["offset"], hits["edit"], hits["gi"], hits["tax_id"], read))
    r, h = read[order], hits[order]
    first = np.ones(len(r), bool)
    first[1:] = (r[1:] != r[:-1]) | (h["tax_id"][1:] != h["tax_id"][:-1]) | (h["gi"][1:] != h["gi"][:-1])
    offs = np.zeros(n_reads + 1, np.uint64)
    offs[1:] = np.cumsum(np.bincount(r[first], minlength=n_reads))
    return h[first], offs


def split_parts(rng, read, fields, n_reads, n_parts):
    """Deals each hit to one of n_parts parts, unevenly and differently per read (a read often has no hits in some
    parts); a read's hits keep their order within a part.  Returns [(HIT_DTYPE hits in read order, int32 hits per
    read)] per part."""
    skew = np.floor(n_parts * rng.random(len(read)) ** 3).astype(np.int64)
    part = (skew + rng.integers(0, n_parts, n_reads)[read]) % n_parts
    parts = []
    for p in range(n_parts):
        sel = np.nonzero(part == p)[0]
        sel = sel[np.argsort(read[sel], kind="stable")]
        h = np.zeros(len(sel), HIT_DTYPE)
        for f, v in fields.items():
            h[f] = v[sel]
        parts.append((h, np.bincount(read[sel], minlength=n_reads).astype(np.int32)))
    return parts


def _with_edges(rng, v, edges, frac):
    """v with a fraction `frac` of its entries replaced by values drawn from `edges`."""
    v = v.copy()
    m = rng.random(len(v)) < frac
    v[m] = rng.choice(np.asarray(edges, v.dtype), int(m.sum()))
    return v


def make_keys(rng, sizes, mode):
    """Per-read (tax, edit) keys, sizes[i] of them for read i.  Modes: "random" (full 32-bit range), "equal" (one key
    repeated per read), "few" (a handful of TaxIDs and edits: many duplicates), "sorted" and "reverse" (few TaxIDs,
    keys ascending / descending within a read).  0 and 0xFFFFFFFF occur in both fields; (0xFFFFFFFF, 0xFFFFFFFF) is the
    sorts' padding key ~0."""
    sizes = np.asarray(sizes, np.int64)
    n = int(sizes.sum())
    read = np.repeat(np.arange(len(sizes)), sizes)
    if mode == "random":
        tax = _with_edges(rng, rng.integers(0, 1 << 32, n, dtype=np.uint64).astype(np.uint32), [0, 1, U32 - 1, U32], .05)
        edit = _with_edges(rng, rng.integers(0, 1 << 32, n, dtype=np.uint64).astype(np.uint32), [0, U32], .05)
    elif mode == "equal":
        per = np.stack([rng.integers(0, 1 << 32, len(sizes), dtype=np.uint64).astype(np.uint32),
                        rng.integers(0, 64, len(sizes)).astype(np.uint32)], axis=1)
        per[::3] = [U32, U32]
        per[1::7] = [0, 0]
        per[2::7] = [0, U32]
        per[3::7] = [U32, 0]
        tax, edit = per[read, 0], per[read, 1]
    else:
        tax = rng.choice(np.array([0, 1, 7, 12345, U32 - 1, U32], np.uint32), n)
        edit = rng.choice(np.array([0, 1, 2, 3, U32 - 1, U32], np.uint32), n)
        if mode != "few":
            order = np.lexsort((edit, tax, read)) if mode == "sorted" else np.lexsort((~edit, ~tax, read))
            tax, edit = tax[order], edit[order]
    return read, tax, edit


# keys per read: each class of the segmented sort (none at <= 1, warp <= 32, shared memory <= 4096 padded to a power
# of two >= 64, global memory above) on both sides of its boundaries
SEGMENT_SIZES = [0, 1, 2, 3, 16, 17, 31, 32, 33, 63, 64, 65, 127, 4095, 4096, 4097, 8191, 10000, 70001]
MODES = ["random", "equal", "few", "sorted", "reverse"]


def test_numpy_references_match_the_oracle(oracle):
    """The numpy references of this file against the oracle's restatement of mtsv-collapse, on random small inputs
    with many duplicate TaxIDs, GIs, edits and offsets."""
    rng = np.random.default_rng(1)
    for trial in range(30):
        n_reads, n_parts = int(rng.integers(0, 40)), int(rng.integers(1, 5))
        sizes = rng.integers(0, 25, n_reads)
        read = np.repeat(np.arange(n_reads), sizes)
        n = len(read)
        fields = dict(tax_id=rng.choice(np.array([0, 3, 9, U32], np.uint32), n),
                      gi=rng.choice(np.array([0, 1, U32], np.uint32), n),
                      offset=rng.choice(np.array([0, 5, (1 << 64) - 1], np.uint64), n),
                      edit=rng.choice(np.array([0, 1, 2, U32], np.uint32), n))
        parts = split_parts(rng, read, fields, n_reads, n_parts)
        parts_o = []
        for h, c in parts:
            o = np.zeros(n_reads + 1, np.uint64)
            o[1:] = np.cumsum(c)
            parts_o.append((h, o))
        pairs, offs = ref_taxid(read, fields["tax_id"], fields["edit"], n_reads)
        want_pairs, want_off = oracle.collapse_taxid(parts_o)
        assert np.array_equal(offs, want_off) and np.array_equal(pairs, want_pairs.reshape(-1, 2)), trial
        all_hits = np.concatenate([h for h, _ in parts])
        all_read = np.concatenate([np.repeat(np.arange(n_reads), c) for _, c in parts])
        got, goff = ref_taxid_gi(all_read, all_hits, n_reads)
        want, woff = oracle.collapse_taxid_gi(parts_o)
        assert np.array_equal(goff, woff), trial
        for f in ("tax_id", "gi", "offset", "edit"):
            assert np.array_equal(got[f], want[f]), (trial, f)


# ------------------------------------------------------------------------------------------------
# the merge and the sort through mtsvgpu_collapse_device
# ------------------------------------------------------------------------------------------------
def _to_device(parts):
    import torch
    hits = [torch.from_numpy(np.frombuffer(h.tobytes() or bytes(24), np.uint8).copy()).cuda() for h, _ in parts]
    counts = [torch.from_numpy(c if len(c) else np.zeros(1, np.int32)).cuda() for _, c in parts]
    return hits, counts


def _collapse_check(rng, read, tax, edit, n_reads, n_parts, what):
    from mtsv_tools_b200 import chunked
    parts = split_parts(rng, read, dict(tax_id=tax, edit=edit), n_reads, n_parts)
    want_pairs, want_off = ref_taxid(read, tax, edit, n_reads)
    pairs, offs = chunked.collapse_parts_device(0, None, *_to_device(parts), n_reads)
    got_off = offs.cpu().numpy().astype(np.uint64)
    assert np.array_equal(got_off, want_off), "%s: offsets differ at reads %s" % (
        what, np.nonzero(got_off != want_off)[0][:8])
    got = pairs.cpu().numpy().view(np.uint32).reshape(-1, 2)
    bad = np.nonzero(np.any(got != want_pairs, axis=1))[0] if len(got) == len(want_pairs) else [len(got)]
    assert len(bad) == 0, "%s: records differ from %s on" % (what, bad[:8])


@pytest.mark.gpu
@pytest.mark.parametrize("n_parts", [1, 2, 16])
@pytest.mark.parametrize("mode", MODES)
def test_collapse_every_sort_class(n_parts, mode):
    """Reads of every segment size of SEGMENT_SIZES in one call (the small ones several times), shuffled, their hits
    dealt unevenly over the parts."""
    rng = np.random.default_rng([n_parts, MODES.index(mode)])
    sizes = [s for s in SEGMENT_SIZES for _ in range(4 if s <= 127 else 1)]
    sizes = np.asarray(sizes)[rng.permutation(len(sizes))]
    read, tax, edit = make_keys(rng, sizes, mode)
    _collapse_check(rng, read, tax, edit, len(sizes), n_parts, "%s, %d parts" % (mode, n_parts))


@pytest.mark.gpu
def test_collapse_scan_tiles():
    """0 reads; 2047, 2048 and 2049 reads (one scan tile is 2048 entries); 2048 x 1024 + 1 reads, mostly without
    hits, so that the tile sums exceed one 1024-thread pass and the scan carries between passes."""
    rng = np.random.default_rng(7)
    for n_reads in (0, 2047, 2048, 2049, 2048 * 1024 + 1):
        sizes = np.zeros(n_reads, np.int64)
        if n_reads < 4096:
            sizes[:] = rng.integers(0, 5, n_reads)
        else:
            sizes[rng.integers(0, n_reads, 20000)] = rng.integers(1, 40, 20000)
            sizes[[0, 2047, 2048, 1024 * 2048 - 1, 1024 * 2048, n_reads - 1]] = [3, 1, 2, 5, 1, 4097]
        for n_parts in (1, 3):
            read, tax, edit = make_keys(rng, sizes, "few")
            _collapse_check(rng, read, tax, edit, n_reads, n_parts, "%d reads, %d parts" % (n_reads, n_parts))


@pytest.mark.gpu
def test_collapse_scratch_grows_and_shrinks():
    """Calls of growing, then shrinking, sizes on one device: the grow-only scratch of the collapse is reused with
    contents left over from larger calls."""
    rng = np.random.default_rng(8)
    for n_reads, big in ((10, 0), (3000, 40), (60000, 5000), (400000, 20000), (60000, 0), (3000, 4097), (10, 33),
                         (0, 0), (2049, 100)):
        sizes = rng.geometric(0.2, n_reads) - 1
        if n_reads and big:
            sizes[rng.integers(0, n_reads)] = big
        read, tax, edit = make_keys(rng, sizes, "few" if n_reads % 2 else "random")
        _collapse_check(rng, read, tax, edit, n_reads, 2, "%d reads" % n_reads)


@pytest.mark.gpu
@pytest.mark.parametrize("n_parts", [1, 2, 16])
def test_collapse_taxid_gi(n_parts):
    """Mode TaxIdGi: minimum edit, ties to the smallest offset, listed by (TaxID, GI); heavy ties on edit and offset,
    groups split across parts, up to 2000 hits per read (the kernel compares every pair of a read's hits)."""
    from mtsv_tools_b200 import chunked
    rng = np.random.default_rng(n_parts)
    sizes = np.asarray([0, 1, 2, 3, 31, 32, 33, 100, 500, 1999, 2000] * 3)
    sizes = sizes[rng.permutation(len(sizes))]
    n_reads = len(sizes)
    read = np.repeat(np.arange(n_reads), sizes)
    n = len(read)
    wide = read % 2 == 0  # even reads: wide values, odd reads: a few values, ties everywhere

    def pick(wide_values, few_values):
        return np.where(wide, wide_values, rng.choice(np.asarray(few_values, np.uint64), n))

    fields = dict(tax_id=pick(rng.integers(0, 40, n, dtype=np.uint64), [0, 5, U32]).astype(np.uint32),
                  gi=pick(rng.integers(0, 1 << 32, n, dtype=np.uint64), [0, 1, U32]).astype(np.uint32),
                  offset=pick(rng.integers(0, 1 << 63, n, dtype=np.uint64), [0, 2, (1 << 64) - 1]),
                  edit=pick(rng.integers(0, 1 << 32, n, dtype=np.uint64), [0, 1, U32]).astype(np.uint32))
    parts = split_parts(rng, read, fields, n_reads, n_parts)
    # the order the device combines them in (part by part within a read) and the reference of that list
    all_hits = np.concatenate([h for h, _ in parts])
    all_read = np.concatenate([np.repeat(np.arange(n_reads), c) for _, c in parts])
    want, want_off = ref_taxid_gi(all_read, all_hits, n_reads)
    hits, offs = chunked.collapse_parts_device_taxid_gi(0, None, *_to_device(parts), n_reads)
    got = np.frombuffer(hits.cpu().numpy().tobytes(), dtype=HIT_DTYPE)
    assert np.array_equal(offs.cpu().numpy().astype(np.uint64), want_off)
    for f in ("tax_id", "gi", "offset", "edit"):
        assert np.array_equal(got[f], want[f]), f


# ------------------------------------------------------------------------------------------------
# the binning pipeline at its per-strand boundaries
# ------------------------------------------------------------------------------------------------
SEED = 18      # seed_size
EDIT_RATE = 0.13
LENS = (100, 64, 65, 71, 83, 97)  # read lengths; uniform batches have L_MAX
L_MAX = max(LENS)
SEG = 300      # length of the copied segment
SRC = 18       # the reads' region [SRC, SRC + L) of the segment
SPACER = 2 * (L_MAX + int(np.ceil(L_MAX * EDIT_RATE))) + 16  # random bases between the copies of the spaced layout
TANDEM = 136   # period of the tandem layout: the segment's first TANDEM bases, which hold the reads' region
# seed hits per strand: the sort (min_count 16, 32), coalesce (light <= 16, heavy <= 1024, monster above), rank
# (16), select and leader (512) boundaries, and the sort's 4096
M_VALUES = [15, 16, 17, 32, 33, 512, 513, 1024, 1025, 4096, 4097]
LAYOUTS = ["distinct", "shared_rc", "spaced", "tandem"]
_ACGT = np.frombuffer(b"ACGT", np.uint8)


def _k(L):
    """The edit budget of a read of L bases."""
    return int(np.ceil(L * EDIT_RATE))


def _mutate(rng, seq, allowed, n_sub):
    """seq with n_sub substitutions (each to a different base) at distinct positions drawn from `allowed`."""
    seq = seq.copy()
    pos = rng.choice(allowed, n_sub, replace=False)
    code = np.searchsorted(_ACGT, seq[pos])
    seq[pos] = _ACGT[(code + rng.integers(1, 4, n_sub)) % 4]
    return seq


def _allowed(n):
    """Positions in [0, n) outside every read's first and last SEED bases (reads start at SRC)."""
    keep = np.ones(n, bool)
    keep[SRC:SRC + SEED] = False
    for L in LENS:
        keep[SRC + L - SEED:SRC + L] = False
    return np.nonzero(keep)[0]


class BoundaryRef:
    """A reference whose group g holds m = M_VALUES[g] copies of a random segment, each with 0-3 substitutions
    outside the seeds of the reads drawn from it.  Layouts:
      distinct  - every copy its own sequence under its own TaxID;
      shared_rc - every copy its own sequence under one of 7 TaxIDs, plus m / 3 reverse-complemented copies under the
                  same TaxIDs (TaxIDs hit on both strands; the forward strand holds m candidates of 7 TaxIDs, which
                  puts m = 512 / 513 on both sides of the leader map's limit);
      spaced    - the group's copies in one sequence, SPACER random bases apart: consecutive seed hits of a strand are
                  at least 2(L + k) apart, every gap is a coalesce chunk boundary;
      tandem    - the first TANDEM bases of each copy, back to back in one sequence: consecutive seed hits are TANDEM
                  apart, less than 2(L + k), so there is no chunk boundary, and more than L + 2k, so every hit is its
                  own candidate.
    A read of group g has one seed per strand (seed_gap > L - seed_size): its first SEED bases, which every forward
    copy holds once, and the reverse complement of its last SEED bases, which every reverse-complemented copy holds
    once.  hits[g]: the seed hits of one read of group g, both strands together."""

    def __init__(self, layout, seed):
        rng = np.random.default_rng(seed)
        allowed = _allowed(SEG)
        seqs, tax, self.bases, self.hits = [], [], [], []
        next_tax = 100
        for g, m in enumerate(M_VALUES):
            base = _ACGT[rng.integers(0, 4, SEG)]
            self.bases.append(base)
            copies = [_mutate(rng, base, allowed, int(rng.integers(0, 4))) for _ in range(m)]
            self.hits.append(m)
            if layout == "distinct":
                seqs += copies
                tax += list(range(next_tax, next_tax + m))
                next_tax += m
            elif layout == "shared_rc":
                n_rc = m // 3
                copies += [np.frombuffer(synth.revcomp(_mutate(rng, base, allowed, int(rng.integers(0, 4))).tobytes()),
                                         np.uint8) for _ in range(n_rc)]
                self.hits[-1] += n_rc
                seqs += copies
                tax += [next_tax + (i * 5) % 7 for i in range(len(copies))]
                next_tax += 7
            else:
                parts = []
                for c in copies:
                    parts += [c, _ACGT[rng.integers(0, 4, SPACER)]] if layout == "spaced" else [c[:TANDEM]]
                seqs.append(np.concatenate(parts))
                tax.append(next_tax)
                next_tax += 1
        self.seqs = [s.tobytes() for s in seqs]
        self.gi = np.arange(1, len(seqs) + 1, dtype=np.uint32)
        self.tax = np.asarray(tax, np.uint32)

    def reads(self, g, n, ragged, seed):
        """n reads of group g from the segment's region at SRC, 0-2 substitutions outside both seeds."""
        rng = np.random.default_rng(seed)
        out = []
        for i in range(n):
            L = LENS[i % len(LENS)] if ragged else L_MAX
            r = self.bases[g][SRC:SRC + L]
            out.append(_mutate(rng, r, np.arange(SEED, L - SEED), int(rng.integers(0, 3))).tobytes())
        return out

    def sites(self, ix, g):
        """Text positions of the forward seed of group g's reads, ascending (oracle index)."""
        r, lo, up, _ = ix.backward_search(self.bases[g][SRC:SRC + SEED].tobytes())
        assert r == 2
        return np.sort(np.array([ix.locate(row)[0] for row in range(lo, up)], np.int64))


def _boundary_params(oracle):
    from tests.test_gpu_parity import _params
    return _params(oracle, edit_rate=EDIT_RATE, seed_gap=L_MAX, max_hits=10000, tune_max_hits=10000)


def _check_everything(oracle, g, ix, reads, po, pg, seed_hits, one_sub_batch=False):
    """Every bin and assign entry point against the oracle; with `seed_hits`, the oracle's and every call's count of
    seed hits against it (the library does not count the hits of strands it can tell will never be accepted, such as
    reads with more N than their edit budget, so the two counts agree only on batches without such reads).
    one_sub_batch: every call ran the whole batch as one device sub-batch (so its kernels saw all of its reads)."""
    import torch
    from mtsv_tools_b200.index import pack_reads, pack_reads_planes
    from tests.test_assign import _check, _from_device
    names = ["r%d" % i for i in range(len(reads))]
    ctr = oracle.Counters()
    h1, o1 = ix.bin_reads(reads, po, threads=8, counters=ctr)
    if seed_hits is not None:
        assert ctr.rows_located == seed_hits, (ctr.rows_located, seed_hits)

    def same(h, o, what):
        assert np.array_equal(np.asarray(o, np.uint64), o1), "%s: hit offsets differ at reads %s" % (
            what, np.nonzero(np.asarray(o, np.uint64) != o1)[0][:8])
        for f in ("tax_id", "gi", "offset", "edit"):
            assert np.array_equal(h[f], h1[f]), (what, f)
        stats(what)

    def stats(what=""):
        st = g.last_batch_stats()
        assert seed_hits is None or st["n_seed_hits"] == seed_hits, what
        assert not one_sub_batch or st["n_sub_batches"] == 1, what

    same(*g.bin_reads(reads, pg), "bin")
    same(*g.bin_reads_packed(*pack_reads_planes(reads), pg), "bin packed")
    cat, off = pack_reads(reads)
    d_seqs = torch.from_numpy(np.concatenate([cat, np.zeros(1, np.uint8)])).cuda()
    d_off = torch.from_numpy(off.astype(np.int64)).cuda()
    dh, do, nh = g.bin_reads_device(d_seqs.data_ptr(), d_off.data_ptr(), len(reads), pg)
    same(_from_device(dh, nh, HIT_DTYPE), _from_device(do, len(reads) + 1, np.dtype(np.uint64)), "bin device")
    _check(g, reads, names, pg, oracle.results_lines(names, h1, o1, False))
    stats("assign")
    return h1, o1


@pytest.mark.gpu
@pytest.mark.parametrize("layout", LAYOUTS)
def test_bin_at_per_strand_boundaries(oracle, layout):
    """For each m of M_VALUES: 20 reads of uniform and 20 of ragged lengths (8 and 8 from m = 4096 on) whose two
    strands have exactly the seed hits the layout gives them (n_seed_hits proves it), then all groups in one batch."""
    from tests.test_gpu_parity import _gpu_index
    ref = BoundaryRef(layout, seed=LAYOUTS.index(layout) + 40)
    ix = oracle.Index.build(ref.seqs, ref.gi, ref.tax, 64, 32)
    if layout in ("spaced", "tandem"):  # where coalesce_monster_kernel can and cannot cut a strand's hits
        for grp, m in enumerate(M_VALUES):
            gaps = np.diff(ref.sites(ix, grp))
            assert len(gaps) == m - 1
            for L in LENS:
                if layout == "spaced":
                    assert gaps.min() >= 2 * (L + _k(L)), (m, L, gaps.min())
                else:
                    assert L + 2 * _k(L) < gaps.min() and gaps.max() < 2 * (L + _k(L)), (m, L, gaps.min(), gaps.max())
    po, pg = _boundary_params(oracle)
    both_strands = 0
    with _gpu_index(ix) as g:
        mixed = []
        for grp, m in enumerate(M_VALUES):
            n = 20 if m < 4096 else 8
            for ragged in (False, True):
                reads = ref.reads(grp, n, ragged, seed=1000 * grp + ragged)
                h, o = _check_everything(oracle, g, ix, reads, po, pg, n * ref.hits[grp])
                if layout == "distinct":  # every copy passes: one hit per copy and read
                    assert len(h) == n * m
                if layout == "shared_rc":
                    for i in range(len(reads)):
                        t = h["tax_id"][int(o[i]):int(o[i + 1])]
                        both_strands += len(t) - len(np.unique(t))
            mixed += ref.reads(grp, 3, True, seed=77 + grp)
        _check_everything(oracle, g, ix, mixed, po, pg, 3 * sum(ref.hits))
    if layout == "shared_rc":
        assert both_strands > 0  # TaxIDs hit on both strands: the assign merge keeps the smaller edit


READ_LENGTHS = [64, 65, 128, 129, 192, 193, 253, 254, 255]


@pytest.mark.gpu
def test_bin_read_length_sweep(oracle, small_ref, small_index):
    """Uniform batches of each length of READ_LENGTHS: the warp verifier at 1-4 words in its UNIFORM instantiation,
    the per-lane + SW route from 254 bases on.  A batch mixing the lengths up to 253 (the warp verifier at 4 words,
    not UNIFORM), and one mixing all of them.  Each batch is one device sub-batch, so its kernels see all its reads."""
    from tests.test_gpu_parity import _gpu_index, _params
    cat, off = small_ref[0], small_ref[1]
    po, pg = _params(oracle)
    mixed = []
    with _gpu_index(small_index) as g:
        for L in READ_LENGTHS:
            rc, ro = synth.make_reads(cat, off, 300, L, seed=L)
            reads = [rc[int(ro[i]):int(ro[i + 1])].tobytes() for i in range(300)]
            h, _ = _check_everything(oracle, g, small_index, reads, po, pg, None, one_sub_batch=True)
            assert len(h) > 100, L
            mixed += reads[:40]
        rng = np.random.default_rng(3)
        short = [r for r in mixed if len(r) <= 253]
        for batch in (short, mixed):
            order = rng.permutation(len(batch))
            _check_everything(oracle, g, small_index, [batch[i] for i in order], po, pg, None, one_sub_batch=True)
