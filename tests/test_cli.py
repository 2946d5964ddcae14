"""The mtsv-binner command-line driver (mtsv_tools_b200/csrc/mtsv_binner_main.cpp): reference flag surface,
FASTA/FASTQ(.gz) parsing, exit codes, results text and resume — src/bin/mtsv-binner.rs, src/binner.rs."""
import gzip
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "mtsv_tools_b200", "bin", "mtsv-binner")


def _run(*args):
    return subprocess.run([BIN, *args], capture_output=True, text=True)


@pytest.fixture(scope="module", autouse=True)
def built():
    if not os.path.exists(BIN):
        subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "mtsv_tools_b200", "csrc")])


def test_fastx_parsing(tmp_path):
    fa = tmp_path / "t.fa"
    fa.write_text(">r1 desc\nACGT\nACGT\n>r2\nNNNN\n\n>r3 x\nAC\n")
    out = _run("--dump-reads", "--fasta", str(fa))
    assert out.returncode == 0 and out.stdout == "r1\tACGTACGT\nr2\tNNNN\nr3\tAC\n"
    fq = tmp_path / "t.fq"
    fq.write_text("@q1 d\nACGT\n+\nIIII\n@q2\nAC\nGT\n+q2\n@III\n@q3\n\n+\n\n@q4\nA\n+\nI\n")
    want = "q1\tACGT\nq2\tACGT\nq3\t\nq4\tA\n"
    assert _run("--dump-reads", "--fastq", str(fq)).stdout == want
    gz = tmp_path / "t.fq.gz"
    with gzip.open(gz, "wt") as f:  # src/binner.rs:474-499: gz and plain read identically
        f.write(fq.read_text())
    assert _run("--dump-reads", "--fastq", str(gz)).stdout == want
    assert _run("--dump-reads", "--fastq", str(gz), "--read-offset", "2").stdout == "q3\t\nq4\tA\n"
    bad = tmp_path / "bad.fq"
    bad.write_text("@q1\nACGT\n+\nII\n")
    assert _run("--dump-reads", "--fastq", str(bad)).returncode == 12  # src/binner.rs:81-84


def test_dump_reads_give_the_records_written(tmp_path):
    """--dump-reads prints id<TAB>sequence of every record; --dump-reads-mt drives the production path (block reader,
    parser pool, ordered writer) without a GPU and prints id<TAB>length.  Both must give the records the generators
    wrote, on awkward files and in particular where 4 MiB block edges cut lines and records."""
    rng = np.random.default_rng(3)

    def bases(alphabet, L):
        return rng.choice(np.frombuffer(alphabet, np.uint8), size=L).tobytes().decode()

    def fastq(n, multi=False, crlf=False, final_newline=True):
        nl = "\r\n" if crlf else "\n"
        parts, recs = [], []
        for i in range(n):
            L = int(rng.integers(0, 400))
            s = bases(b"ACGTN", L)
            q = bases(b"@+I#>", L)  # quality lines that look like headers / separators
            recs.append(("r%d" % i, s))
            if multi and L > 10:
                k = int(rng.integers(1, L))
                s, q = s[:k] + nl + s[k:], q[:k // 2] + nl + q[k // 2:]
            parts.append("@r%d extra words%s%s%s+%s%s%s" % (i, nl, s, nl, nl, q, nl))
            if i % 97 == 0:
                parts.append(nl)  # blank line between records
        t = "".join(parts)
        return (t if final_newline else t.rstrip("\r\n")), recs

    def fasta(n, crlf=False, final_newline=True, long_record=None):
        nl = "\r\n" if crlf else "\n"
        parts, recs = [], []
        for i in range(n):
            L = 9 << 20 if i == long_record else int(rng.integers(0, 900))  # (9 MiB: more than two blocks)
            s = bases(b"ACGTNacgtn", L)
            recs.append(("s%d-%d" % (i, i % 7), s))
            lines = [s[j:j + 70] for j in range(0, L, 70)] or [""]
            head = ">s%d-%d desc%s" % (i, i % 7, nl)
            if i == long_record:  # pad the header so that the first 4 MiB block ends right after a sequence line
                start = sum(map(len, parts)) + len(head)
                head = head.replace(" desc", " desc" + " " * (((4 << 20) - start) % (70 + len(nl))))
            parts.append(head + nl.join(lines) + nl)
        t = "".join(parts)
        return (t if final_newline else t.rstrip("\r\n")), recs

    def dump(recs):
        return "".join("%s\t%s\n" % r for r in recs)

    def lens(recs):
        return "".join("%s\t%d\n" % (i, len(s)) for i, s in recs)

    cases = [("a.fq", fastq(30000), "--fastq"), ("b.fq", fastq(3000, multi=True, crlf=True), "--fastq"),
             ("c.fq", fastq(2000, final_newline=False), "--fastq"), ("d.fa", fasta(20000), "--fasta"),
             ("e.fa", fasta(1500, crlf=True, final_newline=False), "--fasta"),
             ("f.fa", fasta(3000, long_record=2000), "--fasta")]
    for name, (text, recs), flag in cases:
        f = tmp_path / name
        f.write_text(text, newline="")
        got = _run("--dump-reads", flag, str(f))
        assert got.returncode == 0 and got.stdout == dump(recs), name
        for extra in ([], ["--threads", "3", "--batch-reads", "1000"], ["--read-offset", "1234"]):
            got = _run("--dump-reads-mt", flag, str(f), *extra)
            assert got.returncode == 0, (name, extra, got.stderr)
            assert got.stdout == lens(recs[1234:] if "--read-offset" in extra else recs), (name, extra)
    gzf = tmp_path / "a.fq.gz"
    with gzip.open(gzf, "wt", newline="") as f:
        f.write(cases[0][1][0])
    assert _run("--dump-reads-mt", "--fastq", str(gzf)).stdout == lens(cases[0][1][1])
    # malformed input: quality shorter than the sequence, in the middle of a large file
    bad = tmp_path / "bad.fq"
    good = cases[0][1][0][:5_000_000].rsplit("@r", 1)[0]
    bad.write_text(good + "@x\nACGT\n+\nII\n" + "@y\nAC\n+\nII\n")
    assert _run("--dump-reads-mt", "--fastq", str(bad)).returncode == 12
    got = _run("--dump-reads", "--fastq", str(bad))  # the records before the malformed one, then the error
    want = cases[0][1][1][:good.count("@r")] + [("x", "ACGT")]  # (x's quality ends in the "@y" line; "AC" is bad)
    assert got.returncode == 12 and got.stdout == dump(want)


def test_exit_codes_without_gpu(tmp_path):
    fa = tmp_path / "t.fa"
    fa.write_text(">r1\nACGT\n")
    assert _run("--fasta", str(fa), "--index", "/nonexistent").returncode == 3  # no results path (:262-265)
    r = _run("--fasta", str(fa), "--index", "/nonexistent", "--results", str(tmp_path / "r.txt"))
    assert r.returncode == 2 and "cannot open" in r.stderr  # query error (:319-322)
    assert _run("--fasta", str(fa), "--index", "x", "--results", "y", "--edit-rate", "1.5").returncode == 101
    assert _run("--fasta", str(fa), "--index", "x", "--results", "y", "--min-seed", "0").returncode == 101


@pytest.mark.gpu
def test_cli_end_to_end(oracle, tmp_path):
    from mtsv_tools_b200 import synth
    cat, off, gi, tax = synth.make_reference(8, 20000, seed=1, n_frac=0.002, shared_frac=0.1, seqs_per_taxid=2)
    ix = oracle.Index.build((cat, off), gi, tax, 64, 32)
    index_path = str(tmp_path / "ref.index")
    ix.write(index_path)
    rc, ro = synth.make_reads(cat, off, 3000, 150, seed=2)
    names = ["read_%d" % i for i in range(3000)]
    fq = tmp_path / "reads.fq.gz"
    with gzip.open(fq, "wt") as f:
        for i, n in enumerate(names):
            s = bytes(rc[int(ro[i]):int(ro[i + 1])]).decode()
            f.write("@%s some description\n%s\n+\n%s\n" % (n, s, "I" * len(s)))
    hits, offs = ix.bin_reads((rc, ro), oracle.default_params(), threads=4)
    for long in (False, True):
        res = tmp_path / ("res_%d.txt" % long)
        args = ["--fastq", str(fq), "--index", index_path, "--results", str(res), "--threads", "8"]
        if long:
            args += ["--output-format", "long"]
        r = _run(*args)
        assert r.returncode == 0, r.stderr
        want = oracle.results_lines(names, hits, offs, long)
        assert sorted(res.read_text().splitlines(True)) == sorted(want)
    # resume: results holding the first 1000 reads' lines -> the run continues after the last id present
    res = tmp_path / "resume.txt"
    first = oracle.results_lines(names[:1000], hits[:int(offs[1000])], offs[:1001], False)
    res.write_text("".join(first))
    r = _run("--fastq", str(fq), "--index", index_path, "--results", str(res))
    assert r.returncode == 0, r.stderr
    last_present = max(i for i in range(1000) if offs[i + 1] > offs[i])
    tail = oracle.results_lines(names[last_present + 1:], hits, offs[last_present + 1:], False)
    assert res.read_text() == "".join(first) + "".join(tail)
    # --force-overwrite starts over; parameters are honoured
    r = _run("--fastq", str(fq), "--index", index_path, "--results", str(res), "--force-overwrite",
             "--edit-rate", "0.05", "--seed-interval", "10", "--max-candidates", "2")
    assert r.returncode == 0, r.stderr
    h2, o2 = ix.bin_reads((rc, ro), oracle.default_params(edit_rate=0.05, seed_gap=10, max_candidates=2), threads=4)
    assert res.read_text() == "".join(oracle.results_lines(names, h2, o2, False))


# ------------------------------------------------------------------------------------------------
# mtsv-build (mtsv_tools_b200/csrc/mtsv_build_main.cpp): src/bin/mtsv-build.rs, src/builder.rs, src/io.rs:35-184
# ------------------------------------------------------------------------------------------------
BUILD = os.path.join(ROOT, "mtsv_tools_b200", "bin", "mtsv-build")


def _build(*args):
    return subprocess.run([BUILD, *args], capture_output=True, text=True)


def test_mtsv_build_input_errors_without_gpu(tmp_path):
    """Everything that fails before the index is built exits 1 with the reference's messages: header format
    (src/util.rs:26-55), mapping file rules (src/io.rs:35-112), records missing from the mapping (:153-184)."""
    fa = tmp_path / "db.fa"
    fa.write_text(">12-34\nACGT\n>56-78-9\nACGT\n")
    r = _build("--fasta", str(fa), "--index", str(tmp_path / "x.index"))
    assert r.returncode == 1 and "Invalid header: 56-78-9" in r.stderr
    fa.write_text(">12-34\nACGT\n>ab-78\nACGT\n")
    r = _build("--fasta", str(fa), "--index", str(tmp_path / "x.index"))
    assert r.returncode == 1 and "Invalid integer: ab" in r.stderr
    assert _build("--fasta", str(fa)).returncode == 1  # --index is required
    assert _build("--fasta", str(tmp_path / "nope.fa"), "--index", str(tmp_path / "x.index")).returncode == 1
    fa.write_text(">foo desc\nACGT\n>bar\nTTTT\n")
    mp = tmp_path / "map.tsv"
    mp.write_text("header\ttaxid\n foo\t2\n")
    r = _build("--fasta", str(fa), "--index", str(tmp_path / "x.index"), "--mapping", str(mp))
    assert r.returncode == 1 and "Missing 'seqid' column" in r.stderr
    mp.write_text("Header, TaxID, GI\nfoo, 2, 1\nfoo, 3, 4\n")
    r = _build("--fasta", str(fa), "--index", str(tmp_path / "x.index"), "--mapping", str(mp))
    assert r.returncode == 1 and "Duplicate header mapping for foo" in r.stderr
    mp.write_text("header taxid seqid\nfoo 2 1\n")
    r = _build("--fasta", str(fa), "--index", str(tmp_path / "x.index"), "--mapping", str(mp))
    assert r.returncode == 1 and "Missing mapping for header bar" in r.stderr
    mp.write_text("header taxid seqid\nfoo x 1\n")
    r = _build("--fasta", str(fa), "--index", str(tmp_path / "x.index"), "--mapping", str(mp))
    assert r.returncode == 1 and "Invalid integer: x" in r.stderr


@pytest.mark.gpu
def test_mtsv_build_writes_the_oracles_index_and_feeds_the_binner(oracle, tmp_path):
    from mtsv_tools_b200 import synth
    cat, off, gi, tax = synth.make_reference(9, 15000, seed=3, n_frac=0.002, shared_frac=0.1)
    tax = np.array([7, 3, 9, 3, 5, 7, 1, 9, 2], dtype=np.uint32)
    fa = tmp_path / "db.fa.gz"
    with gzip.open(fa, "wt") as f:
        for i in range(9):
            s = bytes(cat[int(off[i]):int(off[i + 1])]).decode()
            s = s[:5000].lower() + s[5000:]  # lower case is folded (src/index.rs:543-553)
            f.write(">%d-%d some text\n" % (gi[i], tax[i]))
            for j in range(0, len(s), 60):
                f.write(s[j:j + 60] + "\n")
    ix = oracle.Index.build((cat, off), gi, tax, 64, 32)
    want = tmp_path / "oracle.index"
    ix.write(str(want))
    out = tmp_path / "gpu.index"
    r = _build("--fasta", str(fa), "--index", str(out))
    assert r.returncode == 0, r.stderr
    assert out.read_bytes() == want.read_bytes()
    # other intervals; mapping file instead of ACCESSION-TAXID headers, one record skipped
    ix2 = oracle.Index.build((cat[:int(off[8])], off[:9]), gi[:8], tax[:8], 128, 16)
    ix2.write(str(want))
    fa2 = tmp_path / "db2.fa"
    mp = tmp_path / "map.csv"
    with open(fa2, "w") as f, open(mp, "w") as m:
        m.write("seqid,header,taxid\n")
        for i in range(9):
            f.write(">seq_%d\n%s\n" % (i, bytes(cat[int(off[i]):int(off[i + 1])]).decode()))
            if i < 8:
                m.write("%d,seq_%d,%d\n" % (gi[i], i, tax[i]))
    r = _build("--fasta", str(fa2), "--index", str(out), "--mapping", str(mp), "--skip-missing",
               "--sample-interval", "128", "--sa-sample", "16")
    assert r.returncode == 0 and "Missing mapping for header seq_8, skipping" in r.stderr, r.stderr
    assert out.read_bytes() == want.read_bytes()
    r = _build("--fasta", str(fa2), "--index", str(out), "--mapping", str(mp))
    assert r.returncode == 1
    # the index the GPU builder wrote drives the binner binary to the oracle's result lines
    r = _build("--fasta", str(fa), "--index", str(out))
    assert r.returncode == 0
    rc, ro = synth.make_reads(cat, off, 1000, 150, seed=4)
    names = ["r%d" % i for i in range(1000)]
    fq = tmp_path / "reads.fa"
    with open(fq, "w") as f:
        for i, n in enumerate(names):
            f.write(">%s\n%s\n" % (n, bytes(rc[int(ro[i]):int(ro[i + 1])]).decode()))
    res = tmp_path / "res.txt"
    r = _run("--fasta", str(fq), "--index", str(out), "--results", str(res))
    assert r.returncode == 0, r.stderr
    hits, offs = ix.bin_reads((rc, ro), oracle.default_params(), threads=4)
    assert res.read_text() == "".join(oracle.results_lines(names, hits, offs, False))


@pytest.mark.gpu
def test_cli_two_gpus_give_the_same_file(oracle, tmp_path):
    """--gpus 2: batches go to the devices round-robin, the ordered writer makes the results file identical to the
    one-GPU run (and to the oracle's lines)."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from mtsv_tools_b200 import synth
    cat, off, gi, tax = synth.make_reference(8, 20000, seed=1, n_frac=0.002, shared_frac=0.1, seqs_per_taxid=2)
    ix = oracle.Index.build((cat, off), gi, tax, 64, 32)
    index_path = str(tmp_path / "ref.index")
    ix.write(index_path)
    rc, ro = synth.make_reads(cat, off, 20000, 150, seed=2)
    names = ["read_%d" % i for i in range(20000)]
    fq = tmp_path / "reads.fq"
    with open(fq, "w") as f:
        for i, n in enumerate(names):
            s = bytes(rc[int(ro[i]):int(ro[i + 1])]).decode()
            f.write("@%s\n%s\n+\n%s\n" % (n, s, "I" * len(s)))
    hits, offs = ix.bin_reads((rc, ro), oracle.default_params(), threads=4)
    want = "".join(oracle.results_lines(names, hits, offs, False))
    for gpus in ("1", "2"):
        res = tmp_path / ("res_%s.txt" % gpus)
        r = _run("--fastq", str(fq), "--index", index_path, "--results", str(res), "--gpus", gpus,
                 "--batch-reads", "1500", "--threads", "6")
        assert r.returncode == 0, r.stderr
        assert res.read_text() == want, gpus
