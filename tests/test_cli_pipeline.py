"""mtsv-binner's host pipeline (mtsv_tools_b200/csrc/mtsv_binner_main.cpp: reader thread, parse and format workers,
GPU threads, ordered writer) built with AddressSanitizer and driven on the CPU through --dump-reads-mt, which runs every
stage except the library call.  Leak detection stays on: these runs never initialise the CUDA runtime."""
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "mtsv_tools_b200")
CSRC = os.path.join(PKG, "csrc")
BIN = os.path.join(PKG, "bin", "mtsv-binner")
N_READS = 400_000  # 100 bases each: about 85 MB, some 20 blocks of 4 MiB
MALFORMED = "@x\nACGT\n+\nII\n@y\nAC\n+\nII\n"  # x's quality ends in the "@y" line; "AC" then has no quality


def _run(exe, *args):
    return subprocess.run([exe, *args], capture_output=True, text=True)


@pytest.fixture(scope="module")
def asan_binner(tmp_path_factory):
    if not os.path.exists(BIN):
        subprocess.check_call(["make", "-s", "-C", CSRC])
    exe = str(tmp_path_factory.mktemp("asan") / "mtsv-binner")
    subprocess.check_call(["g++", "-std=c++17", "-pthread", "-g", "-fsanitize=address", "-fno-omit-frame-pointer",
                           "-o", exe, os.path.join(CSRC, "mtsv_binner_main.cpp"), "-L" + PKG, "-lmtsv_b200", "-lz",
                           "-Wl,-rpath," + PKG])
    return exe


@pytest.fixture(scope="module")
def good_fastq(tmp_path_factory):
    """N_READS well-formed FASTQ records r0000000, r0000001, ... of 100 random bases."""
    L, n = 100, N_READS
    rows = np.empty((n, 9 + 1 + L + 3 + L + 1), np.uint8)
    rows[:, :2] = np.frombuffer(b"@r", np.uint8)
    for d in range(7):
        rows[:, 8 - d] = 48 + (np.arange(n) // 10 ** d) % 10
    rows[:, 9] = 10
    rows[:, 10:10 + L] = np.frombuffer(b"ACGT", np.uint8)[np.random.default_rng(7).integers(0, 4, (n, L))]
    rows[:, 10 + L:13 + L] = np.frombuffer(b"\n+\n", np.uint8)
    rows[:, 13 + L:13 + 2 * L] = ord("I")
    rows[:, -1] = 10
    path = tmp_path_factory.mktemp("reads") / "good.fq"
    rows.tofile(str(path))
    return path


def test_a_failing_run_does_not_touch_freed_state(asan_binner, good_fastq, tmp_path):
    """A malformed record after many blocks fails the run while parse and format tasks are still queued.  Those
    tasks must finish before the state they use is destroyed; before, they could write into freed memory."""
    bad = tmp_path / "bad.fq"
    bad.write_bytes(good_fastq.read_bytes() + MALFORMED.encode())
    for _ in range(5):
        r = _run(asan_binner, "--dump-reads-mt", "--fastq", str(bad), "--threads", "16")
        assert r.returncode == 12, r.stderr[-4000:]
        assert "Sanitizer" not in r.stderr, r.stderr[-4000:]


@pytest.mark.parametrize("extra", [["--threads", "16"], ["--threads", "3", "--batch-reads", "1000"],
                                   ["--read-offset", "1234"]])
def test_a_clean_run_prints_what_the_regular_binary_prints(asan_binner, good_fastq, extra):
    r = _run(asan_binner, "--dump-reads-mt", "--fastq", str(good_fastq), *extra)
    assert r.returncode == 0 and "Sanitizer" not in r.stderr, r.stderr[-4000:]
    want = _run(BIN, "--dump-reads-mt", "--fastq", str(good_fastq), *extra)
    assert want.returncode == 0, want.stderr
    assert r.stdout == want.stdout
    assert r.stdout.count("\n") == N_READS - (1234 if "--read-offset" in extra else 0)
