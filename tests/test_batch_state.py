"""The state of one batch call stays with that call: a failed batch leaves nothing on its handle that changes the next
call, and the MTSV_B200_TRACE slice timeline of host-API calls is per call, also with several handles driven from
several threads at once."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from mtsv_tools_b200 import LibraryError, MGIndex, synth
from mtsv_tools_b200.index import Params
from tests.test_assign import small_index, small_ref  # noqa: F401  (fixtures)

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ELIMIT = -7
STEP = 16  # reads per slice: below 1024 the host API cuts equal slices (no ramp)
HIT_CAP = 1000  # max_batch_hits: a slice of ordinary reads stays far below it
SEG, COPIES = 300, 150  # the repeat: COPIES tandem copies of one random segment of SEG bases


def _stats(g):
    """The stats of the last batch without the stage times."""
    st = g.last_batch_stats()
    del st["ms"]
    return st


@pytest.fixture(scope="module")
def repeat_ref(oracle):
    """A random reference plus one sequence that is a tandem repeat; reads from the random part, and one read from
    the repeat whose forward seeds hit every copy."""
    cat, off, gi, tax = synth.make_reference(6, 20000, seed=21, n_frac=0.002, shared_frac=0.1)
    rng = np.random.default_rng(22)
    seg = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, SEG)]
    rep = np.tile(seg, COPIES)
    all_cat = np.concatenate([cat, rep])
    all_off = np.append(off, off[-1] + np.uint64(len(rep))).astype(np.uint64)
    gi = np.append(gi, gi[-1] + 1).astype(np.uint32)
    tax = np.append(tax, tax[-1] + 1).astype(np.uint32)
    ix = oracle.Index.build((all_cat, all_off), gi, tax, 64, 32)
    rc, ro = synth.make_reads(cat, off, 40 * STEP, 150, seed=23)
    good = [rc[int(ro[i]):int(ro[i + 1])].tobytes() for i in range(len(ro) - 1)]
    return ix, good, seg[20:170].tobytes()


def test_failed_batch_leaves_no_state(repeat_ref):
    """A host-API batch of 41 slices on two lanes fails with MTSVGPU_ELIMIT in slice 31 (lane 1): one read of the
    repeat has more seed hits than the handle's max_batch_hits, so its group is split down to that read, which still
    does not fit.  The next call on the same handle, with per-stage timing off and on, gives the results and the stats
    (all but the stage times) of a fresh handle."""
    ix, good, bad_read = repeat_ref
    params = Params(max_hits=10000, tune_max_hits=10000)
    failing = good[:31 * STEP + 5] + [bad_read] + good[31 * STEP + 5:]
    opts = dict(max_batch_hits=HIT_CAP, batch_reads=STEP)

    def from_parts(**kw):
        return MGIndex.from_parts(ix.text, ix.bins(), ix.bwt, ix.sa_sample, ix.sa_sample_rate, **kw)

    with from_parts() as g:  # no cap: the read of the repeat alone is over it
        g.bin_reads([bad_read], params)
        assert g.last_batch_stats()["n_seed_hits"] > HIT_CAP
    for profiling in (False, True):
        for call in ("bin_reads", "assign_reads"):
            with from_parts(**opts) as f:
                f.set_profiling(profiling)
                want = getattr(f, call)(good, params)
                want_st = _stats(f)
            assert want_st["n_sub_batches"] >= 40
            with from_parts(**opts) as g:
                g.set_profiling(profiling)
                for attempt in range(2):
                    with pytest.raises(LibraryError) as ei:
                        getattr(g, call)(failing, params)
                    assert ei.value.code == ELIMIT, str(ei.value)
                    what = "%s after a failed call, attempt %d, profiling %d" % (call, attempt, profiling)
                    recs, offs = getattr(g, call)(good, params)
                    assert np.array_equal(offs, want[1]), what
                    assert recs.tobytes() == want[0].tobytes(), what
                    assert _stats(g) == want_st, what


TRACE_SCRIPT = r"""
import sys, threading
import numpy as np
from mtsv_tools_b200 import MGIndex
path, reads_path, out = sys.argv[1:4]
sizes = [[int(x) for x in s.split(",")] for s in sys.argv[4:]]
z = np.load(reads_path)
cat, off = z["cat"], z["off"]
handles = [MGIndex.from_file(path, batch_reads=%d) for _ in sizes]
errors = []

def drive(t):
    try:
        for k in range(6):
            n = sizes[t][k %% 2]
            hits, offs = handles[t].bin_reads_pinned((cat[:int(off[n])], off[:n + 1].copy()))
            np.save("%%s/%%d_%%d_hits.npy" %% (out, t, k), hits.copy())
            np.save("%%s/%%d_%%d_offs.npy" %% (out, t, k), offs.copy())
    except Exception as e:
        errors.append(repr(e))

threads = [threading.Thread(target=drive, args=(t,)) for t in range(len(sizes))]
for th in threads:
    th.start()
for th in threads:
    th.join()
for h in handles:
    h.close()
assert not errors, errors
"""


def _trace_tables(stderr):
    """The slice tables of the trace: per table, the reads column of its rows in order."""
    tables, cur = [], None
    for line in stderr.splitlines():
        if line == "[mtsv_b200 trace] slice: reads, landed at ms, compute started at ms":
            cur = []
            tables.append(cur)
            continue
        m = re.fullmatch(r"\[mtsv_b200 trace\]   *(\d+): +(\d+) +-?[\d.]+ +-?[\d.]+", line)
        if m:
            assert cur is not None and int(m.group(1)) == len(cur), line
            cur.append(int(m.group(2)))
        else:
            cur = None
    return tables


def test_trace_timeline_is_per_call(small_index, small_ref, tmp_path):  # noqa: F811
    """MTSV_B200_TRACE=1 in a separate process: two handles on device 0, each driven by its own thread, alternate
    pinned calls of two sizes (2, 7 and 4, 10 slices).  The results equal those without the trace, and every call's
    table has one row per slice of that call, with the slice's reads."""
    step = 100
    sizes = [(150, 620), (350, 1000)]
    cat, off = synth.make_reads(small_ref[0], small_ref[1], 1000, 150, seed=31)
    path, reads_path = str(tmp_path / "ref.index"), str(tmp_path / "reads.npz")
    small_index.write(path)
    np.savez(reads_path, cat=cat, off=np.asarray(off, np.uint64))
    out = tmp_path / "out"
    out.mkdir()
    env = dict(os.environ, MTSV_B200_TRACE="1", PYTHONPATH=ROOT)
    r = subprocess.run([sys.executable, "-c", TRACE_SCRIPT % step, path, reads_path, str(out)] +
                       ["%d,%d" % s for s in sizes], capture_output=True, text=True, env=env, cwd=ROOT, timeout=600)
    assert r.returncode == 0, r.stderr[-4000:]
    off = np.asarray(off, np.uint64)
    with MGIndex.from_file(path, batch_reads=step) as g:
        for t, pair in enumerate(sizes):
            for k in range(6):
                n = pair[k % 2]
                hits, offs = g.bin_reads_pinned((cat[:int(off[n])], off[:n + 1].copy()))
                assert np.array_equal(np.load(out / ("%d_%d_offs.npy" % (t, k))), offs), (t, k)
                assert np.load(out / ("%d_%d_hits.npy" % (t, k))).tobytes() == hits.tobytes(), (t, k)
    want = sorted([min(step, n - i) for i in range(0, n, step)] for pair in sizes for n in pair for _ in range(3))
    assert sorted(_trace_tables(r.stderr)) == want
