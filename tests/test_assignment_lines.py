"""binner.assignment_lines (the default results format from merged (TaxID, edit) records) against results_lines on
the Hit records they were merged from.  No GPU: the records are merged on the host here."""
import numpy as np

from mtsv_tools_b200 import assignment_lines, results_lines
from mtsv_tools_b200.index import HIT_DTYPE, TAXHIT_DTYPE


def _merge(hits, off):
    recs, roff = [], [0]
    for i in range(len(off) - 1):
        best = {}
        for h in hits[int(off[i]):int(off[i + 1])]:
            t, e = int(h["tax_id"]), int(h["edit"])
            best[t] = min(e, best.get(t, e))
        recs += sorted(best.items())
        roff.append(len(recs))
    out = np.zeros(len(recs), TAXHIT_DTYPE)
    if recs:
        out["tax_id"], out["edit"] = zip(*recs)
    return out, np.array(roff, np.uint64)


def test_assignment_lines_equal_results_lines_on_random_hits():
    rng = np.random.default_rng(4)
    for trial in range(40):
        n = int(rng.integers(0, 60))
        counts = rng.integers(0, 12, size=n) * (rng.random(n) < 0.7)
        off = np.zeros(n + 1, np.uint64)
        off[1:] = np.cumsum(counts)
        hits = np.zeros(int(off[-1]), HIT_DTYPE)
        n_tax = int(rng.integers(1, 6))
        hits["tax_id"] = rng.choice([0, 1, 7, 4294967295, 123456][:n_tax], size=len(hits))
        hits["gi"] = rng.integers(0, 1 << 32, size=len(hits), dtype=np.uint64)
        hits["offset"] = rng.integers(0, 1 << 40, size=len(hits), dtype=np.uint64)
        hits["edit"] = rng.integers(0, 20, size=len(hits))
        names = ["read_%d desc" % i for i in range(n)]
        recs, roff = _merge(hits, off)
        assert assignment_lines(names, recs, roff) == results_lines(names, hits, off, long_info_output=False)
