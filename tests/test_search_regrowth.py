"""The search's queue regrowth paths against a search that never needs them.  Needs a B200.

With the default capacities no queue overflows, so the seed stage's overflow-and-retry loop, survivors kept across a
regrowth in a later chunk and the batching of k_gap_dp / k_gap_trace never run.  The same push is searched on a fresh
context (capacities only grow) with every queue sized for one entry per read, chunks of a quarter of the reads and a
gapped batch of 7 (not a divisor of the work, so the last batch is partial): every result must be identical."""
import numpy as np
import pytest

from microbecensus_b200 import synth
from microbecensus_b200.engine import MarkerSearch

pytestmark = pytest.mark.gpu

QUEUE_MIN = 1 << 16                  # smallest capacity of the filter-pass, candidate and survivor queues


def _full_state(eng, n):
    res = eng.search(-1)
    return res.counts_vector(), eng.hits(), eng.classified(n), eng.qc_export(False)[0]


@pytest.mark.parametrize("L,n", [(150, 80_000), (100, 120_000)])
def test_forced_regrowth_equals_default_search(markers, monkeypatch, L, n):
    batch = synth.reads(11, 0, n, L)
    eng = MarkerSearch(markers, 0)
    try:
        eng.set_params(L)
        eng.push(batch)
        ref = _full_state(eng, n)
        work = eng.search_counters()
    finally:
        eng.close()
    # the forced run below must regrow every queue it shrinks
    for k in ("filter_passes", "candidates", "ungapped_hsps"):
        assert work[k] > QUEUE_MIN, (k, work)

    for k, v in (("MCX_CAND_PER_READ", 1), ("MCX_PASS_PER_READ", 1), ("MCX_SURV_PER_READ", 1), ("MCX_GAP_BATCH", 7),
                 ("MCX_CHUNK_READS", n // 4 + 1)):
        monkeypatch.setenv(k, str(v))
    eng = MarkerSearch(markers, 0)
    try:
        eng.set_params(L)
        eng.push(batch)
        got = _full_state(eng, n)
    finally:
        eng.close()
    for name, a, b in zip(("counts", "hits", "classified", "qc codes"), ref, got):
        assert a.shape == b.shape and np.array_equal(a, b), name
