"""Output regrowth for every sink: a call whose rows outgrow the first output capacity (max(n * 2048, 2^20) rows) grows
each buffer it writes, on the device and on the host, keeps the rows of the launches already copied, and returns what a
call with enough room returns."""

import numpy as np
import pytest

from attpc_engine_b200 import nuclear_map
from attpc_engine_b200.detector import simulate_batch
from attpc_engine_b200.detector.engine import engine_for
from attpc_engine_b200.detector.simulator import _nuclei_for

pytestmark = pytest.mark.gpu

N_EVENTS = 200  # c12aa: ~11 500 rows per event, ~2.3 M rows against a first capacity of 2^20
SEED = 11

CASES = {
    "float64": dict(),
    "packed_columns": dict(columns=True),
    "columns": dict(columns=True, packed=False),
    "spyral_rows": dict(spyral_rows=True),
    "spyral_row_columns": dict(spyral_rows=True, row_columns=True),
    "spyral_rows_only": dict(spyral_rows=True, rows_only=True),
}


@pytest.fixture(scope="module")
def workload():
    import bench

    cfg, m, v, zs, as_, idx = bench.build_workload("c12aa", N_EVENTS)
    # references from an engine that already holds the rows: they do not go through a regrowth themselves
    for _ in range(2):
        plain = simulate_batch(m, v, zs, as_, cfg, SEED, idx)
        spyral = simulate_batch(m, v, zs, as_, cfg, SEED, idx, spyral_rows=True)
    return cfg, m, v, zs, as_, idx, plain, spyral


def _returned(batch, kw):
    """The arrays a call with these options returns, by name."""
    got = {"offsets": batch.offsets}
    if kw.get("columns"):
        got.update(("columns." + k, a) for k, a in batch.columns.items())
    if not kw.get("rows_only"):
        got["cloud"], got["labels"] = batch.cloud, batch.labels
    if kw.get("spyral_rows"):
        got["row_offsets"], got["rows"], got["row_labels"] = batch.row_offsets, batch.rows, batch.row_labels
    if kw.get("row_columns"):
        got.update(("row_columns." + k, a) for k, a in batch.row_columns.items())
    return got


@pytest.mark.parametrize("case", list(CASES))
def test_output_regrowth_keeps_every_sink(workload, case):
    cfg, m, v, zs, as_, idx, plain, spyral = workload
    kw = CASES[case]
    # an engine of its own, so that its first call starts from the first output capacity; launches of 64 events, so
    # that the overflow lands after the rows of earlier launches are on the host, and copy chunks of 16 events
    eng = engine_for(cfg, _nuclei_for(zs, as_, idx, nuclear_map), instance=100 + list(CASES).index(case),
                     max_events_per_launch=64, copy_events_per_launch=16)  # fmt: skip
    first = eng.simulate_batch(m, v, zs, as_, idx, seed=SEED, **kw)
    second = eng.simulate_batch(m, v, zs, as_, idx, seed=SEED, **kw)
    assert first.stats["n_points"] > 1 << 20  # more rows than the first capacity: the output buffers were regrown
    assert first.stats["n_retries"] >= 1 and second.stats["n_retries"] == 0
    a, b = _returned(first, kw), _returned(second, kw)
    assert a.keys() == b.keys()
    for k in a:
        assert a[k].dtype == b[k].dtype and np.array_equal(a[k], b[k]), k
    assert np.array_equal(a["offsets"], plain.offsets)
    if "cloud" in a:
        assert np.array_equal(a["cloud"], plain.cloud) and np.array_equal(a["labels"], plain.labels)
    if kw.get("spyral_rows"):
        assert first.stats["n_rows"] == spyral.stats["n_rows"] > 0
        assert np.array_equal(a["row_offsets"], spyral.row_offsets)
        assert np.array_equal(a["rows"], spyral.rows) and np.array_equal(a["row_labels"], spyral.row_labels)
