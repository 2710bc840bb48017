"""CPU tests of the synthetic event builder (`tests/synthetic_events.py`): a failing test of
`test_gpu_finalize_edges.py` then points at the library, not at the builder."""

import numpy as np
import pytest

from attpc_engine_b200 import nuclear_map
from attpc_engine_b200.detector.engine import build_pad_lut
from attpc_engine_b200.detector.pairing import unpair
from oracle import attpc_oracle as oracle
from tests.common import make_config
from tests.synthetic_events import Event, build, position, track_rows, usable_pads


@pytest.fixture(scope="module")
def cfg():
    return make_config(diffusion=0.0)


def test_four_row_deuteron_track(cfg):
    """A leading row and three points give electrons [0, 5, 70000, 12] and exactly the keys (tb, pad) = (0, 100),
    (300, 2000), (511, 5000)."""
    b = build(cfg, [Event([(100, 0, 5, 0), (2000, 300, 70000, 0), (5000, 511, 12, 0)])])
    assert np.array_equal(b.electrons[0], [0, 5, 70000, 12])
    keys, charges, labels = b.records[0]
    tb, pad = unpair(keys)
    assert list(zip(tb, pad)) == [(0, 100), (300, 2000), (511, 5000)]
    assert np.array_equal(charges, np.array([5, 70000, 12]) * cfg.det_params.mpgd_gain)
    assert b.predicted_entries == [3]


@pytest.mark.parametrize("e", [1, 2, 7, 1000, 65535, 2**23, 2**24 - 1, 1_300_000, 470_000_000])
def test_electrons_are_exact(cfg, e):
    mass = float(nuclear_map.get_data(1, 2).mass)
    rows = track_rows(cfg, [(10, 5, e), (11, 5, 1), (12, 6, e)], mass)
    got = oracle.fano_electrons(rows, mass, cfg.det_params.w_value, cfg.det_params.fano_factor, normals=np.zeros(4))
    assert np.array_equal(got, [0, e, 1, e])


def test_pad_round_trip(cfg):
    """Every usable pad centre maps back to its pad, in the oracle and in the CUDA path's 1 mm lookup table; beam
    pads and pads whose centre falls on another pad are left out."""
    pads = usable_pads(cfg)
    assert 9000 < len(pads) < len(cfg.pad_centers)
    assert not np.isin(pads, oracle.BEAM_PAD_IDS).any()
    lut, origin = build_pad_lut(cfg.pad_grid, cfg.pad_grid_edges)
    for pad in pads[::7]:
        x, y, _ = position(cfg, int(pad), 0)
        ix, iy = oracle._grid_index(cfg.pad_grid_edges, x, y)
        assert cfg.pad_grid[ix, iy] == pad
        assert lut[int(np.floor(x * 1000.0)) - origin, int(np.floor(y * 1000.0)) - origin] == pad


@pytest.mark.parametrize("tb", [0, 1, 300, 511, 512, 1022, 1023, 1024, 1500, 8191, 8192])
def test_time_bucket_round_trip(cfg, tb):
    """z = length - (tb + 0.5 - micromegas_edge) dv drifts to time bucket tb (`solver.py:386-413`)."""
    _, _, z = position(cfg, 100, tb)
    t = (cfg.det_params.length - z) / cfg.drift_velocity + cfg.elec_params.micromegas_edge
    assert int(t) == tb and abs(t - tb - 0.5) < 1e-6


def test_predicted_entries(cfg):
    pads = usable_pads(cfg)
    copies = [(int(pads[3]), 40, 2, r % 2) for r in range(9)]
    distinct = [(int(pads[i]), 7, 1, 0) for i in range(20)]
    ev = Event(copies + distinct + [(int(pads[5]), 8192, 3, 0)], indices=[2, 0])
    assert build(cfg, [ev], unit_points=1).predicted_entries == [29]  # one entry per active point below 8192
    assert build(cfg, [ev]).predicted_entries == [21]  # one unit: one entry per key
    big = Event([(int(pads[i % 100]), i // 100, 1, 0) for i in range(2000)] + copies, indices=[2, 0])
    assert build(cfg, [big]).predicted_entries == [None]  # copies over several units of 1024 points
    zero = Event([(int(pads[0]), 3, 0, 0), (int(pads[1]), 3, 4, 0)])
    assert build(cfg, [zero]).predicted_entries == [1]  # no electrons, no point
