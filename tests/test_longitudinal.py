"""Longitudinal diffusion on the host side: parameter record, engine configuration, the CPU model (no GPU needed)."""

import dataclasses
import math

import numpy as np
import pytest

from attpc_engine_b200 import _lib
from attpc_engine_b200.detector.engine import Engine, config_fingerprint
from attpc_engine_b200.detector.pairing import unpair
from attpc_engine_b200.detector.parameters import DetectorParams
from oracle import attpc_oracle as oracle
from tests import longitudinal_model as model
from tests.common import gas, make_config

EFIELD, DV = 45000.0, 1.0 / 550.0  # the tests' detector: 1 m over windows_edge - micromegas_edge = 550 time buckets


def _sigma_l(d_l, time):
    return math.sqrt(2.0 * d_l * DV * time / EFIELD) / DV


def _phi(x):
    return 0.5 * math.erfc(-x / math.sqrt(2.0))


PHI3_SUM = _phi(3.0) - _phi(-3.0)  # 0.9973: the window holds at least +-3 sigma_L


def test_positional_detector_params_default_to_off():
    det = DetectorParams(1.0, EFIELD, 3.0, 175000, gas(), 0.277, 0.2, 34.0)
    assert det.longitudinal_diffusion == 0.0
    assert dataclasses.fields(DetectorParams)[-1].name == "longitudinal_diffusion"


def test_fingerprint_follows_the_field():
    cfg = make_config()
    before = config_fingerprint(cfg, [])
    cfg.det_params.longitudinal_diffusion = 0.1
    assert config_fingerprint(cfg, []) != before


def test_ctypes_config_carries_the_field_last():
    names = [f[0] for f in _lib.AttpcConfig._fields_]
    assert names[-1] == "longitudinal_diffusion"
    cfg = _lib.AttpcConfig()
    cfg.longitudinal_diffusion = 0.277
    assert cfg.longitudinal_diffusion == 0.277


@pytest.mark.parametrize("bad", [-0.1, float("nan"), float("inf")])
def test_bad_values_are_rejected(bad):
    cfg = make_config()
    cfg.det_params.longitudinal_diffusion = bad
    with pytest.raises(ValueError, match="longitudinal_diffusion"):
        Engine(cfg, [])


@pytest.mark.parametrize("d_l", [0.1, 0.277, 1.3])
@pytest.mark.parametrize("time", [10.0, 10.37, 137.5, 285.0001, 559.99])
def test_split_matches_the_closed_form(d_l, time):
    q = 175000 * 37
    tbs, es = model.longitudinal_split(time, q, d_l, EFIELD, DV)
    sl = _sigma_l(d_l, time)
    lo, hi = math.floor(time - 3 * sl), math.floor(time + 3 * sl)
    assert tbs == list(range(max(0, lo), hi + 1))
    assert len(tbs) <= math.floor(6 * sl) + 2
    f = [_phi((k + 1 - time) / sl) - _phi((k - time) / sl) for k in tbs]
    assert es == [int(fk * q) for fk in f]
    if lo >= 0:
        assert PHI3_SUM <= sum(f) <= 1.0
        assert q * PHI3_SUM - len(tbs) <= sum(es) <= q


def test_window_clipped_at_bucket_zero():
    """A window that reaches below bucket 0 loses its negative buckets (the reference drops keys with tb < 0)."""
    time, d_l, q = 0.8, 50.0, 10**9
    sl = _sigma_l(d_l, time)
    assert math.floor(time - 3 * sl) < 0
    tbs, es = model.longitudinal_split(time, q, d_l, EFIELD, DV)
    assert tbs[0] == 0 and tbs[-1] == math.floor(time + 3 * sl)
    assert es[0] == int((_phi((1 - time) / sl) - _phi(-time / sl)) * q)


def test_window_straddles_the_last_bucket():
    """Buckets >= 512 are kept by the split (the final time-bucket mask removes them later)."""
    time, d_l = 511.6, 0.277
    tbs, es = model.longitudinal_split(time, 10**8, d_l, EFIELD, DV)
    assert tbs[0] < 511 < 512 < tbs[-1] and len(es) == len(tbs)


def test_no_spread_without_drift():
    assert model.longitudinal_split(0.0, 1000, 0.277, EFIELD, DV) == ([0], [1000])


def test_oracle_cloud_keeps_the_pad_projection():
    """One point through the oracle's drift: the same pads as without the split, charge moved between time buckets."""
    cfg = make_config(diffusion=0.277)
    track = np.array([[0.05, 0.03, 0.4, 0.0, 0.0, 0.0]] * 2)
    electrons = np.array([0, 40], dtype=np.int64)
    off, on, counts = oracle.new_cloud(), oracle.new_cloud(), model.new_counts()
    oracle.track_to_cloud(track, electrons, cfg, off, 2)
    model.track_to_cloud(track, electrons, cfg, on, 2, 0.277, counts)
    k_off, q_off, _ = oracle._cloud_arrays(off)
    k_on, q_on, _ = oracle._cloud_arrays(on)
    _, p_off = unpair(k_off)
    tb_on, p_on = unpair(k_on)
    assert set(p_on.tolist()) == set(p_off.tolist()) and len(set(tb_on.tolist())) > 1
    n_buckets, n_deposits = len(set(tb_on.tolist())), sum(counts.values())
    assert n_deposits % n_buckets == 0 and n_deposits <= 100 * n_buckets  # the same pixels in every bucket
    for pad in set(p_off.tolist()):
        assert q_on[p_on == pad].sum() <= q_off[p_off == pad].sum()
    assert q_on.sum() >= 0.997 * q_off.sum() - sum(counts.values())
