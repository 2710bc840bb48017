"""Longitudinal diffusion on the GPU (DESIGN.md §3a): the CUDA path against the CPU model of
`tests/longitudinal_model.py`, and the properties the split must keep (pad projection, work split, wire formats,
nothing changes when it is off)."""

import copy
import dataclasses
import gc
import math

import numpy as np
import pytest
from scipy.special import erfc

from attpc_engine_b200 import nuclear_map
from attpc_engine_b200.detector import simulate_batch, simulate_stream
from attpc_engine_b200.detector.engine import engine_for
from attpc_engine_b200.detector.pairing import unpair
from oracle import attpc_oracle as oracle
from tests import longitudinal_model as model
from tests.common import (
    WORKLOAD_NAMES, case_config, case_names, case_tracks, cloud_keys, digest, load_golden, load_workload, make_config,
    nuclei_of, workload_config, workload_tracks,
)  # fmt: skip

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def _free_engines():
    """Every test builds engines of its own (configs with D_L): release their device buffers when it ends."""
    yield
    gc.collect()


SPLITS = [None, dict(unit_points=40, table_spill_keys=120)]
SPLIT_IDS = ["default", "stress-split"]
D_LS = [0.1, 0.277]
MAX_DIFF_FRACTION = 1e-4  # keys whose charge may differ (CUDA's and libm's erfc differ in the last bits)


def with_dl(config, d_l):
    """A copy of ``config`` with longitudinal diffusion ``d_l`` (and its own engine cache)."""
    out = copy.copy(config)
    out.__dict__.pop("_b200_engines", None)
    out.det_params = dataclasses.replace(config.det_params, longitudinal_diffusion=d_l)
    return out


def nuclei_for(zs, as_, indices):
    return [nuclear_map.get_data(int(zs[i]), int(as_[i])) for i in dict.fromkeys(i for i in indices if zs[i] != 0)]


def oracle_event(cfg, tracks, d_l):
    """Oracle keys (canonical order), charges, labels and (sub-point, pixel) deposits per key of one replayed event."""
    cloud, counts = oracle.new_cloud(), model.new_counts()
    for t in tracks:
        electrons = np.asarray(t["electrons"], dtype=np.int64)
        model.track_to_cloud(np.asarray(t["rows"], dtype=np.float64), electrons, cfg, cloud, t["idx"], d_l, counts)
    keys, charges, labels = oracle._cloud_arrays(cloud)
    tb, pad = unpair(keys)
    order = np.lexsort((pad, tb))
    keys = keys[order]
    return keys, charges[order], labels[order], np.array([counts[k] for k in keys], dtype=np.int64)


def compare(cloud, labels, want, report):
    keys, charges, want_labels, counts = want
    assert np.array_equal(cloud_keys(cloud), keys), "keys (pad, time bucket) differ"
    assert np.array_equal(labels, want_labels), "labels differ"
    assert np.array_equal(cloud[:, 1], np.floor(cloud[:, 1])), "no wiggle was asked for"
    delta = np.abs(cloud[:, 2].astype(np.int64) - charges)
    assert np.all(delta <= counts), "a charge differs by more than one electron per (sub-point, pixel) deposit"
    report.append((int((delta != 0).sum()), len(keys)))


def check_report(report, capsys):
    diff, total = map(sum, zip(*report))
    with capsys.disabled():
        print(f"\n  keys with a different charge: {diff} of {total}")
    assert diff <= MAX_DIFF_FRACTION * total


# ------------------------------------------------------------------------------------------- 1. oracle parity
@pytest.mark.parametrize("tuning", SPLITS, ids=SPLIT_IDS)
@pytest.mark.parametrize("d_l", D_LS)
def test_golden_cases_match_the_oracle(golden_events, d_l, tuning, capsys):
    ev, report = golden_events, []
    for name in case_names():
        tracks = case_tracks(ev, name)
        if not tracks:
            continue
        cfg = with_dl(case_config(name), d_l)
        eng = engine_for(cfg, nuclei_of(tracks), **(tuning or {}))
        batch, _ = eng.simulate_replay(
            [t["rows"] for t in tracks], [t["normals"] for t in tracks], [0] * len(tracks), [t["rank"] for t in tracks],
            [t["idx"] for t in tracks], [t["za"] for t in tracks], 1, keep_all_tb=True, no_wiggle=True,
        )  # fmt: skip
        cloud, labels = batch.event(0)
        compare(cloud, labels, oracle_event(cfg, tracks, d_l), report)
    check_report(report, capsys)


@pytest.mark.parametrize("tuning", SPLITS, ids=SPLIT_IDS)
@pytest.mark.parametrize("d_l", D_LS)
@pytest.mark.parametrize("name", WORKLOAD_NAMES)
def test_workload_events_match_the_oracle(name, d_l, tuning, capsys):
    fx = load_workload(name)
    cfg = with_dl(workload_config(name), d_l)
    tracks = workload_tracks(fx)
    n_events = len(fx["digests"])
    eng = engine_for(cfg, nuclei_of(tracks), **(tuning or {}))
    batch, _ = eng.simulate_replay(
        [t["rows"] for t in tracks], [t["normals"] for t in tracks], [t["event"] for t in tracks],
        [t["rank"] for t in tracks], [t["idx"] for t in tracks], [t["za"] for t in tracks], n_events,
        keep_all_tb=True, no_wiggle=True,
    )  # fmt: skip
    report = []
    for e in range(n_events):
        cloud, labels = batch.event(e)
        compare(cloud, labels, oracle_event(cfg, [t for t in tracks if t["event"] == e], d_l), report)
    check_report(report, capsys)


# ------------------------------------------------------------------------------------ 2. one point, analytic
@pytest.mark.parametrize("z", [0.05, 0.5, 0.93])
def test_single_point_follows_the_closed_form(z):
    d_l = 0.277
    cfg = with_dl(make_config(diffusion=0.0), d_l)
    # a slow proton that stays in place: the energy step between the two rows (gamma beta 20 -> 10 MeV/c over m) makes
    # the electrons of one point
    rows = np.array([[0.05, 0.031, z, 0.0, 0.0, 20.0 / 938.272], [0.05, 0.031, z, 0.0, 0.0, 10.0 / 938.272]])
    eng = engine_for(cfg, [nuclear_map.get_data(1, 1)])
    batch, electrons = eng.simulate_replay([rows], [np.zeros(2)], [0], [0], [0], [(1, 1)], 1, keep_all_tb=True,
                                           no_wiggle=True)  # fmt: skip
    cloud, _ = batch.event(0)
    q = [int(e) * cfg.det_params.mpgd_gain for e in electrons[0] if e >= 1]
    assert q and len(np.unique(cloud[:, 0])) == 1, "diffusion = 0: one pad"
    dv = cfg.drift_velocity
    time = (cfg.det_params.length - z) / dv + cfg.elec_params.micromegas_edge
    sl = math.sqrt(2.0 * d_l * dv * time / cfg.det_params.efield) / dv
    ks = np.arange(max(0, math.floor(time - 3 * sl)), math.floor(time + 3 * sl) + 1)
    assert np.array_equal(cloud[:, 1].astype(np.int64), ks), "window bounds"
    phi = lambda x: 0.5 * erfc(-x / math.sqrt(2.0))  # noqa: E731
    f = phi((ks + 1 - time) / sl) - phi((ks - time) / sl)
    want = sum(np.trunc(f * qq) for qq in q)
    assert np.all(np.abs(cloud[:, 2] - want) <= len(q))
    w = cloud[:, 2] / cloud[:, 2].sum()
    mean = (w * (ks + 0.5)).sum()
    var = (w * (ks + 0.5 - mean) ** 2).sum()
    assert abs(mean - time) < 0.02
    assert abs(var - (sl**2 + 1.0 / 12.0)) < 0.05 * sl**2 + 0.02  # a window of +-3 sigma_L holds 97 % of the variance


# ------------------------------------------------------------------------------------ 3. pad projection
@pytest.mark.parametrize("name", WORKLOAD_NAMES)
def test_pad_projection_is_preserved(name, capsys):
    import bench

    cfg, m, v, zs, as_, idx = bench.build_workload(name, 2000)
    nuclei = nuclei_for(zs, as_, idx)
    off = engine_for(cfg, nuclei).simulate_batch(m, v, zs, as_, idx, seed=3, keep_all_tb=True)
    on_eng = engine_for(with_dl(cfg, 0.277), nuclei)
    on = on_eng.simulate_batch(m, v, zs, as_, idx, seed=3, keep_all_tb=True)
    assert on.stats["n_active_points"] == off.stats["n_active_points"]
    # events whose charge is large against their truncations: >= 1000 electrons per (sub-point, pixel) deposit of an
    # average event, so that truncating every deposit costs at most 0.1 %
    heavy = 1000.0 * on.stats["n_deposits"] / len(m)
    ratios, growth = [], []
    for e in range(len(m)):
        c_off, _ = off.event(e)
        c_on, _ = on.event(e)
        if len(c_off) == 0:
            assert len(c_on) == 0
            continue
        pads, q_off = np.unique(c_off[:, 0], return_inverse=True)
        sum_off = np.bincount(q_off, weights=c_off[:, 2])
        assert np.array_equal(np.unique(c_on[:, 0]), pads), "the same pads fire"
        sum_on = np.bincount(np.searchsorted(pads, c_on[:, 0]), weights=c_on[:, 2], minlength=len(pads))
        # every pixel keeps sum_k trunc(w trunc(f_k q)) <= trunc(w q) electrons: a pad never gains.  What it loses is
        # the <= 0.27 % outside +-3 sigma_L plus at most one electron per (sub-point, pixel) deposit (bounded key by
        # key against the oracle in test_*_match_the_oracle); the latter dominates events of a few hundred electrons.
        assert np.all(sum_on <= sum_off)
        if sum_off.sum() >= heavy:
            ratios.append(sum_on.sum() / sum_off.sum())
            growth.append(_pad_time_spread(c_on) - _pad_time_spread(c_off))
    ratios, growth = np.array(ratios), np.array(growth)
    with capsys.disabled():
        print(f"\n  {name}: {len(ratios)} events of >= {heavy:.3g} electrons: charge on / off min {ratios.min():.5f} "
              f"mean {ratios.mean():.5f}; time spread per pad grew in {(growth > 0).sum()}, by {growth.mean():.3f} "
              "buckets^2 on average")
    assert len(ratios) >= 0.8 * len(m)
    assert np.all((ratios >= 0.99) & (ratios <= 1.0)) and ratios.mean() >= 0.997
    assert growth.mean() > 0.0 and (growth > 0).mean() >= 0.85


def _pad_time_spread(c):
    """Charge-weighted mean over the pads of an event of the charge-weighted variance of the time bucket on the pad.

    (Per pad, because the spread of a whole event is dominated by the track's extent in z, against which sigma_L^2
    is lost in the quantisation of the points' drift times.)"""
    tb, q = np.floor(c[:, 1]), c[:, 2]
    pads, inv = np.unique(c[:, 0], return_inverse=True)
    w = np.bincount(inv, weights=q, minlength=len(pads))
    mu = np.bincount(inv, weights=q * tb, minlength=len(pads)) / np.maximum(w, 1e-300)
    var = np.bincount(inv, weights=q * (tb - mu[inv]) ** 2, minlength=len(pads))
    return var.sum() / max(w.sum(), 1.0)


# ------------------------------------------------------------------------------------ 4. invisible work split
def _dist_workload(name, n):
    dist = load_golden("distributions.npz")
    cfg = with_dl(make_config("He4_600" if name == "c12aa" else "D2_600"), 0.277)
    return cfg, dist[f"{name}/momenta"][:n], dist[f"{name}/vertices"][:n], dist[f"{name}/Z"], dist[f"{name}/A"], list(
        dist[f"{name}/indices"]
    )


def _same(a, b, what):
    assert np.array_equal(a.offsets, b.offsets), what
    assert np.array_equal(a.cloud, b.cloud) and np.array_equal(a.labels, b.labels), what


@pytest.mark.parametrize("name, n", [("c16dd", 96), ("c12aa", 48)])
def test_work_split_is_invisible(name, n):
    cfg, m, v, zs, as_, idx = _dist_workload(name, n)
    base = simulate_batch(m, v, zs, as_, cfg, 9, idx)
    assert base.stats["n_deposits"] > 100 * base.stats["n_active_points"], "points were split over several buckets"
    third = n // 3
    parts = [simulate_batch(m[a:b], v[a:b], zs, as_, cfg, 9, idx, first_event=a) for a, b in ((0, third), (third, n))]
    from attpc_engine_b200.detector.sharding import concat_batches

    _same(base, concat_batches(parts), "batching")
    tiny = simulate_batch(m, v, zs, as_, cfg, 9, idx, max_events_per_launch=24, hash_capacity=256)
    assert tiny.stats["n_retries"] >= 1
    _same(base, tiny, "small launches and tables")
    for tuning in (dict(unit_points=40, table_spill_keys=120), dict(unit_points=96), dict(table_spill_keys=150)):
        _same(base, simulate_batch(m, v, zs, as_, cfg, 9, idx, **tuning), tuning)
    chunks = [(m[a : a + 16], v[a : a + 16], a) for a in range(0, n, 16)]
    streamed = [b for _, b in simulate_stream(chunks, zs, as_, cfg, 9, idx, engines_per_device=2)]
    _same(base, concat_batches(streamed), "simulate_stream, two engines")


def test_sub_point_buffers_grow_on_demand():
    """A group that needs more sub-points than the first guess raises the overflow flag; the launch is redone."""
    cfg, m, v, zs, as_, idx = _dist_workload("c12aa", 48)
    big = with_dl(cfg, 2.5)  # windows of up to 36 buckets
    base = simulate_batch(m, v, zs, as_, big, 4, idx)
    # four-event groups: a first guess of 4 x 256 x 16 sub-points per group, where c12aa needs ~4 x 20000
    grown = simulate_batch(m, v, zs, as_, with_dl(cfg, 2.5), 4, idx, max_events_per_launch=4)
    assert grown.stats["n_retries"] >= 1
    _same(base, grown, "sub-point buffers grown")


# ------------------------------------------------------------------------------------ 5. outputs
@pytest.mark.parametrize("name, n", [("c16dd", 300), ("c12aa", 60)])
def test_wire_formats_with_longitudinal_diffusion(name, n):
    import bench

    cfg, m, v, zs, as_, idx = bench.build_workload(name, n)
    cfg = with_dl(cfg, 0.277)
    plain = simulate_batch(m, v, zs, as_, cfg, 31, idx)  # copies its rows to the host: tier (iii) ordering
    cols = simulate_batch(m, v, zs, as_, cfg, 31, idx, columns=True, packed=False)
    packed = simulate_batch(m, v, zs, as_, cfg, 31, idx, columns=True, max_events_per_launch=64, copy_events_per_launch=64)
    if name == "c12aa":
        assert np.diff(plain.offsets).max() > 8192, "entry lists beyond 8192 entries: global-memory ordering tier"
    for b in (cols, packed):
        assert np.array_equal(b.offsets, plain.offsets)
        assert np.array_equal(b.cloud, plain.cloud) and np.array_equal(b.labels, plain.labels)
    rows = simulate_batch(m, v, zs, as_, cfg, 31, idx, spyral_rows=True)
    rcols = simulate_batch(m, v, zs, as_, cfg, 31, idx, spyral_rows=True, row_columns=True, rows_only=True)
    assert np.array_equal(rcols.row_offsets, rows.row_offsets)
    assert np.array_equal(rcols.rows, rows.rows) and np.array_equal(rcols.row_labels, rows.row_labels)
    conv = engine_for(cfg, nuclei_for(zs, as_, idx)).convert_to_spyral(plain.offsets, plain.cloud, plain.labels)
    assert np.array_equal(conv.row_offsets, rows.row_offsets)
    assert np.array_equal(conv.rows, rows.rows) and np.array_equal(conv.row_labels, rows.row_labels)


# ------------------------------------------------------------------------------------ 6. off means off
@pytest.mark.parametrize("name", WORKLOAD_NAMES)
def test_explicit_zero_is_the_default_path(name):
    import bench

    cfg, m, v, zs, as_, idx = bench.build_workload(name, 200)
    default = simulate_batch(m, v, zs, as_, cfg, 12, idx)
    zero = simulate_batch(m, v, zs, as_, with_dl(cfg, 0.0), 12, idx)
    assert digest(default.offsets, default.cloud, default.labels) == digest(zero.offsets, zero.cloud, zero.labels)
    assert zero.stats["n_deposits"] <= 100 * zero.stats["n_active_points"]
