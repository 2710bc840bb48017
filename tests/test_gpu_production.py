"""The production path (Philox draws, 16-bit wiggles) against the oracle, draw for draw (DESIGN.md §2 (c)).

Every other exact test replays recorded rows and random numbers.  Here the reference of one event is rebuilt on the CPU
from what the production path itself is documented to do:

* the trajectory rows of every charged nucleus from `Engine.trajectories(..., stride=1)`, which runs the same
  integrator (`track_kernel` with RECORD) as the production call;
* per grid row k >= 1: KE in the stable form, mean = |dKE| 1e6 / W, spread = sqrt(F mean), the Fano normal of counter
  (event_lo, event_hi, nucleus, k) (`tests/philox_model.py`), n_e = trunc(mean + spread z);
* the oracle's drift of the rows with n_e >= 1, the wiggle of counter (event_lo, event_hi, 0xFFFFFFFF, key), the
  0 <= tb + u < 512 mask and the canonical (time bucket, pad) order.

The device's float32 Box-Muller and the KE of a row (4 ulp: the device may contract into FMAs) are known within a bound,
so a row whose mean + spread z lies within that bound of an integer is "flippable": both candidate counts are drifted,
which gives every key an exact [lo, hi] charge envelope.  Keys that only a flippable 0 <-> 1 row creates are optional,
and a key such a row touches may carry another label.  Everything else must match exactly; an event without flippable
rows must be bit identical.
"""

import copy
import dataclasses
import gc

import numpy as np
import pytest

from attpc_engine_b200 import nuclear_map
from attpc_engine_b200.detector.engine import engine_for
from attpc_engine_b200.detector.pairing import unpair
from oracle import attpc_oracle as oracle
from tests import longitudinal_model as model
from tests import philox_model as pm
from tests.common import WORKLOAD_NAMES, canonical_order, cloud_keys

pytestmark = pytest.mark.gpu

VARIANTS = [(7, 0), (0x9E3779B97F4A7C15, 2**32 - 100)]  # (seed, first_event); the second crosses the event high word
VARIANT_IDS = ["seed7", "high-words"]
N_EVENTS = 256
TRACK_CHUNK = 256  # trajectories per `Engine.trajectories` call (480 KB each on the host)
KE_ULPS = 4
# share of events without a flippable row, compared bit for bit; measured 0.953 - 1.000 on a B200 (sn132dp lowest,
# 1.3e-4 of its active rows flippable)
EXACT_SHARE_FLOOR = 0.9

_WORKLOADS: dict = {}
_REFS: dict = {}


@pytest.fixture(autouse=True)
def _free_engines():
    yield
    gc.collect()


def _workload(name, n):
    import bench

    if (name, n) not in _WORKLOADS:
        _WORKLOADS[(name, n)] = bench.build_workload(name, n)
    return _WORKLOADS[(name, n)]


def _charged(zs, indices):
    return [int(i) for i in indices if zs[i] != 0]


def _nuclei_for(zs, as_, indices):
    return [nuclear_map.get_data(int(zs[i]), int(as_[i])) for i in dict.fromkeys(_charged(zs, indices))]


def _with_det(config, **changes):
    """A copy of ``config`` with detector parameters changed (and an engine cache of its own)."""
    out = copy.copy(config)
    out.__dict__.pop("_b200_engines", None)
    out.det_params = dataclasses.replace(config.det_params, **changes)
    return out


# ------------------------------------------------------------------------------------------ one trajectory's draws
def track_draws(rows, mass, cfg, seed, event, idx):
    """Rows of one trajectory that may carry electrons, with the candidate counts ``lo <= hi`` of each.

    ``lo < hi`` marks a flippable row: trunc(mean + spread z) is within the bound of the device's KE (KE_ULPS ulp per
    row) and float32 normal (`philox_model.fano_normal`) of an integer.  Rows with ``hi == 0`` are dropped.  The last
    value counts the kept rows with mean + 3 spread < 1: their electron comes from the tail of the normal."""
    det = cfg.det_params
    ev_per_w = 1.0e6 / det.w_value
    ux, uy, uz = rows[:, 3], rows[:, 4], rows[:, 5]
    g2 = ux * ux + uy * uy + uz * uz
    ke = mass * g2 / (np.sqrt(1.0 + g2) + 1.0)
    dke = np.abs(np.diff(ke))
    mean = dke * ev_per_w
    spread = np.sqrt(det.fano_factor * mean)
    # the gate mean + spread * 8.66 >= 1 is exact (tests/test_philox_model.py): rows far below it make nothing
    gate = np.flatnonzero(mean + spread * pm.NORMAL_ABS_MAX >= 0.999)
    if len(gate) == 0:
        return rows[:0], np.zeros(0, np.int64), np.zeros(0, np.int64), 0
    mean, spread = mean[gate], spread[gate]
    z, z_err = pm.fano_normal(seed, event, idx, gate + 1)
    r = mean + spread * z
    ke_err = KE_ULPS * np.spacing(ke)
    mean_err = ((ke_err[1:] + ke_err[:-1])[gate] + np.spacing(dke[gate])) * ev_per_w + np.spacing(mean)
    r_err = (mean_err * (1.0 + np.sqrt(det.fano_factor) * np.abs(z) / (2.0 * np.sqrt(mean))) + spread * z_err
             + 4.0 * np.spacing(np.abs(r)))  # fmt: skip
    lo = np.maximum(np.trunc(r - r_err), 0).astype(np.int64)
    hi = np.maximum(np.trunc(r + r_err), 0).astype(np.int64)
    keep = hi >= 1
    tail = int((mean + 3.0 * spread < 1.0)[keep].sum())
    return rows[1:][gate][keep], lo[keep], hi[keep], tail


# ------------------------------------------------------------------------------------------ one event's reference
def _drift(cfg, rows, electrons, label, cloud, d_l, counts):
    if d_l:
        model.track_to_cloud(rows, electrons, cfg, cloud, label, d_l, counts)
    else:
        oracle.track_to_cloud(rows, electrons, cfg, cloud, label)


def _alone(cfg, row, n, d_l):
    """Keys, charges and deposit counts of one row drifted on its own with n electrons."""
    cloud, counts = oracle.new_cloud(), model.new_counts()
    _drift(cfg, row[None], np.array([n], dtype=np.int64), 0, cloud, d_l, counts)
    keys, q, _ = oracle._cloud_arrays(cloud)
    return keys, q, np.array([counts.get(k, 0) for k in keys], dtype=np.int64)


def event_reference(cfg, tracks, seed, event, d_l=None):
    """Reference of one event from its tracks [(nucleus idx, rows, lo, hi)] in `indices` order.

    Returns a dict of per-key arrays in canonical order after the time-bucket mask: ``keys``, ``cloud`` ([pad, tb + u,
    charge at lo]), ``hi`` (charge at hi), ``labels``, ``optional`` (only flippable 0 <-> 1 rows make the key),
    ``free`` (the label may differ), ``slack`` (longitudinal: one electron per (sub-point, pixel) deposit), and
    ``n_flip``, the number of flippable rows."""
    cloud, counts = oracle.new_cloud(), model.new_counts()
    for idx, rows, lo, hi in tracks:
        base = lo >= 1
        if base.any():
            _drift(cfg, rows[base], lo[base], idx, cloud, d_l, counts)
    keys, q_lo, labels = oracle._cloud_arrays(cloud)
    slack = {int(k): int(counts.get(k, 0)) for k in keys} if d_l else {}
    extra, free, n_flip = {}, set(), 0
    for _, rows, lo, hi in tracks:
        for i in np.flatnonzero(hi > lo):
            n_flip += 1
            kh, qh, ch = _alone(cfg, rows[i], hi[i], d_l)
            delta = dict(zip(kh.tolist(), qh.tolist()))
            if lo[i] >= 1:
                kl, ql, _ = _alone(cfg, rows[i], lo[i], d_l)
                for k, v in zip(kl.tolist(), ql.tolist()):
                    delta[k] -= v
            else:
                free.update(kh.tolist())
            for k, v in delta.items():
                extra[k] = extra.get(k, 0) + v
            for k, c in zip(kh.tolist(), ch.tolist()):
                slack[k] = slack.get(k, 0) + c
    known = set(keys.tolist())
    opt = np.array(sorted(free - known), dtype=np.int64)
    keys = np.concatenate([keys, opt])
    q_lo = np.concatenate([q_lo, np.zeros(len(opt), np.int64)])
    labels = np.concatenate([labels, np.full(len(opt), -1, np.int64)])
    optional = np.concatenate([np.zeros(len(keys) - len(opt), bool), np.ones(len(opt), bool)])
    tb, pad = unpair(keys)
    u = pm.wiggle16(seed, event, keys.astype(np.uint64)) if len(keys) else np.zeros(0)
    t = tb + u
    m = (0 <= t) & (t < oracle.NUM_TB)
    order = np.lexsort((pad[m], tb[m]))
    keys, tb, pad, t, q_lo, labels, optional = (a[m][order] for a in (keys, tb, pad, t, q_lo, labels, optional))
    kl = keys.tolist()
    out = np.empty((len(keys), 3))
    out[:, 0], out[:, 1], out[:, 2] = pad, t, q_lo
    return dict(
        keys=keys, cloud=out, labels=labels, optional=optional,
        hi=q_lo + np.array([extra.get(k, 0) for k in kl], dtype=np.int64),
        free=np.array([k in free for k in kl], dtype=bool),
        slack=np.array([slack.get(k, 0) for k in kl], dtype=np.int64), n_flip=n_flip,
    )  # fmt: skip


def build_references(eng, cfg, momenta, vertices, zs, as_, indices, seed, first_event, events, d_l=None):
    """References of ``events`` (slots of the arrays) plus the totals the production call's statistics must meet."""
    charged = _charged(zs, indices)
    nuc = {i: nuclear_map.get_data(int(zs[i]), int(as_[i])) for i in charged}
    jobs = [(e, i) for e in events for i in charged]
    per_event = {e: [] for e in events}
    tot = dict(traj=0, active_lo=0, active_hi=0, prim_lo=0, prim_hi=0, rows=0, flip=0, tail=0)
    for a in range(0, len(jobs), TRACK_CHUNK):
        chunk = jobs[a : a + TRACK_CHUNK]
        pts, counts = eng.trajectories(
            np.array([momenta[e, i] for e, i in chunk]), np.array([vertices[e] for e, _ in chunk]),
            [nuc[i] for _, i in chunk], stride=1, max_points=10001,
        )  # fmt: skip
        for t, (e, i) in enumerate(chunk):
            n = int(counts[t])
            assert 1 <= n <= 10001
            tot["traj"] += n
            rows, lo, hi, tail = track_draws(pts[t, :n], nuc[i].mass, cfg, seed, first_event + e, i)
            per_event[e].append((i, rows.copy(), lo, hi))
            tot["active_lo"] += int((lo >= 1).sum())
            tot["active_hi"] += len(hi)
            tot["prim_lo"] += int(lo.sum())
            tot["prim_hi"] += int(hi.sum())
            tot["rows"] += len(hi)
            tot["flip"] += int((hi > lo).sum())
            tot["tail"] += tail
        del pts
    refs = {e: event_reference(cfg, per_event[e], seed, first_event + e, d_l) for e in events}
    return refs, tot


def compare_event(cloud, labels, ref, d_l=None):
    """Checks one event of the production call against its reference; returns True when it was compared bit for
    bit (no flippable row)."""
    keys = cloud_keys(cloud)
    assert np.array_equal(canonical_order(cloud), np.arange(len(cloud))), "rows are not in canonical order"
    rk = ref["keys"]
    assert np.all(np.isin(rk[~ref["optional"]], keys)), "a key of the reference is missing"
    assert np.all(np.isin(keys, rk)), "a key the reference cannot make"
    by_key = np.argsort(rk)
    p = by_key[np.searchsorted(rk, keys, sorter=by_key)]
    assert np.array_equal(cloud[:, 0], ref["cloud"][p, 0]) and np.array_equal(cloud[:, 1], ref["cloud"][p, 1]), "tb + u"
    q = cloud[:, 2].astype(np.int64)
    lo, hi, slack = ref["cloud"][p, 2].astype(np.int64), ref["hi"][p], ref["slack"][p]
    assert np.all((q >= lo - slack) & (q <= hi + slack)), "a charge outside its envelope"
    fixed = ~ref["free"][p]
    assert np.array_equal(labels[fixed], ref["labels"][p][fixed]), "labels differ"
    if ref["n_flip"] or d_l:
        return False
    assert np.array_equal(cloud, ref["cloud"]) and np.array_equal(labels, ref["labels"])
    return True


def _check_stats(stats, tot):
    assert stats["n_trajectory_points"] == tot["traj"], "the production trajectories differ from trajectories()"
    assert tot["active_lo"] <= stats["n_active_points"] <= tot["active_hi"]
    assert tot["prim_lo"] <= stats["n_primary_electrons"] <= tot["prim_hi"]


def _report(capsys, what, tot, exact=None, n=None):
    line = f"\n  {what}: flippable rows {tot['flip']} of {tot['rows']} active ({tot['flip'] / max(tot['rows'], 1):.2e})"
    if n is not None:
        line += f"; events compared bit for bit {exact} of {n} ({exact / max(n, 1):.3f})"
    with capsys.disabled():
        print(line)


def _reference(name, seed, first_event, n=N_EVENTS):
    """Cached: (workload, engine, references of all events, totals)."""
    key = (name, seed, first_event, n)
    if key not in _REFS:
        cfg, m, v, zs, as_, idx = _workload(name, n)
        eng = engine_for(cfg, _nuclei_for(zs, as_, idx))
        refs, tot = build_references(eng, cfg, m, v, zs, as_, idx, seed, first_event, range(n))
        _REFS[key] = (refs, tot)
    return _REFS[key]


# ----------------------------------------------------------------------------------------------------------- tests
@pytest.mark.parametrize("variant", VARIANTS, ids=VARIANT_IDS)
@pytest.mark.parametrize("name", WORKLOAD_NAMES)
def test_production_events_match_the_oracle(name, variant, capsys):
    seed, first = variant
    cfg, m, v, zs, as_, idx = _workload(name, N_EVENTS)
    eng = engine_for(cfg, _nuclei_for(zs, as_, idx))
    refs, tot = _reference(name, seed, first)
    batch = eng.simulate_batch(m, v, zs, as_, idx, seed=seed, first_event=first)
    _check_stats(batch.stats, tot)
    exact = sum(compare_event(*batch.event(e), refs[e]) for e in range(N_EVENTS))
    _report(capsys, f"{name} {variant}", tot, exact, N_EVENTS)
    assert exact >= EXACT_SHARE_FLOOR * N_EVENTS


def test_production_groups_and_launches(capsys):
    """Several event groups per launch and several launches: the append of rounds that hold tracks of several groups
    (longest tracks first), and the global event numbers of later launches."""
    name, n, seed = "c16dd", 6000, 424242
    cfg, m, v, zs, as_, idx = _workload(name, n)
    eng = engine_for(cfg, _nuclei_for(zs, as_, idx), max_events_per_launch=2500)
    batch = eng.simulate_batch(m, v, zs, as_, idx, seed=seed, first_event=0)
    assert batch.stats["n_track_launches"] >= 3
    # launches [0, 2048) (one group, so that the first copy starts early), [2048, 4548), [4548, 6000)
    events = sorted({0, 2047, 2048, 2499, 2500, 4095, 4096, 4547, 4548, n - 1} | set(range(0, n, 97)))
    refs, tot = build_references(eng, cfg, m, v, zs, as_, idx, seed, 0, events)
    exact = sum(compare_event(*batch.event(e), refs[e]) for e in events)
    _report(capsys, f"{name} {n} events, launches of 2500, sample", tot, exact, len(events))
    assert exact >= EXACT_SHARE_FLOOR * len(events)


def test_device_resident_production_matches(capsys):
    """host_copy=False: the second ordering tier and the device float64 sink, against the oracle."""
    name, n, seed = "c12aa", 300, 99
    cfg, m, v, zs, as_, idx = _workload(name, n)
    eng = engine_for(cfg, _nuclei_for(zs, as_, idx))
    refs, tot = _reference(name, seed, 0, n)
    dev = eng.simulate_batch(m, v, zs, as_, idx, seed=seed, host_copy=False)
    _check_stats(dev.stats, tot)
    batch = eng.read_device_result(dev)
    longest = int(np.diff(batch.offsets).max())
    exact = sum(compare_event(*batch.event(e), refs[e]) for e in range(n))
    _report(capsys, f"{name} device-resident, up to {longest} rows per event", tot, exact, n)
    assert longest > 8192, "entry lists beyond the first shared-memory tier"
    assert exact >= EXACT_SHARE_FLOOR * n


def _spyral_reference(cfg, ref, response):
    """`oracle.spyral_rows` + ADC threshold on the reference cloud, in the documented z order: tb + u descending,
    then pad ascending."""
    rows = oracle.spyral_rows(ref["cloud"], cfg.elec_params.windows_edge, cfg.elec_params.micromegas_edge,
                              cfg.det_params.length, response, cfg.pad_centers, cfg.pad_sizes)  # fmt: skip
    keep = rows[:, 3] > cfg.elec_params.adc_threshold
    rows, labels = rows[keep], ref["labels"][keep]
    order = np.lexsort((rows[:, 5], -rows[:, 6]))
    return rows[order], labels[order]


@pytest.mark.parametrize("name", ["c12aa", "sn132dp"])
def test_production_spyral_rows(name, capsys):
    seed, first = VARIANTS[0]
    cfg, m, v, zs, as_, idx = _workload(name, N_EVENTS)
    eng = engine_for(cfg, _nuclei_for(zs, as_, idx))
    refs, _ = _reference(name, seed, first)
    batch = eng.simulate_batch(m, v, zs, as_, idx, seed=seed, first_event=first, spyral_rows=True)
    response = oracle.get_response(cfg)
    compared = ties = saturated = 0
    for e in range(N_EVENTS):
        ref = refs[e]
        if ref["n_flip"]:
            continue
        rows, labels = batch.event_rows(e)
        want, want_labels = _spyral_reference(cfg, ref, response)
        assert rows.shape == want.shape, f"event {e}: rows above the threshold"
        cols = [0, 1, 2, 3, 5, 6, 7]
        assert np.array_equal(rows[:, cols], want[:, cols]), f"event {e}"
        assert np.allclose(rows[:, 4], want[:, 4], rtol=1e-12, atol=0.0), f"event {e}: integral"
        assert np.array_equal(labels, want_labels), f"event {e}: labels"
        _, n_same = np.unique(rows[:, 6], return_counts=True)
        ties += int((n_same > 1).sum())
        saturated += int((rows[:, 3] == 4095.0).sum())
        compared += 1
    with capsys.disabled():
        print(f"\n  {name}: Spyral rows of {compared} events compared exactly; time buckets with a tie in the 16-bit "
              f"wiggle: {ties}; saturated amplitudes: {saturated}")  # fmt: skip
    assert compared >= EXACT_SHARE_FLOOR * N_EVENTS
    assert ties > 0, "no wiggle tie: the tie rule was not exercised"
    if name == "sn132dp":
        assert saturated > 0


def test_production_longitudinal(capsys):
    name, n, seed, d_l = "c16dd", 128, 5, 0.277
    cfg0, m, v, zs, as_, idx = _workload(name, n)
    cfg = _with_det(cfg0, longitudinal_diffusion=d_l)
    eng = engine_for(cfg, _nuclei_for(zs, as_, idx))
    batch = eng.simulate_batch(m, v, zs, as_, idx, seed=seed)
    refs, tot = build_references(eng, cfg, m, v, zs, as_, idx, seed, 0, range(n), d_l=d_l)
    _check_stats(batch.stats, tot)
    for e in range(n):
        compare_event(*batch.event(e), refs[e], d_l=d_l)
    _report(capsys, f"{name} longitudinal {d_l} (charges within the erfc rounding bound, not bit for bit)", tot)


def test_production_draw_gate(capsys):
    """The low-yield regime.  With a W value 12000 times the workloads' most grid rows of 16C(d,d') expect about 0.25
    electrons, and a point fires only when its normal lies beyond 3 sigma: the draw gate (mean + spread * 8.66 >= 1)
    and the tail of the float32 Box-Muller decide every point."""
    name, n, seed = "c16dd", 1024, 13
    cfg0, m, v, zs, as_, idx = _workload(name, n)
    cfg = _with_det(cfg0, w_value=34.0 * 12000)
    eng = engine_for(cfg, _nuclei_for(zs, as_, idx))
    batch = eng.simulate_batch(m, v, zs, as_, idx, seed=seed)
    refs, tot = build_references(eng, cfg, m, v, zs, as_, idx, seed, 0, range(n))
    _check_stats(batch.stats, tot)
    exact = sum(compare_event(*batch.event(e), refs[e]) for e in range(n))
    _report(capsys, f"{name} W x 12000, {tot['tail']} points beyond mean + 3 spread", tot, exact, n)
    assert exact >= EXACT_SHARE_FLOOR * n
    assert tot["tail"] >= 40  # 80 of 149 active points measured on a B200
