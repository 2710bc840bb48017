"""Finalize and the Spyral passes at their size and value limits, on synthetic replay events checked against the oracle.

Every other exact test replays physics events (golden cases, workload events), which almost never land on the limits
written into `attpc_kernels.cuh`.  Here `tests/synthetic_events.py` builds events with an exact number of keys,
entries, copies, electrons, time buckets and labels, and every case compares the CUDA path with the oracle: cloud,
labels, keys and charges bit for bit; Spyral rows bit for bit except the integral (a 512-term sum in the reference,
prefix sums on the device: 1e-12).  ``stats["n_keys"]`` (occupied entries over the call) is checked against the
builder's prediction, which shows that the intended ordering tier was reached:

* ``order_kernel``: lists of up to FIN_ITEMS = 8192 entries in shared memory;
* ``order_queue_kernel<1024, 16384, 1>``: up to FIN_BIG_ITEMS = 16384, device-resident calls only;
* ``order_queue_kernel<512, 0, 2>``: 64-bit items in global scratch, the rest, and every list once hash_cap > 2^17.
"""

from contextlib import contextmanager
from functools import lru_cache

import numpy as np
import pytest

from attpc_engine_b200 import nuclear_map
from oracle import attpc_oracle as oracle
from tests.common import cloud_keys, make_config
from tests.synthetic_events import Event, build, expected_spyral, usable_pads

pytestmark = pytest.mark.gpu

DEUTERON = nuclear_map.get_data(1, 2)


@lru_cache(maxsize=None)
def _config(gain=175000, diffusion=0.0, threshold=40.0):
    cfg = make_config(diffusion=diffusion, threshold=threshold)
    cfg.det_params.mpgd_gain = gain
    return cfg


@contextmanager
def _engine(cfg, **tuning):
    from attpc_engine_b200.detector.engine import Engine

    eng = Engine(cfg, [DEUTERON], **{"max_events_per_launch": 16, **tuning})
    try:
        yield eng
    finally:
        eng.close()


def _replay(eng, b, **kw):
    batch, electrons = eng.simulate_replay(*b.replay_args(), uniforms=b.uniforms, **kw)
    for got, want in zip(electrons, b.electrons):
        assert np.array_equal(got, want)
    return batch


def _check_cloud(b, batch, events=None):
    for e in range(b.n_events) if events is None else events:
        cloud, labels = batch.event(e)
        want, want_labels = b.clouds[e]
        assert cloud.shape == want.shape, e
        assert np.array_equal(cloud_keys(cloud), cloud_keys(want)), e
        assert np.array_equal(cloud, want), e  # pad, tb + wiggle, charge
        assert np.array_equal(labels, want_labels), e


def _check_rows(cfg, rows, labels, want_cloud, want_labels, threshold=None):
    want_rows, want_row_labels = expected_spyral(cfg, want_cloud, want_labels, threshold)
    assert rows.shape == want_rows.shape
    for col in (0, 1, 2, 3, 5, 6, 7):
        assert np.array_equal(rows[:, col], want_rows[:, col]), col
    assert np.allclose(rows[:, 4], want_rows[:, 4], rtol=1e-12, atol=0.0)
    assert np.array_equal(labels, want_row_labels)


def _check_spyral(cfg, b, batch):
    for e in range(b.n_events):
        rows, labels = batch.event_rows(e)
        _check_rows(cfg, rows, labels, *b.clouds[e])


def _distinct(cfg, n, tb0=0, tb_span=509, electrons=lambda i: 1 + i % 7, rank=0, pad_from=0):
    """n points on n distinct (pad, tb) keys, spread over tb_span time buckets."""
    pads = usable_pads(cfg)
    return [(int(pads[pad_from + i // tb_span]), tb0 + i % tb_span, electrons(i), rank) for i in range(n)]


# ---------------------------------------------------------------------------------------------- 1. tier boundaries
TIER_SIZES = (0, 1, 8191, 8192, 8193, 16383, 16384, 16385)


@lru_cache(maxsize=None)
def _tier_events():
    cfg = _config()
    events = [Event(_distinct(cfg, n)) for n in TIER_SIZES]
    events.append(Event(_distinct(cfg, 300, tb0=512, tb_span=100)))  # every entry masked: queued with no rows left
    b = build(cfg, events)
    assert b.predicted_entries == [*TIER_SIZES, 300]
    return cfg, b


def test_tier_boundaries_copying_call():
    """Tiers i (order_kernel) and iii (global scratch) of a call that copies to the host, and the hash_cap regrowth of
    the 16385-entry list (seg0 + n > hash_cap)."""
    cfg, b = _tier_events()
    with _engine(cfg) as eng:
        batch = _replay(eng, b)
    assert batch.stats["n_keys"] == b.entries
    assert batch.stats["n_retries"] >= 1 and batch.stats["hash_capacity"] == 32768
    _check_cloud(b, batch)
    assert len(batch.event(len(TIER_SIZES))[0]) == 0


def test_tier_boundaries_device_resident_call():
    """Tiers i and ii (order_queue_kernel in shared memory, 8193..16384 entries) of a device-resident call."""
    cfg, b = _tier_events()
    with _engine(cfg) as eng:
        there = _replay(eng, b, host_copy=False)
        assert there.device is not None
        batch = eng.read_device_result(there)
    assert batch.stats["n_keys"] == b.entries and batch.stats["hash_capacity"] == 32768
    _check_cloud(b, batch)


def test_tier_boundaries_all_in_global_scratch():
    """hash_cap = 2^18 > 2^17: every list, even an empty one, through the 64-bit global tier."""
    cfg, b = _tier_events()
    with _engine(cfg, hash_capacity=1 << 18, max_events_per_launch=4) as eng:
        batch = _replay(eng, b)
    assert batch.stats["n_keys"] == b.entries and batch.stats["hash_capacity"] == 1 << 18
    _check_cloud(b, batch)


@pytest.mark.parametrize("n, regrows", [(8192, False), (8193, True)])
def test_hash_capacity_at_the_exact_entry_count(n, regrows):
    """An event whose entries exactly fill hash_capacity fits; one entry more regrows the regions and redoes the call."""
    cfg = _config()
    b = build(cfg, [Event(_distinct(cfg, 5)), Event(_distinct(cfg, n, electrons=lambda i: 1 + i % 3))])
    with _engine(cfg, hash_capacity=8192) as eng:
        batch = _replay(eng, b)
    assert batch.stats["n_keys"] == b.entries == n + 5
    assert batch.stats["hash_capacity"] == (16384 if regrows else 8192)
    assert (batch.stats["n_retries"] >= 1) == regrows
    _check_cloud(b, batch)


# --------------------------------------------------------------------------------------------------- 2. copies
def test_copies_of_one_key():
    """unit_points=1: every point is a work unit, so a key hit by k points is listed k times and merged in step 5 of
    order_event.  9000 copies put one key across the 8192 boundary; that group has > 8192 units (MAX_UNITS_SORT), so
    point_scan_kernel takes its unsorted branch.  The copies come from several ranks with non-ascending labels."""
    cfg = _config()
    pads = usable_pads(cfg)
    events = []
    for k in (1, 2, 32, 33, 9000):
        pts = _distinct(cfg, 40, pad_from=100)
        pts += [(int(pads[7]), 123, 1 + i % 5, (i * 7) % 4) for i in range(k)]  # one key, ranks 0..3 interleaved
        events.append(Event(pts, indices=[6, 2, 9, 4]))
    b = build(cfg, events, unit_points=1)
    assert b.predicted_entries == [40 + k for k in (1, 2, 32, 33, 9000)]
    with _engine(cfg, unit_points=1) as eng:
        batch = _replay(eng, b, spyral_rows=True)
    assert batch.stats["n_keys"] == b.entries
    _check_cloud(b, batch)
    _check_spyral(cfg, b, batch)


# --------------------------------------------------------------------------------------------------- 3. labels
SPLITS = [None, dict(unit_points=1), dict(unit_points=40, table_spill_keys=120)]
SPLIT_IDS = ["default", "unit-per-point", "stress-split"]


@pytest.mark.parametrize("tuning", SPLITS, ids=SPLIT_IDS)
def test_highest_rank_labels_a_key(tuning):
    """The label of a key is the index of the highest rank that touched it (transporter.py:166-169, 247-249), not the
    highest index: 16 charged tracks (ranks 0..15, the top 4 bits of the table word), indices in no order, neutral
    ranks in between, and keys shared by several ranks."""
    cfg = _config()
    pads = usable_pads(cfg)
    rng = np.random.default_rng(5)
    shared = [(int(pads[200 + j]), 40 + j) for j in range(24)]

    def event(indices, neutral):
        pts = []
        for r in range(len(indices)):
            if r in neutral:
                continue
            pts += _distinct(cfg, 30, tb0=100 + 10 * r, tb_span=10, rank=r, pad_from=300 + 3 * r)
            for j in rng.choice(len(shared), size=8, replace=False):  # several ranks on one key
                pts.append((*shared[j], 1 + r, r))
        rng.shuffle(pts)
        return Event([tuple(int(v) for v in p) for p in pts], indices=indices, neutral=frozenset(neutral))

    events = [
        event([int(v) for v in rng.permutation(16) * 3 + 1], ()),  # 16 charged tracks
        event([30, 2, 17, 5, 11, 0, 8, 25, 1, 9], (1, 4, 8)),  # neutral ranks in between
        event([3, 1], ()),
    ]
    b = build(cfg, events, unit_points=(tuning or {}).get("unit_points"))
    with _engine(cfg, **(tuning or {})) as eng:
        batch = _replay(eng, b)
    if tuning is None or tuning.get("unit_points") == 1:
        assert batch.stats["n_keys"] == b.entries
    _check_cloud(b, batch)
    labels_of_rank = [set(ev.indices) for ev in events]
    for e in range(len(events)):
        assert set(batch.event(e)[1]) <= labels_of_rank[e]


def test_zero_charge_deposit_relabels_keys():
    """diffusion > 0, mpgd_gain = 1: a later track's one-electron point spreads integer shares of 0 over the mesh;
    they relabel the keys the earlier track made and create keys of zero charge (transporter.py:166-169, 247-249)."""
    cfg = _config(gain=1, diffusion=0.277, threshold=-1.0)
    pads = usable_pads(cfg)
    p = int(pads[len(pads) // 2])
    c = np.asarray(cfg.pad_centers)[pads]
    d = np.hypot(*(c - cfg.pad_centers[p]).T)
    q = int(pads[np.argsort(d)[1]])  # the nearest other pad: the two meshes overlap in part
    events = [Event([(p, 200, 2_000_000, 0), (q, 200, 1, 1)], indices=[4, 1]),
              Event([(q, 200, 1, 0), (p, 200, 2_000_000, 1)], indices=[4, 1])]  # fmt: skip
    b = build(cfg, events)
    keys, charges, labels = b.records[0]
    assert ((charges == 0) & (labels == 1)).any() and ((charges > 0) & (labels == 1)).any()
    with _engine(cfg) as eng:
        batch = _replay(eng, b, spyral_rows=True)
    _check_cloud(b, batch)
    _check_spyral(cfg, b, batch)


# -------------------------------------------------------------------------------------------------- 4. charges
SMEM_SLOTS = 4864  # attpc_kernels.cuh


def _smem_home(pad, tb):
    key1 = ((tb << 15) | pad) + 1
    return ((key1 * 2654435761) & 0xFFFFFFFF) * SMEM_SLOTS >> 32


def _hi2_pair(cfg, tb):
    """Two keys in time bucket tb whose home slots 2k, 2k + 1 share one 32-bit hi2 word of the deposit table."""
    seen = {}
    for pad in usable_pads(cfg)[:2000]:
        h = _smem_home(int(pad), tb)
        if h ^ 1 in seen:
            return sorted([(seen[h ^ 1], tb), (int(pad), tb)], key=lambda k: _smem_home(k[0], k[1]))
        seen[h] = int(pad)
    raise AssertionError("no pair")


@pytest.mark.parametrize("unit_points", [None, 1], ids=["one-segment", "copies"])
def test_charges_beyond_32_bits(unit_points):
    """Sums that cross 2^32 several times, in one segment (carry into the 16-bit high part, two keys sharing a hi2
    word) and across copies (64-bit sum in order_event); sums of exactly 2^32 - 1 and 2^32, where the carry test
    `> ~vlo` decides."""
    pads = usable_pads(_config())
    a, b_ = _hi2_pair(_config(), 77)
    cases = []
    cfg = _config(gain=(1 << 31) + 12345)
    pts = [(*a, 3, 0)] * 5 + [(*b_, 2, 0)] * 7 + [(int(pads[50]), 90, 1, 0)] * 3
    cases.append((cfg, [Event(pts)]))
    for gain, split in ((65537, (30000, 35535)), (65536, (30000, 35536))):  # 65535 * 65537 = 2^32 - 1; 2^32
        cfg = _config(gain=gain)
        pts = [(int(pads[60]), 10, split[0], 0), (int(pads[60]), 10, split[1], 0), (int(pads[61]), 10, 65535, 0)]
        cases.append((cfg, [Event(pts)]))
    sums = []
    for cfg, events in cases:
        b = build(cfg, events, unit_points=unit_points)
        with _engine(cfg, **({"unit_points": 1} if unit_points else {})) as eng:
            batch = _replay(eng, b)
        assert batch.stats["n_keys"] == b.entries
        _check_cloud(b, batch)
        sums += list(b.clouds[0][0][:, 2])
    assert (1 << 32) - 1 in sums and 1 << 32 in sums and max(sums) > 7 * (1 << 32)


def test_charge_of_2_to_the_48():
    """2^48 - 1 electrons on a key are fine; 2^48 raise the capacity error, whether one segment reaches it or only the
    sum of copies in order_event does (the flag keeps the high bits out of the pad field of the staged row); the
    engine gives correct results on the next call."""
    gain = (1 << 24) + 1  # (2^24 - 1)(2^24 + 1) = 2^48 - 1
    cfg = _config(gain=gain)
    pads = usable_pads(cfg)
    key = (int(pads[33]), 250)
    fine = build(cfg, [Event([(*key, (1 << 23) - 1, 0), (*key, 1 << 23, 0)]), Event(_distinct(cfg, 20))])
    assert fine.clouds[0][0][0, 2] == (1 << 48) - 1
    over = build(cfg, [Event([(*key, 1 << 23, 0), (*key, 1 << 23, 0)]), Event(_distinct(cfg, 20))])
    assert over.records[0][1][0] >= 1 << 48
    for unit_points in (None, 1):
        with _engine(cfg, **({"unit_points": 1} if unit_points else {})) as eng:
            with pytest.raises(RuntimeError, match="2\\^48"):
                _replay(eng, over)
            batch = _replay(eng, fine)
            _check_cloud(fine, batch)


# ---------------------------------------------------------------------------------------------- 5. time buckets
def test_last_time_bucket_mask_reads_the_wiggle():
    """tb = 511 is kept only while 511 + u < 512: u = 1 - 2^-53 rounds up to 512.0 (masked), u = 1 - 2^-44 does not;
    tb = 0 with u = 0 is kept, tb = 512 is not."""
    from attpc_engine_b200.detector.pairing import pair

    cfg = _config()
    pads = usable_pads(cfg)
    pts = [(int(pads[10]), 511, 3, 0), (int(pads[11]), 511, 3, 0), (int(pads[12]), 0, 3, 0), (int(pads[13]), 512, 3, 0),
           (int(pads[14]), 511, 3, 0)]  # fmt: skip
    u = {int(pair(511, pts[0][0])): 1.0 - 2.0**-53, int(pair(511, pts[1][0])): 1.0 - 2.0**-44,
         int(pair(0, pts[2][0])): 0.0, int(pair(511, pts[4][0])): 0.5}  # fmt: skip
    b = build(cfg, [Event(pts)], uniforms=[u])
    want = b.clouds[0][0]
    assert len(want) == 3 and pts[0][0] not in want[:, 0] and pts[3][0] not in want[:, 0]
    with _engine(cfg) as eng:
        for spyral in (False, True):
            batch = _replay(eng, b, spyral_rows=spyral)
            assert batch.stats["n_keys"] == 5
            _check_cloud(b, batch)
            if spyral:
                _check_spyral(cfg, b, batch)


@pytest.mark.parametrize("spyral", [False, True], ids=["cloud", "spyral"])
def test_keep_all_time_buckets_share_the_last_bin(spyral):
    """keep_all_tb: buckets >= 1023 share the last counting-sort bin, where step 4 compares whole keys; buckets 8191
    (kept) and 8192 (beyond the 13-bit time bucket of the table key: dropped, a documented deviation)."""
    cfg = _config()
    pads = usable_pads(cfg)
    pts = []
    for j, tb in enumerate((1022, 1023, 1024, 1500, 1023, 1500, 1024, 8191)):
        for i in range(12):
            pts.append((int(pads[(5000 - 397 * j + 31 * i) % len(pads)]), tb, 2 + i, i % 2))
    pts.append((int(pads[77]), 8192, 9, 0))
    b = build(cfg, [Event(pts, indices=[3, 8]), Event(_distinct(cfg, 50, tb0=1020, tb_span=25))], keep_all_tb=True)
    cloud, labels = b.clouds[0]
    beyond = np.floor(cloud[:, 1]) >= 8192
    assert beyond.sum() == 1  # the oracle keeps it
    b.clouds[0] = (cloud[~beyond], labels[~beyond])
    with _engine(cfg) as eng:
        batch = _replay(eng, b, keep_all_tb=True, spyral_rows=spyral)
    assert batch.stats["n_keys"] == b.entries == len(pts) - 1 + 50
    _check_cloud(b, batch)
    if spyral:
        _check_spyral(cfg, b, batch)


def test_windows_edge_beyond_8191_is_rejected():
    from attpc_engine_b200.detector.engine import Engine

    for edge, ok in ((8191, True), (8192, False)):
        cfg = make_config()
        cfg.elec_params.windows_edge = edge
        cfg.calculate_drift_velocity()
        if ok:
            Engine(cfg, [DEUTERON]).close()
        else:
            with pytest.raises(ValueError, match="windows_edge"):
                Engine(cfg, [DEUTERON])


# ---------------------------------------------------------------------------------- 6. stand-alone Spyral pass
def _converter(cfg, threshold=None):
    from attpc_engine_b200.detector.engine import Engine

    el = cfg.elec_params
    return Engine.for_conversion(el.windows_edge, el.micromegas_edge, cfg.det_params.length, oracle.get_response(cfg),
                                 cfg.pad_centers, cfg.pad_sizes, el.adc_threshold if threshold is None else threshold)  # fmt: skip


def _e_keep(cfg):
    """Smallest electron count whose amplitude exceeds the threshold."""
    r = oracle.get_response(cfg).max()
    e = int(cfg.elec_params.adc_threshold / r)
    while not min(r * e, 4095.0) > cfg.elec_params.adc_threshold:
        e += 1
    return e


def test_convert_to_spyral_at_its_limits():
    """Events of 4095, 4096 (shared memory) and 4097 (global scratch) kept rows, 5000 rows of one time bucket with
    tied z, empty events and an event whose rows are all below threshold, > 1024 events (several scan tiles)."""
    cfg = _config()
    pads = usable_pads(cfg)
    keep = _e_keep(cfg)
    rng = np.random.default_rng(11)

    def rows(n_kept, n_low, tbf=None):
        n = n_kept + n_low
        c = np.empty((n, 3))
        c[:, 0] = rng.choice(pads, n)
        c[:, 1] = tbf if tbf is not None else rng.integers(0, 512, n) + rng.integers(0, 65536, n) / 65536.0
        c[:, 2] = np.concatenate([rng.integers(keep, 200 * keep, n_kept), rng.integers(0, keep, n_low)])
        return c[rng.permutation(n)]

    clouds = [rows(4095, 300), rows(0, 0), rows(4096, 10), rows(4097, 0), rows(0, 500), rows(5000, 30, tbf=200.25)]
    clouds += [rows(int(rng.integers(0, 6)), int(rng.integers(0, 3))) for _ in range(1100)]
    clouds.append(rows(4097, 1))
    offsets = np.concatenate([[0], np.cumsum([len(c) for c in clouds])])
    cloud = np.concatenate(clouds)
    labels = rng.integers(0, 9, len(cloud))
    eng = _converter(cfg)
    try:
        got = eng.convert_to_spyral(offsets, cloud, labels)
        every = eng.convert_to_spyral(offsets, cloud, labels, keep_all=True)
    finally:
        eng.close()
    kept = np.diff(got.row_offsets)
    assert list(kept[:6]) == [4095, 0, 4096, 4097, 0, 5000] and kept[-1] == 4097
    for e in range(len(clouds)):
        a, b = offsets[e], offsets[e + 1]
        r, lab = got.event_rows(e)
        _check_rows(cfg, r, lab, cloud[a:b], labels[a:b])
    want = oracle.spyral_rows(cloud, cfg.elec_params.windows_edge, cfg.elec_params.micromegas_edge,
                              cfg.det_params.length, oracle.get_response(cfg), cfg.pad_centers, cfg.pad_sizes)  # fmt: skip
    for col in (0, 1, 2, 3, 5, 6, 7):
        assert np.array_equal(every.rows[:, col], want[:, col]), col
    assert np.allclose(every.rows[:, 4], want[:, 4], rtol=1e-12, atol=0.0)
    assert np.array_equal(every.row_labels, labels)


# ------------------------------------------------------------------------------------------------ 7. ADC threshold
def _clip_counts(cfg):
    """Electron counts at the 4095 clip and at the boundary of the clipped prefix k for several r_i."""
    rs = np.sort(oracle.get_response(cfg))[::-1]
    out = []
    for i in (0, 1, 3, 10, 40):
        if rs[i] < rs[0] / 16:  # (keeps the counts within a replayable kinetic energy)
            continue
        e = int(4095.0 / rs[i])
        out += [e - 1, e, e + 1]
    return out


@pytest.mark.parametrize("q_at", [0, 1])
def test_adc_threshold_of_the_standalone_pass(q_at):
    """mpgd_gain = 1 replay (the Spyral rows of a replay come from the stand-alone pass over the float64 cloud): the
    threshold is fl(r_max q) for a q of the event, so q and q - 1 electrons are dropped and q + 1 kept; plus the clip."""
    r = oracle.get_response(_config()).max()
    q = (1_300_000, 2_000_003)[q_at]
    cfg = _config(gain=1, threshold=float(r * q))
    pads = usable_pads(cfg)
    counts = [q - 1, q, q + 1, q + 2] + _clip_counts(cfg)
    pts = [(int(pads[400 + i]), 30 + 7 * i, e, 0) for i, e in enumerate(counts)]
    b = build(cfg, [Event(pts)])
    with _engine(cfg) as eng:
        batch = _replay(eng, b, spyral_rows=True)
    _check_cloud(b, batch)
    _check_spyral(cfg, b, batch)
    rows = batch.event_rows(0)[0]
    assert len(rows) == len(counts) - 2 and (rows[:, 3] == 4095.0).sum() >= 5


@lru_cache(maxsize=None)
def _production():
    """200 16C(d,d') events, their species and the electron counts of their cloud (which no threshold changes)."""
    import bench
    from attpc_engine_b200.detector.engine import Engine
    from attpc_engine_b200.detector.simulator import _nuclei_for

    cfg, m, v, zs, as_, idx = bench.build_workload("c16dd", 200)
    species = _nuclei_for(zs, as_, idx, nuclear_map)
    eng = Engine(cfg, species)
    try:
        electrons = eng.simulate_batch(m, v, zs, as_, idx, seed=3).cloud[:, 2].copy()
    finally:
        eng.close()
    return cfg, (m, v, zs, as_, idx), species, electrons


FUSED_PICKS = ["q10", "q50", "q90", "qmax", "q50-1", "minus1", "zero", "below4095", "4095"]


@pytest.mark.parametrize("pick", FUSED_PICKS)
def test_adc_threshold_of_the_fused_path(pick):
    """A production call with Spyral rows keeps a row when its charge >= e_keep_min (init_sim); the stand-alone pass
    when min(r_max e, 4095) > threshold.  With thresholds fl(r_max q) for charges q of the call's own cloud, plus -1, 0,
    4095 - 2^-40 and 4095, the fused rows equal convert_to_spyral of the call's float64 cloud bit for bit, every row of
    charge <= q is dropped and every row above q kept.  Two thresholds also go through the typed row columns."""
    from attpc_engine_b200.detector.engine import Engine

    cfg, args, species, electrons = _production()
    r = oracle.get_response(cfg).max()
    below_clip = np.unique(electrons[(electrons > 0) & (electrons * r < 4000.0)])
    quantile = {"q10": 0.1, "q50": 0.5, "q90": 0.9, "qmax": 1.0, "q50-1": 0.5}
    q = None
    if pick in quantile:
        q = float(np.quantile(below_clip, quantile[pick], method="nearest")) - (pick == "q50-1")
        threshold = float(r * q)  # amplitude of q electrons: q is dropped, q + 1 kept
    else:
        threshold = {"minus1": -1.0, "zero": 0.0, "below4095": 4095.0 - 2.0**-40, "4095": 4095.0}[pick]
    saved = cfg.elec_params.adc_threshold
    cfg.elec_params.adc_threshold = threshold
    try:
        eng = Engine(cfg, species)
    finally:
        cfg.elec_params.adc_threshold = saved
    try:
        batch = eng.simulate_batch(*args, seed=3, spyral_rows=True)
        ref = eng.convert_to_spyral(batch.offsets, batch.cloud, batch.labels)
        cols = None
        if pick in ("q50", "below4095"):
            cols = eng.simulate_batch(*args, seed=3, spyral_rows=True, row_columns=True, rows_only=True)
    finally:
        eng.close()
    ce = batch.cloud[:, 2]
    assert np.array_equal(ce, electrons)
    assert np.array_equal(batch.row_offsets, ref.row_offsets)
    assert np.array_equal(batch.rows, ref.rows) and np.array_equal(batch.row_labels, ref.row_labels)
    event_of_row = np.repeat(np.arange(len(batch.offsets) - 1), np.diff(batch.offsets))
    amp = np.minimum(r * ce, 4095.0)
    per_event = np.bincount(event_of_row, weights=amp > threshold, minlength=len(batch.offsets) - 1)
    assert np.array_equal(np.diff(batch.row_offsets), per_event.astype(np.int64))
    if q is not None:
        assert (ce == q + 1).any() if pick == "q50-1" else (ce == q).any()
        assert len(batch.rows) == (ce > q).sum() > 0
    elif pick == "minus1":
        assert len(batch.rows) == len(ce)
    elif pick == "zero":
        assert len(batch.rows) == (ce > 0).sum()
    elif pick == "below4095":
        assert len(batch.rows) > 0 and (batch.rows[:, 3] > threshold).all()
    else:
        assert len(batch.rows) == 0
    if cols is not None:
        assert np.array_equal(cols.row_offsets, batch.row_offsets)
        assert np.array_equal(cols.rows, batch.rows) and np.array_equal(cols.row_labels, batch.row_labels)
