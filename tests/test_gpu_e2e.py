"""GPU tests of the public surface: simulate / simulate_batch / run_simulation / writers, sharding invariance,
Spyral conversion against the oracle, and the statistical half of parity part (b) (KS tests against distribution
samples of the unmodified reference, tests/golden/make_distributions.py)."""

import sys
import types

import numpy as np
import pytest
from scipy.stats import ks_2samp

from attpc_engine_b200 import nuclear_map
from attpc_engine_b200.detector import ArrayWriter, SpyralWriter, convert_to_spyral, run_simulation, simulate, simulate_batch
from attpc_engine_b200.detector.sharding import concat_batches, shard_range
from oracle import attpc_oracle as oracle
from tests.common import case_config, load_golden, make_config

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dist():
    return load_golden("distributions.npz")


def _workload(dist, name, n=None):
    cfg = make_config("He4_600" if name == "c12aa" else "D2_600")
    m, v = dist[f"{name}/momenta"], dist[f"{name}/vertices"]
    n = len(m) if n is None else n
    return cfg, m[:n], v[:n], dist[f"{name}/Z"], dist[f"{name}/A"], list(dist[f"{name}/indices"])


def test_simulate_reference_signature(golden_events):
    """`simulate(momenta, vertex, Z, A, config, rng, indices)` -> (cloud [N,3], labels [N]) like the reference."""
    ev, name = golden_events, "dd_exit"
    cfg = case_config(name)
    event = simulate(ev[f"{name}/momenta"], ev[f"{name}/vertex"], ev[f"{name}/Z"], ev[f"{name}/A"], cfg,
                     np.random.default_rng(3), list(ev[f"{name}/indices"]))  # fmt: skip
    assert len(event) == 2
    cloud, labels = event
    assert cloud.ndim == 2 and cloud.shape[1] == 3 and labels.shape == (len(cloud),) and labels.dtype == np.int64
    assert len(cloud) > 500 and set(np.unique(labels)) <= {2, 3}
    assert np.all((cloud[:, 1] >= 0) & (cloud[:, 1] < 512)) and np.all(cloud[:, 0] == np.floor(cloud[:, 0]))
    assert np.all(cloud[:, 2] % 1 == 0)


def test_reference_smoke_case_outside_detector():
    """The reference's own detector test (tests/test_detector.py:44-63): protons far outside -> empty 2-tuple."""
    cfg = make_config(bfield=2.85)
    fake = np.array([[0.0, 0.0, 10.0, 938.0]] * 4)
    event = simulate(fake, np.array([1.0, 1.0, 1.0]), np.array([1, 1, 1, 1]), np.array([1, 1, 1, 1]), cfg,
                     np.random.default_rng(), [0])  # fmt: skip
    assert len(event) == 2 and len(event[0]) == 0 and len(event[1]) == 0


def test_results_do_not_depend_on_batching(dist):
    """Counter-based streams: splitting a batch (as the multi-GPU shards do) reproduces it bit for bit."""
    cfg, m, v, zs, as_, idx = _workload(dist, "c16dd", 96)
    whole = simulate_batch(m, v, zs, as_, cfg, 77, idx, first_event=1000)
    parts = []
    for rank in range(3):
        a, b = shard_range(len(m), rank, 3)
        parts.append(simulate_batch(m[a:b], v[a:b], zs, as_, cfg, 77, idx, first_event=1000 + a))
    merged = concat_batches(parts)
    assert np.array_equal(whole.offsets, merged.offsets)
    assert np.array_equal(whole.cloud, merged.cloud) and np.array_equal(whole.labels, merged.labels)
    other_seed = simulate_batch(m, v, zs, as_, cfg, 78, idx, first_event=1000)
    assert not np.array_equal(whole.cloud[:, 1], other_seed.cloud[: len(whole.cloud), 1])


def test_small_launches_and_small_tables_give_identical_results(dist):
    """Capacity retries (hash tables, point buffers) and launch splitting are invisible in the output."""
    cfg, m, v, zs, as_, idx = _workload(dist, "c16dd", 64)
    base = simulate_batch(m, v, zs, as_, cfg, 5, idx)
    tiny = simulate_batch(m, v, zs, as_, cfg, 5, idx, max_events_per_launch=24, hash_capacity=256)
    assert tiny.stats["n_retries"] >= 1
    assert np.array_equal(base.offsets, tiny.offsets) and np.array_equal(base.cloud, tiny.cloud)
    assert np.array_equal(base.labels, tiny.labels)


@pytest.mark.parametrize("name, n", [("c16dd", 96), ("c12aa", 48), ("sn132dp", 48)])
def test_work_splitting_is_invisible(dist, name, n):
    """Events split over many deposit CTAs (tiny work units) and tables appended to the entry list in many segments
    (tiny spill threshold) give the same rows, charges and labels: copies of a key are merged after sorting."""
    if name in ("c16dd", "c12aa"):
        cfg, m, v, zs, as_, idx = _workload(dist, name, n)
    else:
        import bench

        cfg, m, v, zs, as_, idx = bench.build_workload(name, n)
    base = simulate_batch(m, v, zs, as_, cfg, 9, idx)
    for tuning in (dict(unit_points=48), dict(table_spill_keys=150), dict(unit_points=96, table_spill_keys=400)):
        split = simulate_batch(m, v, zs, as_, cfg, 9, idx, **tuning)
        assert np.array_equal(base.offsets, split.offsets), tuning
        assert np.array_equal(base.cloud, split.cloud) and np.array_equal(base.labels, split.labels), tuning
    assert split.stats["n_table_flushes"] > n  # the stress really went through the segment path


def test_many_species_share_the_track_kernels_shared_memory(dist):
    """An engine built for eight species keeps their stopping-power tables in shared memory with fewer warps per track
    CTA; the tracks of a two-species workload come out exactly as from the two-species engine."""
    from attpc_engine_b200.detector.engine import engine_for

    cfg, m, v, zs, as_, idx = _workload(dist, "c16dd", 300)
    base = simulate_batch(m, v, zs, as_, cfg, 21, idx)
    many = [nuclear_map.get_data(z, a) for z, a in ((1, 1), (1, 2), (1, 3), (2, 3), (2, 4), (6, 12), (6, 14), (6, 16))]
    wide = engine_for(cfg, many).simulate_batch(m, v, zs, as_, idx, seed=21)
    assert np.array_equal(base.offsets, wide.offsets)
    assert np.array_equal(base.cloud, wide.cloud) and np.array_equal(base.labels, wide.labels)


def test_convert_to_spyral_function_matches_oracle(golden_events):
    ev, name = golden_events, "alpha_breakup"
    cfg = case_config(name)
    cloud = ev[f"{name}/cloud"]
    resp = oracle.get_response(cfg)
    got = convert_to_spyral(cloud, cfg.elec_params.windows_edge, cfg.elec_params.micromegas_edge, cfg.det_params.length,
                            resp, cfg.pad_centers, cfg.pad_sizes)  # fmt: skip
    want = oracle.spyral_rows(cloud, cfg.elec_params.windows_edge, cfg.elec_params.micromegas_edge,
                              cfg.det_params.length, resp, cfg.pad_centers, cfg.pad_sizes)  # fmt: skip
    assert got.shape == want.shape
    for col in (0, 1, 2, 3, 5, 6, 7):
        assert np.array_equal(got[:, col], want[:, col])
    assert np.allclose(got[:, 4], want[:, 4], rtol=1e-12, atol=0)


def test_run_simulation_with_array_writer(dist, tmp_path):
    """run_simulation over an .npz kinematics file, batched writer hook, Spyral rows from the GPU."""
    from attpc_engine_b200.kinematics import save_kinematics_npz

    cfg, m, v, zs, as_, idx = _workload(dist, "c16dd", 40)
    path = tmp_path / "kin.npz"
    save_kinematics_npz(path, v, m, zs, as_)
    writer = ArrayWriter(None, cfg, max_events_per_file=25)
    run_simulation(cfg, path, writer, seed=9, batch_size=16, verbose=False)
    direct = simulate_batch(m, v, zs, as_, cfg, 9, idx, spyral_rows=True)
    non_empty = np.nonzero(np.diff(direct.offsets) > 0)[0]  # empty clouds are skipped (`simulator.py:204`)
    assert len(non_empty) >= 30
    assert [len(f["event_numbers"]) for f in writer.files] == [25, len(non_empty) - 25]
    numbers = np.concatenate([f["event_numbers"] for f in writer.files])
    assert np.array_equal(numbers, non_empty)
    rows = np.concatenate([f["rows"] for f in writer.files])
    assert np.array_equal(rows, direct.rows)
    assert np.all(rows[:, 3] > cfg.elec_params.adc_threshold)

    class PerEvent:  # a user writer that only knows the reference's protocol
        def __init__(self):
            self.seen, self.closed = [], False

        def write(self, data, labels, config, event_number):
            self.seen.append((event_number, data, labels))

        def get_directory_name(self):
            return tmp_path

        def close(self):
            self.closed = True

    w = PerEvent()
    run_simulation(cfg, path, w, seed=9, batch_size=16, verbose=False)
    assert w.closed and [s[0] for s in w.seen] == list(non_empty)
    assert np.array_equal(np.concatenate([s[1] for s in w.seen]), direct.cloud)


def test_run_simulation_over_several_devices(dist, tmp_path):
    """`run_simulation(devices=[...])`: one worker thread and one engine per entry (here two engines on the one GPU of
    the test box), event ranges dealt round-robin, the writer fed in event order: the same files as a one-device run."""
    from attpc_engine_b200.kinematics import save_kinematics_npz

    cfg, m, v, zs, as_, idx = _workload(dist, "c16dd", 150)
    path = tmp_path / "kin.npz"
    save_kinematics_npz(path, v, m, zs, as_)
    one = ArrayWriter(None, cfg, max_events_per_file=1000)
    run_simulation(cfg, path, one, seed=5, batch_size=16, verbose=False)
    two = ArrayWriter(None, cfg, max_events_per_file=1000)
    run_simulation(cfg, path, two, seed=5, batch_size=16, verbose=False, devices=[0, 0, 0])
    assert len(one.files) == len(two.files) == 1
    for key in ("event_numbers", "offsets", "rows", "labels"):
        assert np.array_equal(one.files[0][key], two.files[0][key]), key
    assert len(one.files[0]["event_numbers"]) > 100

    class PerEvent:  # the reference's per-event protocol, raw clouds
        def __init__(self):
            self.seen = []

        def write(self, data, labels, config, event_number):
            self.seen.append((event_number, data, labels))

        def get_directory_name(self):
            return tmp_path

        def close(self):
            pass

    a, b = PerEvent(), PerEvent()
    run_simulation(cfg, path, a, seed=5, batch_size=32, verbose=False)
    run_simulation(cfg, path, b, seed=5, batch_size=8, verbose=False, devices=[0, 0])
    assert [e for e, _, _ in a.seen] == [e for e, _, _ in b.seen] == sorted(e for e, _, _ in a.seen)
    for (_, c1, l1), (_, c2, l2) in zip(a.seen, b.seen):
        assert np.array_equal(c1, c2) and np.array_equal(l1, l2)


def test_run_simulation_with_parquet_writer(dist, tmp_path):
    """run_simulation -> typed columns over PCIe -> ParquetCloudWriter: the file holds what simulate_batch returns."""
    pytest.importorskip("pyarrow")
    from attpc_engine_b200.detector import ParquetCloudWriter, read_parquet_clouds
    from attpc_engine_b200.kinematics import save_kinematics_npz

    cfg, m, v, zs, as_, idx = _workload(dist, "c16dd", 50)
    kin = tmp_path / "kin.npz"
    save_kinematics_npz(kin, v, m, zs, as_)
    writer = ParquetCloudWriter(tmp_path / "out")
    run_simulation(cfg, kin, writer, indices=idx, seed=12, batch_size=32, verbose=False)
    want = simulate_batch(m, v, zs, as_, cfg, 12, idx)
    ev, off, cloud, labels = read_parquet_clouds(tmp_path / "out" / "run_0000.parquet")
    nonempty = np.flatnonzero(np.diff(want.offsets))
    assert np.array_equal(ev, nonempty) and np.array_equal(np.diff(off), np.diff(want.offsets)[nonempty])
    assert np.array_equal(cloud, want.cloud) and np.array_equal(labels, want.labels)


def test_spyral_writer_layout_through_h5py_stand_in(dist, monkeypatch, tmp_path):
    """File layout of the reference's SpyralWriter (writer.py:164-281), with h5py replaced by an in-memory fake."""
    sys.path.insert(0, str((__import__("pathlib").Path(__file__).parent / "golden")))
    import ref_shim

    fake = types.ModuleType("h5py")
    fake.File, fake.Group, fake.Dataset = ref_shim.MemFile, ref_shim.MemGroup, ref_shim.MemDataset
    monkeypatch.setitem(sys.modules, "h5py", fake)
    ref_shim.MemFile.opened.clear()
    cfg, m, v, zs, as_, idx = _workload(dist, "c16dd", 12)
    writer = SpyralWriter(tmp_path, cfg, max_events_per_file=5)
    batch = simulate_batch(m, v, zs, as_, cfg, 4, idx, spyral_rows=True)
    for e in range(len(batch)):  # reference protocol: one write per event
        cloud, labels = batch.event(e)
        writer.write(cloud, labels, cfg, e)
    writer.close()
    files = ref_shim.MemFile.opened
    assert [str(f.path).rsplit("/", 1)[1] for f in files] == ["run_0000.h5", "run_0001.h5", "run_0002.h5"]
    assert all(f.closed for f in files)
    assert [(f["cloud"].attrs["min_event"], f["cloud"].attrs["max_event"]) for f in files] == [(0, 4), (5, 9), (10, 11)]
    d = files[1]["cloud"]["cloud_7"]
    rows, labels = batch.event_rows(7)
    assert np.array_equal(d.data, rows) and np.array_equal(files[1]["cloud"]["labels_7"].data, labels)
    assert d.attrs["orig_run"] == 1 and d.attrs["orig_event"] == 7 and d.attrs["ic_amplitude"] == -1.0
    # what the downstream consumer (Spyral's point-cloud phase; docs/user_guide/detector/index.md:176-196, writer.py:97-110,
    # 240-251) reads: events min_event..max_event of every file, columns x, y, z, amplitude, integral, pad, tb, scale
    win, mm = float(cfg.elec_params.windows_edge), float(cfg.elec_params.micromegas_edge)
    seen = 0
    for f in files:
        group = f["cloud"]
        for e in range(group.attrs["min_event"], group.attrs["max_event"] + 1):
            if f"cloud_{e}" not in group:  # (an event without points is not written, simulator.py:204)
                continue
            c, lab = group[f"cloud_{e}"].data, group[f"labels_{e}"].data
            assert c.ndim == 2 and c.shape[1] == 8 and c.dtype == np.float64 and len(lab) == len(c)
            if len(c) == 0:  # (every point below the ADC threshold: the reference writes the empty dataset too)
                continue
            pad = c[:, 5].astype(np.int64)
            assert np.array_equal(c[:, 5], pad) and pad.min() >= 0 and pad.max() < len(cfg.pad_sizes)
            assert np.array_equal(c[:, 0], cfg.pad_centers[pad, 0]) and np.array_equal(c[:, 1], cfg.pad_centers[pad, 1])
            assert np.array_equal(c[:, 7], cfg.pad_sizes[pad])
            assert np.array_equal(c[:, 2], (win - c[:, 6]) / (win - mm) * cfg.det_params.length * 1000.0)
            assert np.all(np.diff(c[:, 2]) >= 0.0) and c[:, 6].min() >= 0.0 and c[:, 6].max() < 512.0  # z-sorted, tb masked
            assert np.all(c[:, 3] > cfg.elec_params.adc_threshold) and np.all(c[:, 3] <= 4095.0) and np.all(c[:, 4] >= c[:, 3])
            assert set(np.unique(lab)) <= set(idx)
            seen += 1
    assert seen >= 10


@pytest.mark.parametrize("name", ["c16dd", "c12aa"])
def test_distributions_match_reference(dist, name):
    """KS tests at p > 0.01 against the unmodified reference run on the SAME kinematics (paired; the unpaired tests on
    all four workloads, with track observables, are in tests/test_gpu_statistics.py)."""
    cfg, m, v, zs, as_, idx = _workload(dist, name)
    dist = {k: (val[: len(m)] if k.startswith(name) and len(val) > len(m) and "sample" not in k else val)
            for k, val in dist.items()}  # the reference's observables of the same events
    batch = simulate_batch(m, v, zs, as_, cfg, 20261018, idx)
    n = np.diff(batch.offsets).astype(np.float64)
    sums = np.add.reduceat(batch.cloud[:, 2], batch.offsets[:-1][n > 0])
    ext, pads, med, mx, one = [], [], [], [], []
    picker = np.random.default_rng(2)
    for e in range(len(batch)):
        c, _ = batch.event(e)
        ext.append(c[:, 1].max() - c[:, 1].min() if len(c) else 0.0)
        pads.append(len(np.unique(c[:, 0])))
        med.append(np.median(c[:, 2]) if len(c) else 0.0)
        mx.append(c[:, 2].max() if len(c) else 0.0)
        if len(c):  # one random point per event: points of one event are correlated, events are not
            one.append(c[picker.integers(len(c)), 2])
    checks = {
        "points per event": (n, dist[f"{name}/n_points"]),
        "charge per event": (sums, dist[f"{name}/sum_charge"][dist[f"{name}/n_points"] > 0]),
        "time-bucket extent": (np.array(ext), dist[f"{name}/tb_extent"]),
        "pads per event": (np.array(pads, dtype=np.float64), dist[f"{name}/n_pads"]),
        "median point charge per event": (np.array(med), dist[f"{name}/median_charge"]),
        "max point charge per event": (np.array(mx), dist[f"{name}/max_charge"]),
        "charge per point (one point per event)": (np.array(one), dist[f"{name}/point_charge_sample"]),
    }
    for label, (ours, ref) in checks.items():
        p = ks_2samp(ours, ref).pvalue
        assert p > 0.01, f"{name}: {label}: KS p = {p:.4f}"


def _full_size_batch(name, n_events, seed):
    import bench

    config, momenta, vertices, zs, as_, indices = bench.build_workload(name, n_events)
    return config, zs, indices, simulate_batch(momenta, vertices, zs, as_, config, seed, indices), (momenta, vertices, as_)


@pytest.mark.parametrize("name, n_events", [("c16dd", 10000), ("c14dp", 4000), ("c12aa", 2000), ("sn132dp", 2000)])
def test_full_size_properties(name, n_events):
    """Size-independent properties at BASELINE.json config sizes (10k events is the reference's documented run)."""
    from attpc_engine_b200.detector.beam_pads import BEAM_PADS_ARRAY

    config, zs, indices, batch, (momenta, vertices, as_) = _full_size_batch(name, n_events, 99)
    off, cloud, labels = batch.offsets, batch.cloud, batch.labels
    assert len(off) == n_events + 1 and off[0] == 0 and off[-1] == len(cloud) == len(labels)
    assert np.all(np.diff(off) >= 0)
    pad, tbf, charge = cloud[:, 0], cloud[:, 1], cloud[:, 2]
    tb = np.floor(tbf)
    assert np.all((tbf >= 0) & (tbf < 512)) and np.all(tb >= config.elec_params.micromegas_edge)
    assert np.all((pad >= 0) & (pad < 10240) & (pad == np.floor(pad)))
    assert not np.isin(pad.astype(np.int64), BEAM_PADS_ARRAY).any()  # beam pads never fire
    assert np.all(charge >= 0) and np.all(charge == np.floor(charge))
    charged = [i for i in indices if zs[i] != 0]
    assert set(np.unique(labels)) <= set(charged)
    # canonical order inside every event: strictly ascending (time bucket, pad), hence unique keys
    key = tb * 16384 + pad
    inner = np.ones(len(key), dtype=bool)
    inner[off[1:-1][off[1:-1] < len(key)]] = False  # first row of an event may restart the order
    assert np.all(np.diff(key)[inner[1:]] > 0)
    # electrons are conserved up to the mesh truncation: the 10x10 mesh integrates 99.8627 % of the Gaussian and
    # every pixel truncates to an integer, so the cloud can never hold more than gain * primaries
    gain = config.det_params.mpgd_gain
    assert charge.sum() <= batch.stats["n_primary_electrons"] * gain
    assert batch.stats["n_deposits"] <= 100 * batch.stats["n_active_points"]
    assert batch.stats["n_hash_probes"] < 3 * batch.stats["n_deposits"]
    # determinism: the same seed reproduces the batch bit for bit; sharding it reproduces it too
    again = simulate_batch(momenta, vertices, zs, as_, config, 99, indices)
    assert np.array_equal(again.offsets, off) and np.array_equal(again.cloud, cloud) and np.array_equal(again.labels, labels)
    half = n_events // 2
    a = simulate_batch(momenta[:half], vertices[:half], zs, as_, config, 99, indices, first_event=0)
    b = simulate_batch(momenta[half:], vertices[half:], zs, as_, config, 99, indices, first_event=half)
    merged = concat_batches([a, b])
    assert np.array_equal(merged.offsets, off) and np.array_equal(merged.cloud, cloud)


def test_typed_columns_hold_the_same_rows(dist):
    """`columns=True` changes the wire format (11 B/row instead of 32 B/row), not the content."""
    cfg, m, v, zs, as_, idx = _workload(dist, "c16dd", 200)
    plain = simulate_batch(m, v, zs, as_, cfg, 31, idx)
    cols = simulate_batch(m, v, zs, as_, cfg, 31, idx, columns=True, max_events_per_launch=64, copy_events_per_launch=64)
    assert cols.columns is not None and cols.columns["pad"].dtype == np.int16 and cols.columns["label8"].dtype == np.int8
    assert cols.columns["tb_q16"].dtype == np.uint32
    assert np.array_equal(cols.offsets, plain.offsets)
    ev_cloud, ev_labels = cols.event(17)
    assert ev_cloud.dtype == np.float64 and ev_labels.dtype == np.int64
    assert np.array_equal(ev_cloud, plain.event(17)[0]) and np.array_equal(ev_labels, plain.event(17)[1])
    assert np.array_equal(cols.cloud, plain.cloud) and np.array_equal(cols.labels, plain.labels)


@pytest.mark.parametrize("name", ["c16dd", "c12aa", "sn132dp"])
def test_packed_columns_hold_the_same_rows(dist, name):
    """The packed wire form (8 B/row + 1 KB/event: rows per time bucket, wiggle, pad id + track rank in 16 bits) decodes
    to the typed columns of an unpacked call, and both to the float64 cloud; small launches and copy chunks, so that the
    per-event counts of many chunks land in the right places."""
    cfg, m, v, zs, as_, idx = _workload(dist, name, 300)
    n = len(m)
    plain = simulate_batch(m, v, zs, as_, cfg, 31, idx)
    loose = simulate_batch(m, v, zs, as_, cfg, 31, idx, columns=True, packed=False)
    tight = simulate_batch(m, v, zs, as_, cfg, 31, idx, columns=True, max_events_per_launch=64, copy_events_per_launch=64)
    assert loose.packed is None and loose.columns is not None
    if len(idx) <= 4:
        assert tight.packed is not None and tight.packed["tb_counts"].shape == (n, 512)
        assert np.array_equal(tight.packed["tb_counts"].sum(axis=1), np.diff(plain.offsets))
    else:  # more than four tracks: ranks do not fit above the pad id, the library answers with the plain columns
        assert tight.packed is None
    assert np.array_equal(tight.offsets, plain.offsets)
    for e in (0, 17, n - 1):
        assert np.array_equal(tight.event(e)[0], plain.event(e)[0]) and np.array_equal(tight.event(e)[1], plain.event(e)[1])
    assert tight.columns.keys() == loose.columns.keys()
    for key in loose.columns:
        assert np.array_equal(tight.columns[key], loose.columns[key]) and tight.columns[key].dtype == loose.columns[key].dtype, key
    assert np.array_equal(tight.cloud, plain.cloud) and np.array_equal(tight.labels, plain.labels)


@pytest.mark.parametrize("name, n", [("c16dd", 300), ("sn132dp", 150), ("c12aa", 60)])
def test_spyral_columns_rebuild_the_float64_rows(name, n):
    """`row_columns=True` ships the thresholded, z-sorted Spyral rows as typed columns (13 instead of 72 B/row); the
    host rebuilds x, y, z, amplitude, integral, pad, time bucket and pad size from them bit for bit.  Small launches
    and copy chunks: the rows of many chunks land in the right places."""
    import bench

    cfg, m, v, zs, as_, idx = bench.build_workload(name, n)
    full = simulate_batch(m, v, zs, as_, cfg, 17, idx, spyral_rows=True)
    cols = simulate_batch(m, v, zs, as_, cfg, 17, idx, spyral_rows=True, row_columns=True, rows_only=True,
                          max_events_per_launch=64, copy_events_per_launch=16)  # fmt: skip
    assert cols.row_columns is not None and cols.row_columns["pad"].dtype == np.int16
    assert cols.row_columns["e_hi"].dtype == np.uint16 and cols.stats["n_rows"] == full.stats["n_rows"] > 0
    assert np.array_equal(cols.row_offsets, full.row_offsets)
    rows7, labels7 = cols.event_rows(7)
    assert np.array_equal(rows7, full.event_rows(7)[0]) and np.array_equal(labels7, full.event_rows(7)[1])
    assert np.array_equal(cols.rows, full.rows) and np.array_equal(cols.row_labels, full.row_labels)
    if name == "sn132dp":
        assert (cols.row_columns["e_hi"] > 0).any() and (full.rows[:, 3] == 4095.0).any()  # saturated amplitudes were covered
    # and the float64 rows of the chunked call equal those of the plain call
    chunked = simulate_batch(m, v, zs, as_, cfg, 17, idx, spyral_rows=True, max_events_per_launch=64,
                             copy_events_per_launch=16)  # fmt: skip
    assert np.array_equal(chunked.row_offsets, full.row_offsets) and np.array_equal(chunked.rows, full.rows)
    assert np.array_equal(chunked.cloud, full.cloud)
    # unmasked time buckets: the Spyral pass over the float64 cloud writes the typed columns instead of finalize
    from attpc_engine_b200.detector.engine import engine_for
    from attpc_engine_b200.detector.simulator import _nuclei_for

    eng = engine_for(cfg, _nuclei_for(zs, as_, idx, nuclear_map))
    wide = eng.simulate_batch(m, v, zs, as_, idx, seed=17, spyral_rows=True, keep_all_tb=True)
    wide_cols = eng.simulate_batch(m, v, zs, as_, idx, seed=17, spyral_rows=True, keep_all_tb=True, row_columns=True,
                                   rows_only=True)  # fmt: skip
    assert wide_cols.row_columns is not None and wide_cols.stats["n_rows"] == wide.stats["n_rows"] > 0
    assert np.array_equal(wide_cols.row_offsets, wide.row_offsets)
    assert np.array_equal(wide_cols.rows, wide.rows) and np.array_equal(wide_cols.row_labels, wide.row_labels)


@pytest.mark.parametrize("compact", [True, False])
def test_typed_columns_with_large_electron_counts(compact, monkeypatch):
    """Heavy ions put more than 2^32 electrons on a pad: those rows are listed beside the uint32 column; a call with
    more of them than the list takes (forced here through ATTPC_BIG_CAP) comes back with the int64 column.  Both hold
    the same rows as the float64 path."""
    import bench

    cfg, m, v, zs, as_, idx = bench.build_workload("sn132dp", 150)
    plain = simulate_batch(m, v, zs, as_, cfg, 3, idx)
    if not compact:
        monkeypatch.setenv("ATTPC_BIG_CAP", "2")
    # (a tuning value of its own gives the call its own engine, created under the environment above)
    cols = simulate_batch(m, v, zs, as_, cfg, 3, idx, columns=True, hash_capacity=16384 if compact else 32768)
    assert ("electrons_u32" in cols.columns) == compact
    if compact:
        assert len(cols.columns["big_rows"]) > 2 and cols.columns["electrons_u32"].dtype == np.uint32
    else:
        assert cols.columns["electrons"].dtype == np.int64
    assert np.array_equal(cols.offsets, plain.offsets)
    assert np.array_equal(cols.event(7)[0], plain.event(7)[0])
    assert np.array_equal(cols.cloud, plain.cloud) and np.array_equal(cols.labels, plain.labels)


@pytest.mark.parametrize("name, n_events", [("c16dd", 10000), ("c14dp", 3000), ("c12aa", 2000), ("sn132dp", 2000)])
def test_mesh_weight_table_equals_reference_expression(name, n_events):
    """The constant mesh-weight table + exactness guard (default) gives the same integer shares as evaluating
    `pdf * step_x * step_y * electrons` (`transporter.py:36-41, 240-246`) for every pixel (ATTPC_EXACT_MESH)."""
    import bench
    from attpc_engine_b200.detector.engine import engine_for
    from attpc_engine_b200.detector.simulator import _nuclei_for

    config, momenta, vertices, zs, as_, indices = bench.build_workload(name, n_events)
    eng = engine_for(config, _nuclei_for(zs, as_, indices, nuclear_map))
    fast = eng.simulate_batch(momenta, vertices, zs, as_, indices, seed=5)
    eng.exact_mesh = True
    try:
        exact = eng.simulate_batch(momenta, vertices, zs, as_, indices, seed=5)
    finally:
        eng.exact_mesh = False
    assert fast.stats["n_deposits"] == exact.stats["n_deposits"] > 0
    assert np.array_equal(fast.offsets, exact.offsets) and np.array_equal(fast.labels, exact.labels)
    assert np.array_equal(fast.cloud, exact.cloud)


@pytest.mark.parametrize("name", ["c16dd", "c12aa"])
def test_device_resident_call_holds_the_same_rows(name):
    """`host_copy=False` (what `bench.py` times as `value`) takes other code paths than a call that copies to the host:
    all groups of a launch in one chunk, entry lists beyond 8192 entries through `order_queue_kernel` (a few 16C(d,d')
    events, most of 12C(a,a')3a), float64 rows written on the device.  Its rows, read back from the device, equal the
    rows of the copying call."""
    import bench
    from attpc_engine_b200 import nuclear_map
    from attpc_engine_b200.detector.engine import engine_for
    from attpc_engine_b200.detector.simulator import _nuclei_for

    n = 6000 if name == "c16dd" else 1500
    cfg, momenta, vertices, zs, as_, indices = bench.build_workload(name, n, seed_offset=5)
    eng = engine_for(cfg, _nuclei_for(zs, as_, indices, nuclear_map))
    host = eng.simulate_batch(momenta, vertices, zs, as_, indices, seed=11, first_event=70000)
    there = eng.simulate_batch(momenta, vertices, zs, as_, indices, seed=11, first_event=70000, host_copy=False)
    assert there.device is not None and there.stats["n_points"] == host.stats["n_points"] > 0
    back = eng.read_device_result(there)
    assert np.array_equal(back.offsets, host.offsets)
    assert np.array_equal(back.cloud, host.cloud) and np.array_equal(back.labels, host.labels)
    if name == "c12aa":
        assert (np.diff(host.offsets) > 8192).any()  # lists long enough for the second tier (order_queue_kernel)
