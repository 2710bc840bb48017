"""Replay events built from a list of points, and what the oracle says they must give.

A point is ``(pad, tb, electrons, rank)``: ``electrons`` primary electrons of the track at position ``rank`` of the
event's ``indices`` land on pad ``pad`` in time bucket ``tb``.  With ``diffusion = 0`` every active point of a replayed
track makes exactly one (pad, time bucket) key (`transporter.py:123-169`), so such an event fixes the number of keys,
entries, copies, electrons, time buckets and labels that the CUDA path sees, and `oracle.simulate_event` (with
``tracks`` / ``normals`` / ``record``) gives the expected answer.

* Position: the pad centre (``config.pad_centers``, mm -> m); only pads whose centre maps back to the pad through the
  oracle's ``_grid_index`` + ``pad_grid`` and that are not beam pads are used (`usable_pads`).
* Depth: ``z = length - (tb + 0.5 - micromegas_edge) * drift_velocity`` (replayed rows may leave the detector, so any
  time bucket can be reached).
* Electrons: a leading row per track (row 0 of a track makes no electrons, `solver.py:338-339`), then kinetic energies
  that fall by ``(e + 0.5) W`` per row, normal 0: ``int(mean) = e`` exactly (checked against `oracle.fano_electrons`).
"""

from __future__ import annotations

from dataclasses import dataclass, field

import numpy as np

from attpc_engine_b200 import nuclear_map
from oracle import attpc_oracle as oracle
from tests.common import reference_cloud_from_dict, sort_cloud

ZA = (1, 2)  # every charged track is a deuteron
NEUTRAL_ZA = (0, 1)
TAIL_KE_MEV = 1.0  # kinetic energy after the last point of a track


_PADS: dict = {}


def usable_pads(config) -> np.ndarray:
    """Pads whose centre maps back to the pad (oracle ``_grid_index`` + ``pad_grid``) and that are not beam pads."""
    key = (id(config.pad_grid), id(config.pad_centers))
    if key not in _PADS:
        c = np.asarray(config.pad_centers, dtype=np.float64) / 1000.0
        beam = set(int(p) for p in oracle.BEAM_PAD_IDS)
        out = []
        for pad in range(len(c)):
            ix, iy = oracle._grid_index(config.pad_grid_edges, c[pad, 0], c[pad, 1])
            if ix != -1 and iy != -1 and int(config.pad_grid[ix, iy]) == pad and pad not in beam:
                out.append(pad)
        _PADS[key] = np.array(out, dtype=np.int64)
    return _PADS[key]


def position(config, pad: int, tb: int) -> tuple[float, float, float]:
    cx, cy = (float(v) / 1000.0 for v in config.pad_centers[pad])
    z = config.det_params.length - (tb + 0.5 - config.elec_params.micromegas_edge) * config.drift_velocity
    return cx, cy, z


def track_rows(config, points, mass: float) -> np.ndarray:
    """Rows ``[x, y, z, gbx, gby, gbz]`` of one track: a leading row, then one row per ``(pad, tb, electrons)``."""
    w = config.det_params.w_value
    e = np.array([p[2] for p in points], dtype=np.float64)
    # kinetic energy of every row: falls by (e + 0.5) W from one row to the next
    ke = TAIL_KE_MEV + np.concatenate([np.cumsum(((e + 0.5) * w * 1.0e-6)[::-1])[::-1], [0.0]])
    gamma = ke / mass + 1.0
    gb = np.sqrt(gamma * gamma - 1.0)
    rows = np.zeros((len(points) + 1, 6), dtype=np.float64)
    for i, (pad, tb, _) in enumerate(points):
        rows[i + 1, :3] = position(config, pad, tb)
    rows[0, :3] = rows[1, :3] if len(points) else position(config, int(usable_pads(config)[0]), 0)
    rows[:, 5] = gb
    return rows


@dataclass
class Event:
    """Points ``(pad, tb, electrons, rank)`` and the nucleus index (label) of every rank; ``neutral`` ranks make no
    track.  Ranks without points still make a (one-row) track unless they are neutral."""

    points: list
    indices: list = field(default_factory=lambda: [0])
    neutral: frozenset = frozenset()


@dataclass
class Built:
    tracks: list
    normals: list
    track_event: list
    track_rank: list
    track_label: list
    track_za: list
    n_events: int
    electrons: list  # per track, what `solver.py:343-346` gives
    uniforms: list  # per event (keys, u)
    records: list  # per event: the oracle's dict (keys, charges, labels) in insertion order
    clouds: list  # per event: expected (cloud, labels) in canonical order
    predicted_entries: list  # per event, or None where the split does not fix it

    def replay_args(self):
        return (self.tracks, self.normals, self.track_event, self.track_rank, self.track_label, self.track_za,
                self.n_events)  # fmt: skip

    @property
    def entries(self) -> int:
        return int(sum(self.predicted_entries))


def build(config, events, unit_points=None, uniforms=None, seed=0, keep_all_tb=False) -> Built:
    """Replay inputs for `Engine.simulate_replay` and the oracle's expectation of ``events`` (list of `Event`).

    ``uniforms``: per event, a map Szudzik key -> wiggle, or None for a draw seeded by ``seed``; a key the map lacks
    is drawn too.  ``unit_points=1``: every point is its own work unit, so the entries of an event are its active
    points; with the default split an event of at most 1024 points lists each key once.
    """
    mass = float(nuclear_map.get_data(*ZA).mass)
    w, fano = config.det_params.w_value, config.det_params.fano_factor
    rng = np.random.default_rng(seed)
    out = Built([], [], [], [], [], [], len(events), [], [], [], [], [])
    for e, ev in enumerate(events):
        n_ranks = len(ev.indices)
        per_rank = [[] for _ in range(n_ranks)]
        for pad, tb, el, rank in ev.points:
            if rank in ev.neutral:
                raise ValueError("a neutral rank makes no points")
            per_rank[rank].append((int(pad), int(tb), int(el)))
        n_nuclei = max(ev.indices) + 1
        zs = np.full(n_nuclei, NEUTRAL_ZA[0], dtype=np.int64)
        as_ = np.full(n_nuclei, NEUTRAL_ZA[1], dtype=np.int64)
        ev_tracks, ev_normals = [], []
        for rank in range(n_ranks):
            if rank in ev.neutral:
                continue
            zs[ev.indices[rank]], as_[ev.indices[rank]] = ZA
            rows = track_rows(config, per_rank[rank], mass)
            normals = np.zeros(len(rows))
            got = oracle.fano_electrons(rows, mass, w, fano, normals=normals)
            want = np.array([0] + [p[2] for p in per_rank[rank]], dtype=np.int64)
            assert np.array_equal(got, want), "synthetic kinetic energies do not give the intended electrons"
            ev_tracks.append(rows)
            ev_normals.append(normals)
            out.tracks.append(rows)
            out.normals.append(normals)
            out.track_event.append(e)
            out.track_rank.append(rank)
            out.track_label.append(int(ev.indices[rank]))
            out.track_za.append(ZA)
            out.electrons.append(want)
        record: dict = {}
        n_rows = sum(len(t) for t in ev_tracks)
        oracle.simulate_event(
            None, None, zs, as_, config, None, list(ev.indices), nuclear_map, record=record,
            tracks=ev_tracks, normals=ev_normals, uniforms=np.zeros(100 * n_rows + 1),  # (a mesh point makes <= 100 keys)
        )  # fmt: skip
        keys, charges, labels = record["keys"], record["charges"], record["key_labels"]
        given = {} if uniforms is None or uniforms[e] is None else uniforms[e]
        drawn = rng.uniform(size=len(keys))
        u = np.array([given.get(int(k), drawn[i]) for i, k in enumerate(keys)], dtype=np.float64)
        out.uniforms.append((keys.copy(), u))
        out.records.append((keys.copy(), charges.copy(), labels.copy()))
        cloud, lab = reference_cloud_from_dict(keys, charges, labels, u, num_tb=np.inf if keep_all_tb else 512)
        out.clouds.append(sort_cloud(cloud, lab))
        out.predicted_entries.append(predicted_entries(config, ev, unit_points))
    return out


def predicted_entries(config, ev: Event, unit_points=None):
    """Entries of the event's list after the deposit kernel (occupied entries, before the time-bucket mask)."""
    if config.det_params.diffusion != 0.0:
        return None
    active = [(p[0], p[1]) for p in ev.points if p[2] >= 1 and 0 <= p[1] < 8192]
    if unit_points == 1:
        return len(active)
    if unit_points is None and (len(active) <= 1024 or len(set(active)) == len(active)):
        return len(set(active))
    return None


def expected_spyral(config, cloud, labels, threshold=None):
    """`spyral_event` (`writer.py:220-238`) of a cloud in the CUDA path's canonical order, with a STABLE z order: equal
    z keep their cloud order, the documented tie rule of the CUDA path (numpy's default quicksort leaves it open)."""
    resp = oracle.get_response(config)
    rows = oracle.spyral_rows(cloud, config.elec_params.windows_edge, config.elec_params.micromegas_edge,
                              config.det_params.length, resp, config.pad_centers, config.pad_sizes)  # fmt: skip
    thr = config.elec_params.adc_threshold if threshold is None else threshold
    keep = rows[:, 3] > thr
    rows, labels = rows[keep], np.asarray(labels)[keep]
    order = np.argsort(rows[:, 2], kind="stable")
    return rows[order], labels[order]
