"""CPU model of longitudinal diffusion -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

Longitudinal diffusion is an extension outside the reference (DESIGN.md §3a), so `oracle/attpc_oracle.py`, which
restates the reference, has no such term.  This module restates the extension literally on top of the oracle's own
drift helpers, for `tests/test_longitudinal.py` and `tests/test_gpu_longitudinal.py`:

* `longitudinal_split`: time buckets and electrons of the sub-points of one point;
* `track_to_cloud`: the oracle's `track_to_cloud` with every point replaced by its sub-points, which also counts the
  (sub-point, pixel) deposits per key -- the bound of a charge difference that a flipped truncation can cause.
"""

from __future__ import annotations

import math

import numpy as np
from numba import njit, types
from numba.typed import Dict

from oracle.attpc_oracle import BEAM_PAD_IDS, MESH_N, _deposit, _grid_index, _is_beam_pad, szudzik_pair


def longitudinal_split(time, electrons, longitudinal_diffusion, efield, dv):
    """Time buckets and electrons of the sub-points of one point of drift time ``time`` [time buckets].

    sigma_L = sqrt(2 D_L dv t / E) / dv; buckets k = max(0, floor(t - 3 sigma_L)) .. floor(t + 3 sigma_L), each with
    int(q * (Phi((k + 1 - t) / sigma_L) - Phi((k - t) / sigma_L))), Phi(x) = 0.5 erfc(-x / sqrt(2)), zeros included.
    sigma_L <= 0 or NaN (t <= 0): the single bucket int(t) with all electrons (none when int(t) < 0).
    """
    with np.errstate(invalid="ignore"):
        sl = float(np.sqrt(np.float64(2.0 * longitudinal_diffusion * dv * time / efield))) / dv
    if not sl > 0.0:
        tb = int(time)
        return ([tb], [int(electrons)]) if tb >= 0 else ([], [])
    w = 3.0 * sl
    tbs = list(range(max(0, math.floor(time - w)), math.floor(time + w) + 1))
    root2 = math.sqrt(2.0)
    out = []
    for k in tbs:
        hi = 0.5 * math.erfc(-((k + 1 - time) / sl) / root2)
        lo = 0.5 * math.erfc(-((k - time) / sl) / root2)
        out.append(int((hi - lo) * float(electrons)))
    return tbs, out


def new_counts():
    """Typed dict key -> number of (sub-point, pixel) deposits, filled by `track_to_cloud`."""
    return Dict.empty(key_type=types.int64, value_type=types.int64)


@njit(cache=False)
def _drift_subpoints(pad_grid, edges, beam_ids, diffusion, efield, dv, xs, ys, times, tbs, electrons, cloud, label,
                     counts):
    """The oracle's `drift_track` on sub-points: the time bucket is given (tbs), the transverse sigma still follows
    ``times``; every deposit is also counted per key."""
    for k in range(len(times)):
        t = times[k]
        tb = tbs[k]
        cx = xs[k]
        cy = ys[k]
        n_e = electrons[k]
        sigma = np.sqrt(2.0 * diffusion * dv * t / efield)
        if sigma == 0.0:
            ix, iy = _grid_index(edges, cx, cy)
            if ix == -1 or iy == -1:
                continue
            pad = int(pad_grid[ix, iy])
            if pad != -1 and not _is_beam_pad(pad, beam_ids):
                key = szudzik_pair(tb, pad)
                _deposit(cloud, key, n_e, label)
                counts[key] = counts.get(key, 0) + 1
            continue
        lo_x = cx - 3 * sigma
        hi_x = cx + 3 * sigma
        lo_y = cy - 3 * sigma
        hi_y = cy + 3 * sigma
        dx = (hi_x - lo_x) / (MESH_N - 1)
        dy = (hi_y - lo_y) / (MESH_N - 1)
        cell_x = 2 * 3 * sigma / (MESH_N - 1)
        cell_y = 2 * 3 * sigma / (MESH_N - 1)
        norm = 1 / 2 / np.pi / (sigma**2)
        for i in range(MESH_N):
            px = lo_x + i * dx
            if i == MESH_N - 1:
                px = hi_x
            for j in range(MESH_N):
                py = lo_y + j * dy
                if j == MESH_N - 1:
                    py = hi_y
                ix, iy = _grid_index(edges, px, py)
                if ix == -1 or iy == -1:
                    continue
                pad = int(pad_grid[ix, iy])
                if pad == -1 or _is_beam_pad(pad, beam_ids):
                    continue
                arg = (-1 / 2 / sigma**2) * (((px - cx) ** 2) + ((py - cy) ** 2))
                share = int((norm * np.exp(arg)) * (cell_x * cell_y) * n_e)
                key = szudzik_pair(tb, pad)
                _deposit(cloud, key, share, label)
                counts[key] = counts.get(key, 0) + 1


def track_to_cloud(track, electrons, config, cloud, label, longitudinal_diffusion, counts):
    """`oracle.track_to_cloud` (>= 1 mask, gain, z -> time, drift) with longitudinal diffusion: every point becomes
    the sub-points of `longitudinal_split`; ``counts`` (`new_counts`) receives the deposits per key."""
    keep = electrons >= 1
    track = track[keep]
    electrons = electrons[keep] * int(config.det_params.mpgd_gain)
    dv = config.drift_velocity
    times = (config.det_params.length - track[:, 2]) / dv + config.elec_params.micromegas_edge
    sub = ([], [], [], [], [])
    for x, y, t, q in zip(track[:, 0], track[:, 1], times, electrons):
        tbs, es = longitudinal_split(t, q, longitudinal_diffusion, config.det_params.efield, dv)
        for tb, e in zip(tbs, es):
            for col, v in zip(sub, (x, y, t, tb, e)):
                col.append(v)
    _drift_subpoints(
        config.pad_grid, config.pad_grid_edges, BEAM_PAD_IDS, config.det_params.diffusion, config.det_params.efield,
        dv, np.array(sub[0], dtype=np.float64), np.array(sub[1], dtype=np.float64), np.array(sub[2], dtype=np.float64),
        np.array(sub[3], dtype=np.int64), np.array(sub[4], dtype=np.int64), cloud, label, counts,
    )  # fmt: skip
