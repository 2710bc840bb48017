"""User-facing parameter records and ``Config`` (reference: `detector/parameters.py:10-261`).

Field names, constructor argument names and derived attributes are kept one-for-one so that a
reference ``apply_detector.py`` script runs unchanged.  Differences, all deliberate:

* the packaged pad-plane geometry lives in one compressed container
  (``data/attpc_pad_plane.npz``: ``grid``, ``edges``, ``centers``, ``scales``) instead of
  three files; user-supplied paths are still read in the reference's formats
  (``.npz`` with ``grid``/``edges``; CSV with one header line);
* a non-default ``pad_size_path`` is honoured (the reference reads ``geometry_path``
  there, `parameters.py:255`);
* ``gas_target`` is duck-typed (``get_dedx(nucleus, ke_mev)``, ``density``), spyral_utils
  is not imported.
"""

from __future__ import annotations

from dataclasses import dataclass
from functools import lru_cache
from importlib import resources
from pathlib import Path
from typing import Any

import numpy as np

from .constants import NUM_PADS

DEFAULT = "Default"


@dataclass
class DetectorParams:
    """Detector parameters (`parameters.py:10-48`).

    length [m], efield [V/m], bfield [T], mpgd_gain (int, unitless), gas_target,
    diffusion [V] (transverse), fano_factor, w_value [eV], longitudinal_diffusion [V].

    ``longitudinal_diffusion`` is an extension (the reference has no such field) and the last
    field, so that the reference's eight positional arguments still work.  It spreads every
    ionisation point over the time buckets ``floor(t -+ 3 sigma_L)``, with
    ``sigma_L = sqrt(2 D_L dv t / efield) / dv`` time buckets after a drift of ``t`` buckets; the
    default 0 keeps the reference's one bucket per point (see DESIGN.md §3a).
    """

    length: float
    efield: float
    bfield: float
    mpgd_gain: int
    gas_target: Any
    diffusion: float
    fano_factor: float
    w_value: float
    longitudinal_diffusion: float = 0.0


@dataclass
class ElectronicsParams:
    """GET electronics parameters (`parameters.py:51-76`).

    clock_freq [MHz], amp_gain [lsb/fC], shaping_time [ns], micromegas_edge [TB],
    windows_edge [TB], adc_threshold [ADC].
    """

    clock_freq: float
    amp_gain: int
    shaping_time: int
    micromegas_edge: int
    windows_edge: int
    adc_threshold: int


@dataclass
class PadParams:
    """Paths of the pad-plane description (`parameters.py:79-94`); ``"Default"`` = packaged."""

    grid_path: Path | str = DEFAULT
    geometry_path: Path | str = DEFAULT
    pad_size_path: Path | str = DEFAULT


@lru_cache(maxsize=1)
def _packaged_pad_plane() -> dict[str, np.ndarray]:
    handle = resources.files("attpc_engine_b200.detector.data").joinpath("attpc_pad_plane.npz")
    with resources.as_file(handle) as path:
        with np.load(path) as data:
            return {k: data[k] for k in ("grid", "edges", "centers", "scales")}


def _read_csv_columns(path: Path | str, n_cols: int) -> np.ndarray:
    out = np.zeros((NUM_PADS, n_cols))
    with open(path, "r") as handle:
        handle.readline()  # header
        for pad_number, line in enumerate(handle):
            if not line.strip():
                continue
            entries = line.split(",")
            for c in range(n_cols):
                out[pad_number, c] = float(entries[c])
    return out


class Config:
    """All inputs of the detector simulation plus derived data (`parameters.py:97-261`).

    Attributes: ``det_params``, ``elec_params``, ``pad_params``, ``pad_grid`` (int16
    [5600, 5600], pad id or -1), ``pad_grid_edges`` ([low, high, step] in mm), ``pad_centers``
    (float64 [10240, 2], mm), ``pad_sizes`` (float64 [10240]), ``drift_velocity`` (m / TB).
    """

    def __init__(
        self,
        detector_params: DetectorParams,
        electronics_params: ElectronicsParams,
        pad_params: PadParams,
    ):
        self.det_params = detector_params
        self.elec_params = electronics_params
        self.pad_params = pad_params
        self.pad_grid: np.ndarray | None = None
        self.pad_grid_edges: np.ndarray | None = None
        self.pad_centers: np.ndarray | None = None
        self.pad_sizes: np.ndarray | None = None
        self.drift_velocity = 0.0
        self.calculate_drift_velocity()
        self.load_pad_grid()
        self.load_pad_centers()
        self.load_pad_sizes()

    def calculate_drift_velocity(self) -> None:
        """length / (windows_edge - micromegas_edge), in m per time bucket (`:164-174`)."""
        self.drift_velocity = self.det_params.length / float(
            self.elec_params.windows_edge - self.elec_params.micromegas_edge
        )

    def load_pad_grid(self) -> None:
        """Pad-id mesh, inclusive on the low edge and exclusive on the high edge (`:176-205`)."""
        if self.pad_params.grid_path == DEFAULT:
            packed = _packaged_pad_plane()
            self.pad_grid = packed["grid"]
            self.pad_grid_edges = packed["edges"]
        else:
            with np.load(self.pad_params.grid_path) as data:
                self.pad_grid = data["grid"]
                self.pad_grid_edges = data["edges"]

    def load_pad_centers(self) -> None:
        """Pad centres in mm (`:207-235`)."""
        if self.pad_params.geometry_path == DEFAULT:
            self.pad_centers = _packaged_pad_plane()["centers"].copy()
        else:
            self.pad_centers = _read_csv_columns(self.pad_params.geometry_path, 2)

    def load_pad_sizes(self) -> None:
        """Pad size class per pad (`:237-261`)."""
        if self.pad_params.pad_size_path == DEFAULT:
            self.pad_sizes = _packaged_pad_plane()["scales"].copy()
        else:
            self.pad_sizes = _read_csv_columns(self.pad_params.pad_size_path, 1)[:, 0]
