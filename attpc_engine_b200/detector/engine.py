"""Host driver of the CUDA detector path: bakes ``Config`` into device constants and calls the C ABI.

What is baked (once per ``Config`` x species set x device):

* the pad lookup table -- the 1 mm sub-lattice of ``Config.pad_grid`` that
  `detector/transporter.py:102-120` (``position_to_index``) can address, with holes and the
  beam pads of `detector/beam_pads.py` folded to -1 (`transporter.py:165,237`);
* pad centres / sizes (`parameters.py:207-261`), the GET response (`response.py:8-32`);
* one stopping-power table per ion species (``target.DedxTable``), sampled from the user's
  ``gas_target.get_dedx`` (`solver.py:64-66`).
"""

from __future__ import annotations

import ctypes as C
import math

import numpy as np

from .. import _lib
from ..target import TableGasTarget, ensure_table_target
from .beam_pads import BEAM_PADS_ARRAY
from .constants import NUM_TB
from .parameters import Config
from .response import get_response


def build_pad_lut(pad_grid: np.ndarray, edges: np.ndarray) -> tuple[np.ndarray, int]:
    """Fold `position_to_index` + grid read + beam veto into one int16 table on whole millimetres.

    Returns ``(lut, origin_mm)`` with ``lut[fx - origin, fy - origin]`` = pad id or -1 for every
    integer ``fx = floor(x_mm)`` accepted by `transporter.py:109-115` (``low <= fx < high``).
    The grid index uses the reference's own expression ``int((fx - low) / bin)``.
    """
    low, high, step = (float(v) for v in edges[:3])
    first = math.ceil(low)
    last_excl = math.ceil(high)  # integers f with f < high
    fs = np.arange(first, last_excl, dtype=np.float64)
    idx = ((fs - low) / step).astype(np.int64)
    ok = (idx >= 0) & (idx < pad_grid.shape[0])
    safe = np.where(ok, idx, 0)
    lut = pad_grid[np.ix_(safe, safe)].astype(np.int16)
    lut[~ok, :] = -1
    lut[:, ~ok] = -1
    lut[np.isin(lut, BEAM_PADS_ARRAY)] = -1
    return np.ascontiguousarray(lut), int(first)


def default_freeze_ke(fano_factor: float, w_value: float, z_abs_max: float = 8.66) -> float:
    """Energy budget [MeV] below which a grid step can no longer make an electron.

    A grid step produces ``int(n + sqrt(F n) z)`` electrons with ``n = |dKE| / W``
    (`solver.py:338-346`) and the device's Box-Muller normal is bounded by ``z_abs_max``, so
    ``n + sqrt(F n) z_max < 1`` for ``n < n*``.  The integrator ends a track once the kinetic
    energy it can still gain or lose while relaxing to its terminal drift is below ``n* W``
    (`csrc/attpc_kernels.cuh: inert_forever`).  The reference instead integrates the stalled ion
    to 1 us and discards those rows at `solver.py:387`.
    """
    a = math.sqrt(max(fano_factor, 0.0)) * z_abs_max
    root = (-a + math.sqrt(a * a + 4.0)) / 2.0  # sqrt(n*) solves n + a sqrt(n) = 1
    return 0.999 * root * root * w_value * 1.0e-6


class SimBatch:
    """CSR point clouds of a batch: event ``e`` owns rows ``offsets[e]:offsets[e+1]``.

    Rows are either held as the reference's arrays (``cloud`` float64 ``[N, 3]`` = pad, time bucket, electrons;
    ``labels`` int64 ``[N]``) or, for batches simulated with ``columns=True``, as typed columns (``pad`` int16,
    ``tb_q16`` uint32 = the float64 time bucket times 65536, exactly (Q16.16 fixed point), ``label8`` int8 and the
    electron counts either as ``electrons`` int64 or -- the default for light ions -- as ``electrons_u32`` (count modulo
    2^32) plus the sorted ``big_rows`` / ``big_electrons`` of the rows that need more: 11 instead of 32 bytes per row
    over PCIe).  ``cloud`` / ``labels`` / ``event(e)`` work in both
    cases; with columns they are materialised on demand.

    The engine ships the columns in a packed form when it can (``packed``: 8 B/row + 1 KB/event): rows are in ascending
    time-bucket order, so the integer time bucket travels as ``tb_counts [B, 512]`` (rows per time bucket and event), the
    wiggle as ``wiggle`` uint16, and the track rank sits in the two bits above the 14-bit pad id (``pad_rank`` uint16;
    ``labels_of_rank`` maps it to the nucleus index).  ``columns`` then decodes them on first use.
    """

    def __init__(self, first_event, offsets, cloud=None, labels=None, row_offsets=None, rows=None, row_labels=None,
                 stats=None, columns=None, row_columns=None, row_builder=None, packed=None):  # fmt: skip
        self.first_event = first_event
        self.offsets = offsets
        self._cloud = cloud
        self._labels = labels
        self.row_offsets = row_offsets
        self._rows = rows  # [M, 8] Spyral rows
        self._row_labels = row_labels
        self.stats = {} if stats is None else stats
        self._columns = columns  # dict(pad, tb_q16, label8, and electrons or electrons_u32 + big_rows + big_electrons) or None
        #: packed wire form of the same columns: dict(pad_rank uint16, wiggle uint16, tb_counts uint16 [B, 512],
        #: labels_of_rank int8 [4], rank_shift, and the electron columns) or None
        self.packed = packed
        self.device = None  # device pointers of a call made with host_copy=False (`Engine.read_device_result`)
        #: Spyral rows (after ADC threshold, z-sorted) as typed columns: dict(pad int16, tb_q16 uint32, e_lo uint32,
        #: e_hi uint16, label8 int8) -- 13 B/row over PCIe instead of 72; ``rows`` / ``row_labels`` / ``event_rows`` rebuild
        #: the float64 arrays from them on demand, bit for bit (`Engine.rows_from_columns`)
        self.row_columns = row_columns
        self._row_builder = row_builder

    @property
    def columns(self):
        if self._columns is None and self.packed is not None:
            self._columns = self._unpack(0, len(self), 0, len(self.packed["pad_rank"]))
        return self._columns

    @columns.setter
    def columns(self, value):
        self._columns = value

    def _unpack(self, e0: int, e1: int, a: int, b: int) -> dict:
        """Typed columns of events ``e0:e1`` (rows ``a:b``) from the packed wire form."""
        p = self.packed
        shift = p["rank_shift"]
        pad_rank = p["pad_rank"][a:b]
        counts = p["tb_counts"][e0:e1]
        tb = np.repeat(np.tile(np.arange(counts.shape[1], dtype=np.uint32), e1 - e0), counts.ravel())
        out = dict(
            pad=(pad_rank & np.uint16((1 << shift) - 1)).astype(np.int16),
            tb_q16=(tb << np.uint32(16)) | p["wiggle"][a:b],
            label8=p["labels_of_rank"][pad_rank >> np.uint16(shift)],
        )
        if "electrons" in p:
            out["electrons"] = p["electrons"][a:b]
        else:
            lo, hi = np.searchsorted(p["big_rows"], [a, b])
            out.update(electrons_u32=p["electrons_u32"][a:b], big_rows=p["big_rows"][lo:hi] - a,
                       big_electrons=p["big_electrons"][lo:hi])  # fmt: skip
        return out

    @property
    def rows(self):
        if self._rows is None and self.row_columns is not None:
            self._rows, self._row_labels = self._row_builder(self.row_columns)
        return self._rows

    @rows.setter
    def rows(self, value):
        self._rows = value

    @property
    def row_labels(self):
        if self._row_labels is None and self.row_columns is not None:
            self._rows, self._row_labels = self._row_builder(self.row_columns)
        return self._row_labels

    @row_labels.setter
    def row_labels(self, value):
        self._row_labels = value

    def __len__(self) -> int:
        return len(self.offsets) - 1

    def _electrons(self, a: int = 0, b: int | None = None) -> np.ndarray:
        """Electron counts of rows ``a:b`` from the typed columns, as float64 (exact: counts are < 2^53)."""
        c = self.columns
        if "electrons" in c:
            return c["electrons"][a:b].astype(np.float64)
        out = c["electrons_u32"][a:b].astype(np.float64)  # low 32 bits; the few larger counts are listed apart
        rows = c["big_rows"]
        if len(rows):
            b = len(c["electrons_u32"]) if b is None else b
            lo, hi = np.searchsorted(rows, [a, b])
            out[rows[lo:hi] - a] = c["big_electrons"][lo:hi]
        return out

    def _decode_packed(self) -> bool:
        """Cloud and labels straight from the packed columns in one multi-threaded pass (`_decode.py`), when possible."""
        if self.packed is None or self._cloud is not None:
            return False
        from ._decode import decode_packed

        out = decode_packed(self.packed, self.offsets)
        if out is None:
            return False
        self._cloud, self._labels = out
        return True

    @property
    def cloud(self) -> np.ndarray:
        if self._cloud is None and self._decode_packed():
            return self._cloud
        if self._cloud is None and self.columns is not None:
            c = self.columns
            out = np.empty((len(c["pad"]), 3), dtype=np.float64)
            out[:, 0] = c["pad"]
            out[:, 1] = c["tb_q16"]
            out[:, 1] *= 1.0 / 65536.0  # exact: Q16.16 fixed point
            out[:, 2] = self._electrons()
            self._cloud = out
        return self._cloud

    @property
    def labels(self) -> np.ndarray:
        if self._labels is None and self._decode_packed():
            return self._labels
        if self._labels is None and self.columns is not None:
            self._labels = self.columns["label8"].astype(np.int64)
        return self._labels

    def event(self, e: int) -> tuple[np.ndarray, np.ndarray]:
        """``(cloud [n, 3] float64, labels [n] int64)`` of event ``e``, like `simulate` returns them."""
        a, b = self.offsets[e], self.offsets[e + 1]
        if self._cloud is None and self._columns is None and self.packed is not None:  # only this event is decoded
            one = SimBatch(self.first_event + e, np.array([0, b - a]), columns=self._unpack(e, e + 1, int(a), int(b)))
            return one.cloud, one.labels
        if self._cloud is None and self.columns is not None:
            c = self.columns
            cloud = np.empty((b - a, 3), dtype=np.float64)
            cloud[:, 0] = c["pad"][a:b]
            cloud[:, 1] = c["tb_q16"][a:b]
            cloud[:, 1] *= 1.0 / 65536.0
            cloud[:, 2] = self._electrons(int(a), int(b))
            return cloud, c["label8"][a:b].astype(np.int64)
        return self.cloud[a:b], self.labels[a:b]

    def event_rows(self, e: int) -> tuple[np.ndarray, np.ndarray]:
        """``(rows [n, 8] float64, labels [n] int64)`` of event ``e`` as `SpyralWriter.write` stores them."""
        a, b = self.row_offsets[e], self.row_offsets[e + 1]
        if self._rows is None and self.row_columns is not None:  # only this event's rows are materialised
            return self._row_builder({k: v[a:b] for k, v in self.row_columns.items()})
        return self.rows[a:b], self.row_labels[a:b]


def _ptr(arr: np.ndarray, ctype):
    return arr.ctypes.data_as(C.POINTER(ctype))


_STAT_FIELDS = (
    "n_tracks", "n_trajectory_points", "n_active_points", "n_primary_electrons", "n_deposits", "n_keys",
    "ms_h2d", "ms_tracks", "ms_deposit", "ms_finalize", "ms_d2h", "ms_total", "n_kernel_launches", "n_retries",
    "n_track_launches", "n_group_launches", "n_hash_probes", "hash_capacity", "n_table_flushes",
    "n_rk_steps", "n_rk_rejects", "max_track_passes", "ms_order", "n_big",
)  # fmt: skip


class Engine:
    """One CUDA simulator handle (one GPU, one species set)."""

    def __init__(
        self,
        config: Config,
        species: list,
        device: int = 0,
        ode_rtol: float = 1e-6,
        ode_atol: float = 1e-10,
        freeze_ke_mev: float | None = None,
        max_events_per_launch: int = 0,
        hash_capacity: int = 0,
        copy_events_per_launch: int = 0,
        unit_points: int = 0,
        table_spill_keys: int = 0,
    ):
        if config.pad_grid is None or config.pad_grid_edges is None:
            raise ValueError("Pad grid is not loaded")  # solver.py:400-401
        if config.pad_centers is None or config.pad_sizes is None:
            raise ValueError("Pad centers are not assigned")  # writer.py:220-221
        long_diffusion = float(getattr(config.det_params, "longitudinal_diffusion", 0.0))
        if not (math.isfinite(long_diffusion) and long_diffusion >= 0.0):
            raise ValueError(f"longitudinal_diffusion must be finite and >= 0, got {long_diffusion}")
        self.lib = _lib.load()
        self.config = config
        self.device = int(device)
        self.species = list(species)
        self.species_index = {(int(n.Z), int(n.A)): i for i, n in enumerate(self.species)}
        det, elec = config.det_params, config.elec_params
        target: TableGasTarget = ensure_table_target(det.gas_target)
        self.target = target
        tables = [target.table_for(n) for n in self.species]

        lut, origin = build_pad_lut(config.pad_grid, config.pad_grid_edges)
        self._lut = lut
        self._pad_xy = np.ascontiguousarray(config.pad_centers, dtype=np.float64)
        self._pad_scale = np.ascontiguousarray(config.pad_sizes, dtype=np.float64)
        self._response = np.ascontiguousarray(get_response(config), dtype=np.float64)
        self._tables = [np.ascontiguousarray(t.values, dtype=np.float64) for t in tables]

        cfg = _lib.AttpcConfig()
        cfg.length = float(det.length)
        cfg.efield = float(det.efield)
        cfg.bfield = float(det.bfield)
        cfg.mpgd_gain = int(det.mpgd_gain)
        cfg.diffusion = float(det.diffusion)
        cfg.longitudinal_diffusion = long_diffusion
        cfg.fano_factor = float(det.fano_factor)
        cfg.w_value = float(det.w_value)
        cfg.gas_density = float(target.density)
        cfg.micromegas_edge = int(elec.micromegas_edge)
        cfg.windows_edge = int(elec.windows_edge)
        cfg.adc_threshold = float(elec.adc_threshold)
        cfg.drift_velocity = float(config.drift_velocity)
        cfg.grid_low_mm = float(config.pad_grid_edges[0])
        cfg.grid_high_mm = float(config.pad_grid_edges[1])
        cfg.lut_origin_mm = origin
        cfg.lut_n = lut.shape[0]
        cfg.ode_rtol = float(ode_rtol)
        cfg.ode_atol = float(ode_atol)
        if freeze_ke_mev is None:
            freeze_ke_mev = default_freeze_ke(det.fano_factor, det.w_value)
        self.freeze_ke_mev = float(freeze_ke_mev)
        cfg.freeze_ke_mev = self.freeze_ke_mev
        cfg.max_events_per_launch = int(max_events_per_launch)
        cfg.hash_capacity = int(hash_capacity)
        cfg.copy_events_per_launch = int(copy_events_per_launch)
        cfg.unit_points = int(unit_points)
        cfg.table_spill_keys = int(table_spill_keys)

        sp = (_lib.AttpcSpecies * len(self.species))()
        for i, (nuc, tab) in enumerate(zip(self.species, tables)):
            sp[i].z = int(nuc.Z)
            sp[i].a = int(nuc.A)
            sp[i].mass = float(nuc.mass)
            sp[i].lm, sp[i].e_min, sp[i].n_oct = tab.lm, tab.e_min, tab.n_oct
            sp[i].dedx = _ptr(self._tables[i], C.c_double)
        handle = C.c_void_p()
        code = self.lib.attpc_create(
            C.byref(cfg), _ptr(lut, C.c_int16), _ptr(self._pad_xy, C.c_double), _ptr(self._pad_scale, C.c_double),
            len(self._pad_scale), _ptr(self._response, C.c_double), len(self._response), sp, len(self.species),
            self.device, C.byref(handle),
        )  # fmt: skip
        _lib.check(code, None)
        self.handle = handle

    @classmethod
    def for_conversion(cls, window_edge, mm_edge, length, response, pad_centers, pad_sizes, threshold, device=0):
        """Handle without species or pad map: only `convert_to_spyral` works on it (`writer.py:61-112`)."""
        self = cls.__new__(cls)
        self.lib = _lib.load()
        self.config = None
        self.device = int(device)
        self.species, self.species_index = [], {}
        self._lut = np.full((1, 1), -1, dtype=np.int16)
        self._pad_xy = np.ascontiguousarray(pad_centers, dtype=np.float64)
        self._pad_scale = np.ascontiguousarray(pad_sizes, dtype=np.float64)
        self._response = np.ascontiguousarray(response, dtype=np.float64)
        cfg = _lib.AttpcConfig()
        cfg.length = float(length)
        cfg.efield, cfg.bfield, cfg.mpgd_gain = 1.0, 0.0, 1
        cfg.diffusion, cfg.fano_factor, cfg.w_value, cfg.gas_density = 0.0, 0.0, 1.0, 0.0
        cfg.longitudinal_diffusion = 0.0
        cfg.micromegas_edge, cfg.windows_edge = int(mm_edge), int(window_edge)
        cfg.adc_threshold = float(threshold)
        cfg.drift_velocity = float(length) / float(int(window_edge) - int(mm_edge))
        cfg.grid_low_mm, cfg.grid_high_mm, cfg.lut_origin_mm, cfg.lut_n = 0.0, 1.0, 0, 1
        handle = C.c_void_p()
        code = self.lib.attpc_create(
            C.byref(cfg), _ptr(self._lut, C.c_int16), _ptr(self._pad_xy, C.c_double),
            _ptr(self._pad_scale, C.c_double), len(self._pad_scale), _ptr(self._response, C.c_double),
            len(self._response), None, 0, self.device, C.byref(handle),
        )  # fmt: skip
        _lib.check(code, None)
        self.handle = handle
        return self

    # ------------------------------------------------------------------------------ lifecycle
    def close(self) -> None:
        if getattr(self, "handle", None):
            self.lib.attpc_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -------------------------------------------------------------------------------- helpers
    def _species_of(self, proton_numbers, mass_numbers, indices) -> tuple[np.ndarray, np.ndarray]:
        nucleus = np.asarray(indices, dtype=np.int32)
        spec = np.empty(len(nucleus), dtype=np.int32)
        for t, idx in enumerate(nucleus):
            z, a = int(proton_numbers[idx]), int(mass_numbers[idx])
            if z == 0:
                spec[t] = -1  # simulator.py:97
            else:
                spec[t] = self.species_index[(z, a)]
        return np.ascontiguousarray(nucleus), spec

    def _collect(self, res: _lib.AttpcResult, first_event: int, copy: bool, rows: bool, track_labels=()) -> SimBatch:
        n_ev, n_pts = int(res.n_events), int(res.n_points)
        stats = {k: getattr(res, k) for k in _STAT_FIELDS}
        if not res.offsets:  # SKIP_HOST_COPY: the rows stay on the device (`read_device_result` fetches them)
            out = SimBatch(first_event, np.zeros(n_ev + 1, np.int64), np.zeros((0, 3)), np.zeros(0, np.int64),
                           stats=dict(stats, n_points=n_pts))  # fmt: skip
            out.device = dict(offsets=res.offsets_dev, cloud=res.cloud_dev, labels=res.labels_dev, n_events=n_ev, n_points=n_pts)
            return out
        grab = (lambda a: a.copy()) if copy else (lambda a: a)
        offsets = grab(np.ctypeslib.as_array(res.offsets, shape=(n_ev + 1,)))
        columns = packed = None
        if res.col_pad:
            take = (lambda p: grab(np.ctypeslib.as_array(p, shape=(n_pts,)))) if n_pts > 0 else None
            if res.col_wiggle:  # ATTPC_COLUMNS_PACKED
                labels_of_rank = np.zeros(4, dtype=np.int8)
                labels_of_rank[: len(track_labels)] = track_labels
                columns = packed = dict(
                    pad_rank=take(res.col_pad).view(np.uint16) if take else np.zeros(0, np.uint16),
                    wiggle=take(res.col_wiggle) if take else np.zeros(0, np.uint16),
                    tb_counts=grab(np.ctypeslib.as_array(res.tb_counts, shape=(n_ev, NUM_TB))) if n_ev else np.zeros((0, NUM_TB), np.uint16),
                    labels_of_rank=labels_of_rank, rank_shift=int(res.pad_rank_shift),
                )  # fmt: skip
            else:
                columns = dict(
                    pad=take(res.col_pad) if take else np.zeros(0, np.int16),
                    tb_q16=take(res.col_tb_q16) if take else np.zeros(0, np.uint32),
                    label8=take(res.col_label) if take else np.zeros(0, np.int8),
                )
            if res.col_electrons32:  # compact: low 32 bits + the (row, count) pairs of the counts that need more
                n_big = int(res.n_big)
                rows_big = np.ctypeslib.as_array(res.big_rows, shape=(n_big,)).copy() if n_big else np.zeros(0, np.int64)
                vals_big = np.ctypeslib.as_array(res.big_electrons, shape=(n_big,)).copy() if n_big else np.zeros(0, np.int64)
                order = np.argsort(rows_big, kind="stable")
                columns.update(electrons_u32=take(res.col_electrons32) if take else np.zeros(0, np.uint32),
                               big_rows=rows_big[order], big_electrons=vals_big[order])
            else:
                columns["electrons"] = take(res.col_electrons) if take else np.zeros(0, np.int64)
            cloud = labels = None
        elif n_pts > 0 and res.cloud:
            cloud = grab(np.ctypeslib.as_array(res.cloud, shape=(n_pts, 3)))
            labels = grab(np.ctypeslib.as_array(res.labels, shape=(n_pts,)))
        else:
            cloud, labels = np.zeros((0, 3)), np.zeros(0, np.int64)
        out = SimBatch(first_event, offsets, cloud, labels, stats=dict(stats, n_points=n_pts, packed=int(packed is not None)),
                       columns=None if packed is not None else columns, packed=packed)
        if rows and res.row_col_pad:
            n_rows = int(res.n_rows)
            out.row_offsets = grab(np.ctypeslib.as_array(res.row_offsets, shape=(n_ev + 1,)))
            names = (("pad", res.row_col_pad, np.int16), ("tb_q16", res.row_col_tb_q16, np.uint32),
                     ("e_lo", res.row_col_e_lo, np.uint32), ("e_hi", res.row_col_e_hi, np.uint16),
                     ("label8", res.row_col_label, np.int8))  # fmt: skip
            out.row_columns = {k: (grab(np.ctypeslib.as_array(ptr, shape=(n_rows,))) if n_rows else np.zeros(0, dt))
                               for k, ptr, dt in names}  # fmt: skip
            out._row_builder = self.rows_from_columns
            out.stats["n_rows"] = n_rows
        elif rows:
            n_rows = int(res.n_rows)
            out.row_offsets = grab(np.ctypeslib.as_array(res.row_offsets, shape=(n_ev + 1,)))
            if n_rows > 0:
                out.rows = grab(np.ctypeslib.as_array(res.rows, shape=(n_rows, 8)))
                out.row_labels = grab(np.ctypeslib.as_array(res.row_labels, shape=(n_rows,)))
            else:
                out.rows, out.row_labels = np.zeros((0, 8)), np.zeros(0, np.int64)
            out.stats["n_rows"] = n_rows
        return out

    def read_device_result(self, batch: SimBatch) -> SimBatch:
        """The rows of a device-resident call (`host_copy=False`), copied to fresh host arrays.  Valid until the next
        call on this engine reuses the device buffers."""
        dev = batch.device
        n_ev, n_pts = dev["n_events"], dev["n_points"]
        offsets = np.empty(n_ev + 1, dtype=np.int64)
        cloud = np.empty((n_pts, 3), dtype=np.float64)
        labels = np.empty(n_pts, dtype=np.int64)
        for arr, ptr in ((offsets, dev["offsets"]), (cloud, dev["cloud"]), (labels, dev["labels"])):
            if arr.nbytes:
                _lib.check(self.lib.attpc_read_device(self.handle, ptr, arr.ctypes.data_as(C.c_void_p), arr.nbytes), self.handle)
        return SimBatch(batch.first_event, offsets, cloud, labels, stats=dict(batch.stats))

    def rows_from_columns(self, cols: dict) -> tuple[np.ndarray, np.ndarray]:
        """The eight Spyral columns (`writer.py:61-112`) from the typed columns of ``ATTPC_SPYRAL_COLUMNS``.

        Every column is a function of (pad, time bucket, electrons): x, y, pad size are table lookups, z is
        `writer.py:101-103`, amplitude and integral are `response.py:35-57` in the closed form the device uses
        (``min(r_max e, 4095)`` and ``4095 k + e (S - S_k)`` over the descending-sorted response, with explicitly
        rounded operations on both sides), so the result equals the device's float64 rows bit for bit
        (`tests/test_gpu_e2e.py::test_spyral_columns_rebuild_the_float64_rows`).
        """
        if not hasattr(self, "_resp_sorted"):
            self._resp_sorted = np.sort(self._response)[::-1].copy()
            self._resp_prefix = np.concatenate([[0.0], np.cumsum(self._resp_sorted)])  # sequential, like the device's
        cfg = self.config
        win, mm = float(int(cfg.elec_params.windows_edge)), float(int(cfg.elec_params.micromegas_edge))
        length = float(cfg.det_params.length)
        pad = cols["pad"].astype(np.int64)
        n = len(pad)
        e = ((cols["e_hi"].astype(np.uint64) << np.uint64(32)) | cols["e_lo"].astype(np.uint64)).astype(np.float64)
        tbf = cols["tb_q16"].astype(np.float64)
        tbf *= 1.0 / 65536.0
        rows = np.empty((n, 8), dtype=np.float64)
        rows[:, 0] = self._pad_xy[pad, 0]
        rows[:, 1] = self._pad_xy[pad, 1]
        rows[:, 2] = (win - tbf) / (win - mm) * length * 1000.0
        rs, pre = self._resp_sorted, self._resp_prefix
        top = rs[0] * e
        rows[:, 3] = np.minimum(top, 4095.0)
        k = np.zeros(n, dtype=np.int64)  # response samples clipped at 4095: a prefix of the sorted response
        hot = np.flatnonzero(top > 4095.0)
        if len(hot):
            eh = e[hot]
            kk = np.searchsorted(-rs, -(4095.0 / eh), side="left")
            for _ in range(4):  # settle the boundary with the device's own predicate r_i * e > 4095
                down = (kk > 0) & (rs[np.maximum(kk - 1, 0)] * eh <= 4095.0)
                kk = kk - down
                up = (kk < len(rs)) & (rs[np.minimum(kk, len(rs) - 1)] * eh > 4095.0)
                kk = kk + up
            k[hot] = kk
        rows[:, 4] = 4095.0 * k + e * (pre[len(rs)] - pre[k])
        rows[:, 5] = pad
        rows[:, 6] = tbf
        rows[:, 7] = self._pad_scale[pad]
        return rows, cols["label8"].astype(np.int64)

    #: validation switch: evaluate every mesh pixel with the reference's own expression (`transporter.py:36-41`)
    #: instead of the constant weight table + exactness guard.  Both give identical results.
    exact_mesh = False

    def _mesh_flag(self) -> int:
        return _lib.EXACT_MESH if self.exact_mesh else 0

    # ------------------------------------------------------------------------------ hot path
    def simulate_batch(
        self,
        momenta: np.ndarray,
        vertices: np.ndarray,
        proton_numbers,
        mass_numbers,
        indices,
        seed: int = 0,
        first_event: int = 0,
        spyral_rows: bool = False,
        keep_all_tb: bool = False,
        copy: bool = True,
        host_copy: bool = True,
        rows_only: bool = False,
        columns: bool = False,
        row_columns: bool = False,
        packed: bool = True,
    ) -> SimBatch:
        """`simulate` (`simulator.py:52-115`) for ``B`` events at once: ``momenta [B, K, 4]``, ``vertices [B, 3]``.

        ``rows_only`` (with ``spyral_rows``): bring back offsets and Spyral rows but leave the raw cloud on the GPU.
        ``columns``: bring the rows back as typed columns (11 B/row instead of 32 B/row over PCIe), see `SimBatch`.
        ``row_columns`` (with ``spyral_rows``): the Spyral rows as typed columns too (13 instead of 72 B/row).
        ``packed`` (with ``columns``, default): let the library pack the columns further when it can (8 B/row + 1 KB/event,
        `SimBatch.packed`); ``batch.columns`` decodes them on first use.
        """
        momenta = np.ascontiguousarray(momenta, dtype=np.float64)
        vertices = np.ascontiguousarray(vertices, dtype=np.float64)
        if momenta.ndim != 3 or momenta.shape[2] != 4:
            raise ValueError("momenta must have shape [n_events, n_nuclei, 4]")
        if vertices.shape != (momenta.shape[0], 3):
            raise ValueError("vertices must have shape [n_events, 3]")
        nucleus, spec = self._species_of(proton_numbers, mass_numbers, indices)
        flags = (_lib.SPYRAL_ROWS if spyral_rows else 0) | (_lib.KEEP_ALL_TB if keep_all_tb else 0)
        if spyral_rows and row_columns:
            flags |= _lib.SPYRAL_COLUMNS
        if not host_copy:
            flags |= _lib.SKIP_HOST_COPY
        if rows_only and spyral_rows:
            flags |= _lib.SKIP_CLOUD_COPY
        elif columns:
            flags |= _lib.COLUMNS | _lib.COLUMNS32 | (_lib.COLUMNS_PACKED if packed else 0)
        flags |= self._mesh_flag()
        res = _lib.AttpcResult()
        code = self.lib.attpc_simulate(
            self.handle, _ptr(momenta, C.c_double), _ptr(vertices, C.c_double), momenta.shape[0], momenta.shape[1],
            _ptr(nucleus, C.c_int32), _ptr(spec, C.c_int32), len(nucleus), int(seed) & (2**64 - 1), int(first_event),
            flags, C.byref(res),
        )  # fmt: skip
        _lib.check(code, self.handle)
        return self._collect(res, first_event, copy, spyral_rows, track_labels=nucleus)

    def simulate_device(
        self, momenta_ptr: int, vertices_ptr: int, n_events: int, n_nuclei: int, proton_numbers, mass_numbers,
        indices, seed: int = 0, first_event: int = 0, host_copy: bool = False, spyral_rows: bool = False,
    ) -> SimBatch:  # fmt: skip
        """Same with inputs already resident in device memory (raw CUDA pointers, e.g. ``tensor.data_ptr()``)."""
        nucleus, spec = self._species_of(proton_numbers, mass_numbers, indices)
        flags = (0 if host_copy else _lib.SKIP_HOST_COPY) | (_lib.SPYRAL_ROWS if spyral_rows else 0)
        flags |= self._mesh_flag()
        res = _lib.AttpcResult()
        code = self.lib.attpc_simulate_dev(
            self.handle, C.c_void_p(momenta_ptr), C.c_void_p(vertices_ptr), int(n_events), int(n_nuclei),
            _ptr(nucleus, C.c_int32), _ptr(spec, C.c_int32), len(nucleus), int(seed) & (2**64 - 1), int(first_event),
            flags, C.byref(res),
        )  # fmt: skip
        _lib.check(code, self.handle)
        return self._collect(res, first_event, False, spyral_rows and host_copy)

    # ------------------------------------------------------------------ parity / staged entries
    def simulate_replay(
        self,
        tracks: list[np.ndarray],
        normals: list[np.ndarray],
        track_event,
        track_rank,
        track_label,
        track_za: list[tuple[int, int]],
        n_events: int,
        uniforms: list[tuple[np.ndarray, np.ndarray]] | None = None,
        keep_all_tb: bool = False,
        no_wiggle: bool = False,
        spyral_rows: bool = False,
    ) -> tuple[SimBatch, list[np.ndarray]]:
        """Everything after the trajectory from given rows and random numbers (parity part (a)).

        ``uniforms[e] = (keys, u)`` replays `simulator.py:108` keyed by Szudzik id.
        Returns the batch and, per track, ``electrons`` as `solver.py:343-346` would.
        """
        n_tracks = len(tracks)
        lens = np.array([len(t) for t in tracks], dtype=np.int64)
        offsets = np.zeros(n_tracks + 1, dtype=np.int64)
        np.cumsum(lens, out=offsets[1:])
        rows = np.ascontiguousarray(np.concatenate(tracks) if n_tracks else np.zeros((0, 6)), dtype=np.float64)
        zn = np.ascontiguousarray(np.concatenate(normals) if n_tracks else np.zeros(0), dtype=np.float64)
        if len(zn) != len(rows):
            raise ValueError("one standard normal per trajectory row is required")
        ev = np.ascontiguousarray(track_event, dtype=np.int32)
        rk = np.ascontiguousarray(track_rank, dtype=np.int32)
        lb = np.ascontiguousarray(track_label, dtype=np.int32)
        sp = np.array([-1 if z == 0 else self.species_index[(int(z), int(a))] for z, a in track_za], dtype=np.int32)
        electrons = np.zeros(max(1, len(rows)), dtype=np.int64)
        replay = None
        keep = []
        if uniforms is not None:
            u_off = np.zeros(n_events + 1, dtype=np.int64)
            ks, us = [], []
            for e in range(n_events):
                k, u = uniforms[e]
                order = np.argsort(np.asarray(k, dtype=np.int64), kind="stable")
                ks.append(np.asarray(k, dtype=np.int64)[order])
                us.append(np.asarray(u, dtype=np.float64)[order])
                u_off[e + 1] = u_off[e] + len(order)
            u_keys = np.ascontiguousarray(np.concatenate(ks) if ks else np.zeros(0, np.int64))
            u_vals = np.ascontiguousarray(np.concatenate(us) if us else np.zeros(0))
            keep = [u_off, u_keys, u_vals]
            replay = _lib.AttpcReplay(_ptr(u_off, C.c_int64), _ptr(u_keys, C.c_int64), _ptr(u_vals, C.c_double))
        flags = (
            (_lib.KEEP_ALL_TB if keep_all_tb else 0)
            | (_lib.NO_WIGGLE if no_wiggle else 0)
            | (_lib.SPYRAL_ROWS if spyral_rows else 0)
            | self._mesh_flag()
        )
        res = _lib.AttpcResult()
        code = self.lib.attpc_simulate_replay(
            self.handle, _ptr(offsets, C.c_int64), _ptr(rows, C.c_double), _ptr(zn, C.c_double), _ptr(ev, C.c_int32),
            _ptr(rk, C.c_int32), _ptr(lb, C.c_int32), _ptr(sp, C.c_int32), n_tracks, int(n_events),
            C.byref(replay) if replay is not None else None, flags, _ptr(electrons, C.c_int64), C.byref(res),
        )  # fmt: skip
        _lib.check(code, self.handle)
        del keep
        batch = self._collect(res, 0, True, spyral_rows)
        per_track = [electrons[offsets[t] : offsets[t + 1]].copy() for t in range(n_tracks)]
        return batch, per_track

    def trajectories(self, momenta, vertices, nuclei, stride: int = 1, max_points: int = 10001):
        """`generate_trajectory` (`solver.py:243-305`) for a list of tracks; returns (points, counts)."""
        momenta = np.ascontiguousarray(momenta, dtype=np.float64).reshape(-1, 4)
        vertices = np.ascontiguousarray(vertices, dtype=np.float64).reshape(-1, 3)
        n = len(momenta)
        sp = np.array([self.species_index[(int(nu.Z), int(nu.A))] for nu in nuclei], dtype=np.int32)
        out = np.zeros((n, max_points, 6), dtype=np.float64)
        counts = np.zeros(n, dtype=np.int32)
        code = self.lib.attpc_trajectories(
            self.handle, _ptr(momenta, C.c_double), _ptr(vertices, C.c_double), _ptr(sp, C.c_int32), n, int(stride),
            int(max_points), _ptr(out, C.c_double), _ptr(counts, C.c_int32),
        )  # fmt: skip
        _lib.check(code, self.handle)
        return out, counts

    def convert_to_spyral(self, offsets, cloud, labels, keep_all: bool = False) -> SimBatch:
        """`convert_to_spyral` + threshold + z-sort (`writer.py:61-112, 232-238`) for CSR clouds.

        ``keep_all=True`` is the bare `convert_to_spyral`: every row, input order.
        """
        offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        cloud = np.ascontiguousarray(cloud, dtype=np.float64).reshape(-1, 3)
        labels = np.ascontiguousarray(labels, dtype=np.int64)
        res = _lib.AttpcResult()
        code = self.lib.attpc_convert_to_spyral(
            self.handle, _ptr(offsets, C.c_int64), _ptr(cloud, C.c_double), _ptr(labels, C.c_int64), len(offsets) - 1,
            _lib.ROWS_KEEP_ALL if keep_all else 0, C.byref(res),
        )  # fmt: skip
        _lib.check(code, self.handle)
        n_ev, n_rows = len(offsets) - 1, int(res.n_rows)
        out = SimBatch(0, offsets, cloud, labels)
        out.row_offsets = np.ctypeslib.as_array(res.row_offsets, shape=(n_ev + 1,)).copy()
        if n_rows:
            out.rows = np.ctypeslib.as_array(res.rows, shape=(n_rows, 8)).copy()
            out.row_labels = np.ctypeslib.as_array(res.row_labels, shape=(n_rows,)).copy()
        else:
            out.rows, out.row_labels = np.zeros((0, 8)), np.zeros(0, np.int64)
        return out

    def lookup_pads(self, xy: np.ndarray) -> np.ndarray:
        """`position_to_index` + grid read + beam veto (`transporter.py:78-120, 165`) for ``xy [n, 2]`` in m."""
        xy = np.ascontiguousarray(xy, dtype=np.float64).reshape(-1, 2)
        out = np.empty(len(xy), dtype=np.int32)
        _lib.check(self.lib.attpc_lookup_pads(self.handle, _ptr(xy, C.c_double), len(xy), _ptr(out, C.c_int32)),
                   self.handle)  # fmt: skip
        return out


def _digest(*arrays) -> str:
    import hashlib

    h = hashlib.blake2b(digest_size=16)
    for a in arrays:
        a = np.ascontiguousarray(a)
        h.update(str(a.dtype).encode() + str(a.shape).encode())
        h.update(a.tobytes())
    return h.hexdigest()


def config_fingerprint(config: Config, nuclei: list) -> tuple:
    """Everything `Engine.__init__` bakes into device constants, as a hashable value.

    The reference reads ``config.*`` afresh for every event, so a user may mutate the parameter dataclasses between
    calls (a scan over ``det_params.bfield``, another ``load_pad_grid``, another gas).  `engine_for` compares this
    fingerprint on every call and rebuilds the engine when anything baked has changed.  The dE/dx tables are
    fingerprinted through the target object's identity plus its density and a probe of ``get_dedx`` per species
    (cheap; re-tabulating on every call would not be).
    """
    det, elec = config.det_params, config.elec_params
    scalars = (
        float(det.length), float(det.efield), float(det.bfield), int(det.mpgd_gain), float(det.diffusion),
        float(det.fano_factor), float(det.w_value), float(elec.clock_freq), float(elec.amp_gain),
        float(elec.shaping_time), int(elec.micromegas_edge), int(elec.windows_edge), float(elec.adc_threshold),
        float(config.drift_velocity), float(getattr(det, "longitudinal_diffusion", 0.0)),
    )  # fmt: skip
    target = det.gas_target
    probes = tuple(
        (int(n.Z), int(n.A), float(n.mass), float(target.get_dedx(n, 0.37 * n.A)), float(target.get_dedx(n, 9.1 * n.A)))
        for n in nuclei
    )
    arrays = getattr(config, "_b200_array_digest", None)
    ids = (id(config.pad_grid), id(config.pad_grid_edges), id(config.pad_centers), id(config.pad_sizes))
    if arrays is None or arrays[0] != ids:  # hashing 31 M grid cells takes ~20 ms: only when the arrays were replaced
        arrays = (ids, _digest(config.pad_grid_edges, config.pad_centers, config.pad_sizes,
                               np.asarray(config.pad_grid)[::10, ::10]))  # fmt: skip
        config.__dict__["_b200_array_digest"] = arrays
    return scalars + (id(target), float(target.density), probes, arrays[1])


def engine_for(config: Config, nuclei: list, device: int = 0, instance: int = 0, **tuning) -> Engine:
    """Engine cached on the Config object, keyed by device, species set and tuning; rebuilt when a baked value changed.

    A handle must not be used from two threads at once: concurrent callers on the SAME device ask for different
    ``instance`` numbers.  (In-place edits of the pad arrays are not seen -- replace the array, as ``load_pad_grid`` does.)
    """
    cache = config.__dict__.setdefault("_b200_engines", {})
    key = (int(device), int(instance), tuple(sorted((int(n.Z), int(n.A)) for n in nuclei)), tuple(sorted(tuning.items())))
    uniq = {}
    for n in nuclei:
        uniq.setdefault((int(n.Z), int(n.A)), n)
    species = [uniq[k] for k in sorted(uniq)]
    stamp = config_fingerprint(config, species)
    hit = cache.get(key)
    if hit is not None and hit[0] == stamp:
        return hit[1]
    if hit is not None:
        hit[1].close()  # stale constants: free the device memory before building the replacement
    eng = Engine(config, species, device=device, **tuning)
    cache[key] = (stamp, eng)
    return eng


__all__ = ["Engine", "SimBatch", "engine_for", "config_fingerprint", "build_pad_lut", "default_freeze_ke", "NUM_TB"]
