#!/usr/bin/env python
"""Throughput benchmark of the detector-simulation hot path (see the task contract in DESIGN.md section "Measurement").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--events B]
                    [--dump-outputs DIR]

A *step* is one pass of the whole hot path (`simulate` of detector/simulator.py:52-115 for every event) over one
batch of B synthetic kinematics events per GPU.  Prints ONE JSON line (rank 0).  The inputs depend on the arguments
alone, so `--dump-outputs` of two builds can be compared array for array (see `dump_arrays`).

* value      events/s with the inputs resident in HBM and the results left in HBM (device time, CUDA events
             recorded by the library on its own stream, max over ranks; L2 flushed between steps).
* e2e        the same metric through the public Python API `simulate_stream` (the pipelined `simulate_batch` that
             `run_simulation` is built on, `--e2e-engines` engines per GPU): pinned HOST inputs copied in and the full
             point clouds copied back to pinned HOST memory every step, as packed typed columns (8 B/row + 1 KB per
             event, lossless).  e2e_sync: one synchronous `simulate_batch` call per step.  e2e_float64: the pipelined
             call returning the reference's own float64 / int64 arrays (32 B/row).  e2e_decoded: one step plus the
             numpy decode of the columns on one host thread.
* roofline   dominant kernel (by device time): its issue-slot roofline (warp instructions per launch from the committed
             ncu capture over the launch time measured live, against SMs x 4 schedulers x clock), the HBM fraction of
             the whole step (algorithmic bytes of SURVEY.md 8(d) against the measured copy peak) beside it, and the
             kernel's DRAM traffic from the same capture (profiles/traffic.json).
* cpu_baseline / --impl reference
             the CPU oracle port of the reference (oracle/attpc_oracle.py: scipy Radau + numba, the reference's
             own tool chain) on all host cores, on a bounded sample of the same events.
"""

from __future__ import annotations

import argparse
import atexit
import json
import os
import shutil
import statistics
import subprocess
import sys
import tempfile
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.dont_write_bytecode = True  # the benchmark writes nothing into the tree it runs from (which may be read-only)

WORKLOADS = {
    # name: (description, gas, (target, projectile, ejectile), decays [(parent, residual_1)], excitations, beam MeV)
    "c16dd": dict(
        desc="16C(d,d')16C g.s., 184.131 MeV 16C (11.5 MeV/u) on D2 600 Torr, B=3 T, E=45 kV/m; tracks [2,3]",
        gas=([(1, 2, 2)], 600.0), reaction=((1, 2), (6, 16), (1, 2)), decays=[], excitations=[("gauss", 0.0, 0.001)],
        beam=184.131, config_id=1,
    ),
    "c16dd_sweep": dict(
        desc="16C(d,d')16C*, excitation energy swept uniformly over 0-10 MeV (BASELINE config 5), 184.131 MeV 16C on D2 "
             "600 Torr, B=3 T; tracks [2,3]",
        gas=([(1, 2, 2)], 600.0), reaction=((1, 2), (6, 16), (1, 2)), decays=[], excitations=[("uniform", 0.0, 10.0)],
        beam=184.131, config_id=5,
    ),
    "c14dp": dict(
        desc="14C(d,p)15C* -> 14C + n, 161 MeV 14C on D2 600 Torr, B=3 T; tracks [2,4,5] (neutron skipped)",
        gas=([(1, 2, 2)], 600.0), reaction=((1, 2), (6, 14), (1, 1)), decays=[((6, 15), (6, 14))],
        excitations=[("gauss", 3.1, 0.04), ("gauss", 0.0, 0.0)], beam=161.0, config_id=2,
    ),
    "c12aa": dict(
        desc="12C(a,a')12C*(7.654) -> a + 8Be -> 3a, 96 MeV 12C on 4He 600 Torr, B=3 T; tracks [2,4,6,7]",
        gas=([(2, 4, 1)], 600.0), reaction=((2, 4), (6, 12), (2, 4)), decays=[((6, 12), (2, 4)), ((4, 8), (2, 4))],
        excitations=[("gauss", 7.654, 0.0), ("gauss", 0.0, 0.0), ("gauss", 0.0, 0.0)], beam=96.0, config_id=3,
    ),
    "sn132dp": dict(
        desc="132Sn(d,p)133Sn, 1320 MeV 132Sn (10 MeV/u) on D2 600 Torr, B=3 T; tracks [2,3]",
        gas=([(1, 2, 2)], 600.0), reaction=((1, 2), (50, 132), (1, 1)), decays=[], excitations=[("gauss", 0.0, 0.001)],
        beam=1320.0, config_id=4,
    ),
}  # fmt: skip


def make_pipeline(name: str):
    """The vectorised kinematics pipeline of a named reaction and its gas (SURVEY.md 8(d), 8f-1)."""
    from attpc_engine_b200 import nuclear_map as nm
    from attpc_engine_b200.kinematics import (
        Decay, ExcitationGaussian, ExcitationUniform, KinematicsPipeline, KinematicsTargetMaterial, PolarUniform, Reaction,
    )  # fmt: skip
    from attpc_engine_b200.target import AnalyticGasTarget, TableGasTarget

    w = WORKLOADS[name]
    gas = TableGasTarget(AnalyticGasTarget(*w["gas"]))
    t, p, e = (nm.get_data(*za) for za in w["reaction"])
    steps = [Reaction(target=t, projectile=p, ejectile=e)]
    steps += [Decay(parent=nm.get_data(*a), residual_1=nm.get_data(*b)) for a, b in w["decays"]]
    pipeline = KinematicsPipeline(
        steps, [ExcitationUniform(a, b) if kind == "uniform" else ExcitationGaussian(a, b) for kind, a, b in w["excitations"]],
        [PolarUniform(0.0, np.pi)] * len(steps),
        beam_energy=w["beam"], target_material=KinematicsTargetMaterial(gas, (0.0, 1.0), 0.007),
    )  # fmt: skip
    return pipeline, gas


def workload_seed(name: str, seed_offset: int = 0) -> int:
    return 20260101 + WORKLOADS[name]["config_id"] + 7919 * seed_offset


def build_workload(name: str, n_events: int, seed_offset: int = 0):
    """Synthetic kinematics of a named reaction + the detector Config (SURVEY.md 8(d))."""
    from attpc_engine_b200.detector import Config, DetectorParams, ElectronicsParams, PadParams
    from attpc_engine_b200.detector.simulator import default_indices

    pipeline, gas = make_pipeline(name)
    pipeline.seed(workload_seed(name, seed_offset))
    vertices, momenta = pipeline.run_batch(n_events)
    det = DetectorParams(length=1.0, efield=45000.0, bfield=3.0, mpgd_gain=175000, gas_target=gas, diffusion=0.277,
                         fano_factor=0.2, w_value=34.0)  # fmt: skip
    elec = ElectronicsParams(clock_freq=6.25, amp_gain=900, shaping_time=1000, micromegas_edge=10, windows_edge=560,
                             adc_threshold=40)  # fmt: skip
    config = Config(det, elec, PadParams())
    zs, as_ = pipeline.get_proton_numbers(), pipeline.get_mass_numbers()
    return config, momenta, vertices, zs, as_, default_indices(len(zs))


# ----------------------------------------------------------------------------------------------- CPU (oracle) arm
_CPU = {}


def _cpu_init(name):
    from attpc_engine_b200 import nuclear_map
    from oracle import attpc_oracle as oracle

    config, momenta, vertices, zs, as_, indices = build_workload(name, 4)
    _CPU.update(config=config, zs=zs, as_=as_, indices=indices, oracle=oracle, nmap=nuclear_map)
    oracle.simulate_event(momenta[0], vertices[0], zs, as_, config, np.random.default_rng(0), indices, nuclear_map)


def _cpu_chunk(args):
    momenta, vertices, first = args
    c = _CPU
    rec = {}
    points = electrons = 0
    t0 = time.perf_counter()
    for i in range(len(momenta)):
        cloud, _ = c["oracle"].simulate_event(
            momenta[i], vertices[i], c["zs"], c["as_"], c["config"], np.random.default_rng(first + i), c["indices"],
            c["nmap"], record=rec,
        )  # fmt: skip
        points += len(cloud)
        electrons += rec["stats"]["primary_electrons"]
    return len(momenta), points, electrons, time.perf_counter() - t0


class CpuArm:
    """The oracle port on all host cores (multiprocessing over disjoint event ranges)."""

    def __init__(self, name, cores=None):
        import multiprocessing as mp

        self.cores = cores or len(os.sched_getaffinity(0))
        self.pool = mp.get_context("spawn").Pool(self.cores, initializer=_cpu_init, initargs=(name,))

    def run(self, momenta, vertices, first=0):
        n = len(momenta)
        per = max(1, -(-n // self.cores))
        jobs = [(momenta[a : a + per], vertices[a : a + per], first + a) for a in range(0, n, per)]
        t0 = time.perf_counter()
        out = self.pool.map(_cpu_chunk, jobs)
        wall = time.perf_counter() - t0
        return dict(events=sum(o[0] for o in out), points=sum(o[1] for o in out), electrons=sum(o[2] for o in out),
                    wall_s=wall, core_s=sum(o[3] for o in out))  # fmt: skip

    def close(self):
        self.pool.close()
        self.pool.join()


# ------------------------------------------------------------------------------------------------------ helpers
class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")  # fmt: skip

    def __init__(self, device):
        self.device, self.proc = device, None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits", "-lms", "100", "-i",
                 str(self.device)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True,
            )  # fmt: skip
        except OSError:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
            out, _ = self.proc.communicate()
        sm, smax, reasons = [], [], set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "samples": len(sm), "reasons": sorted(reasons)}  # fmt: skip


def measured_peak_hbm():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def dist_setup(n_gpus):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist

        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    return rank, world, local, dist


def reduce_max(dist, value, device):
    if dist is None:
        return value
    import torch

    t = torch.tensor([value], dtype=torch.float64, device=f"cuda:{device}")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def reduce_sum(dist, value, device):
    if dist is None:
        return value
    import torch

    t = torch.tensor([value], dtype=torch.float64, device=f"cuda:{device}")
    dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return float(t.item())


DUMP_EVENTS = 128  # events whose rows --dump-outputs keeps: ~49 MB at the ~12k points per event of c12aa
DUMP_BYTES = 64_000_000


def dump_arrays(batch, seed=0):
    """What a caller of the device-resident call gets back (`Engine.read_device_result`: CSR offsets, cloud float64
    [N, 3], labels int64 [N]), cut to at most DUMP_BYTES as float64 arrays: the point count of every event, and the
    cloud rows and labels of a fixed, seeded sample of events (`sample_events`, ascending; its tail is dropped should
    the rows outgrow the budget)."""
    offsets = batch.offsets
    counts = np.diff(offsets)
    sample = np.sort(np.random.default_rng(seed).choice(len(counts), size=min(len(counts), DUMP_EVENTS), replace=False))
    row_budget = (DUMP_BYTES - 8 * (len(counts) + len(sample)) - 4 * 128) // 32  # 3 cloud columns + label, 8 B each
    sample = sample[np.cumsum(counts[sample]) <= row_budget]
    rows = np.concatenate([np.arange(offsets[e], offsets[e + 1]) for e in sample] + [np.zeros(0, np.int64)])
    return {"points_per_event": counts, "sample_events": sample, "cloud": batch.cloud[rows], "labels": batch.labels[rows]}


def write_dump(directory, arrays):
    out = Path(directory)
    out.mkdir(parents=True, exist_ok=True)
    for name, a in arrays.items():
        np.save(out / f"{name}.npy", np.asarray(a, dtype=np.float64))


# ------------------------------------------------------------------------------------------------------- arms
def run_ours(args):
    import torch

    from attpc_engine_b200.detector.engine import engine_for
    from attpc_engine_b200.detector.simulator import _nuclei_for
    from attpc_engine_b200 import nuclear_map

    local_env = int(os.environ.get("LOCAL_RANK", "0"))
    numa_cpus = None
    if int(os.environ.get("WORLD_SIZE", "1")) > 1 and not args.no_numa:
        from attpc_engine_b200.detector.sharding import bind_to_gpu_numa_node

        numa_cpus = bind_to_gpu_numa_node(local_env)  # before CUDA starts: pinned buffers land next to the GPU
    rank, world, local, dist = dist_setup(args.gpus)
    torch.cuda.set_device(local)
    B = args.events
    config, momenta, vertices, zs, as_, indices = build_workload(args.workload, B, seed_offset=rank)
    K = momenta.shape[1]
    tuning = dict(max_events_per_launch=args.launch_events, copy_events_per_launch=args.copy_events,
                  **{k: int(v) for k, v in (kv.split("=") for kv in args.tune)})  # fmt: skip
    eng = engine_for(config, _nuclei_for(zs, as_, indices, nuclear_map), device=local, **tuning)
    # pinned host inputs (e2e) and device-resident inputs (value)
    mom_pin = torch.from_numpy(momenta).pin_memory()
    vtx_pin = torch.from_numpy(vertices).pin_memory()
    mom_dev = mom_pin.to(f"cuda:{local}")
    vtx_dev = vtx_pin.to(f"cuda:{local}")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=f"cuda:{local}")
    seed = 20260101
    first = rank * B  # this rank's event range: [rank*B, (rank+1)*B)

    def flush_l2():
        flush.zero_()
        torch.cuda.synchronize()

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()

    def step_device(i):
        return eng.simulate_device(mom_dev.data_ptr(), vtx_dev.data_ptr(), B, K, zs, as_, indices, seed=seed + i,
                                   first_event=first, spyral_rows=args.spyral)  # fmt: skip

    def batch_e2e(i):
        return eng.simulate_batch(mom_pin.numpy(), vtx_pin.numpy(), zs, as_, indices, seed=seed + i, first_event=first,
                                  copy=False, spyral_rows=args.spyral, rows_only=args.spyral,
                                  row_columns=args.spyral and not args.float64_rows,
                                  columns=not args.float64_rows)  # fmt: skip

    e2e_packed = False

    def step_e2e(i):
        nonlocal e2e_packed
        st = batch_e2e(i).stats
        e2e_packed = bool(st.get("packed", 0))
        return st

    def stream_e2e(n_steps, step0, float64_rows=args.float64_rows, engines=None):
        """n_steps batches through `simulate_stream` (the pipelined public call that `run_simulation` uses): engines
        alternate on this GPU, the copy of one batch to the host overlaps the kernels of the next.  Every batch is
        this rank's B events under fresh global event numbers (fresh random streams)."""
        from attpc_engine_b200.detector import simulate_stream

        batches = [(mom_pin.numpy(), vtx_pin.numpy(), (step0 + k) * world * B + first) for k in range(n_steps)]
        pts = rows = big = 0
        was_packed = False
        for _, b in simulate_stream(batches, zs, as_, config, seed, indices, devices=[local],
                                    engines_per_device=engines or args.e2e_engines, copy=False, spyral_rows=args.spyral,
                                    rows_only=args.spyral, row_columns=args.spyral and not float64_rows,
                                    columns=not float64_rows, **tuning):  # fmt: skip
            pts += b.stats["n_points"]
            big += b.stats.get("n_big", 0)
            rows += b.stats.get("n_rows", 0)
            was_packed = bool(b.stats.get("packed", 0))
        return pts, rows, big, was_packed

    sampler = ClockSampler(local)
    sampler.start()  # nvidia-smi needs a moment to come up: started before the warm-up, read after the timed loops
    for i in range(args.warmup):
        step_device(i)
        if not args.no_e2e:
            step_e2e(i)
    if not args.no_e2e and args.e2e_engines > 1:
        stream_e2e(max(args.warmup, args.e2e_engines), 0)  # builds the other engines, sizes their buffers

    # ---- value: device-resident
    barrier()
    dev_ms, stats_sum, launches = 0.0, {}, 0
    wall0 = time.perf_counter()
    for i in range(args.steps):
        flush_l2()
        last = step_device(100 + i)
        st = last.stats
        dev_ms += st["ms_total"]
        launches += st["n_kernel_launches"]
        for k, v in st.items():
            stats_sum[k] = stats_sum.get(k, 0) + v
    barrier()
    wall_dev = time.perf_counter() - wall0
    # the last step's rows stay on the device until the next call on this engine: read back before the e2e legs run
    dump = dump_arrays(eng.read_device_result(last)) if args.dump_outputs and rank == 0 else None
    # ---- e2e: host buffers in, host buffers out
    barrier()
    e2e_s, e2e_points, e2e_rows, e2e_big = 0.0, 0, 0, 0
    for i in range(0 if args.no_e2e else args.steps):
        flush_l2()
        barrier()
        t0 = time.perf_counter()
        st = step_e2e(100 + i)
        torch.cuda.synchronize()
        e2e_s += time.perf_counter() - t0
        e2e_points += st["n_points"]
        e2e_big += st.get("n_big", 0)
        e2e_rows += st.get("n_rows", 0)
    barrier()
    # ---- e2e, pipelined: the same steps through simulate_stream (one call after the other above: e2e_sync)
    piped_s = None
    if not args.no_e2e and args.e2e_engines > 1:
        flush_l2()
        barrier()
        t0 = time.perf_counter()
        p_points, p_rows, p_big, e2e_packed = stream_e2e(args.steps, 1000)
        torch.cuda.synchronize()
        piped_s = time.perf_counter() - t0
        barrier()
    # ---- e2e in the reference's own return type: float64 [N, 3] + int64 [N] (or float64 [M, 8] Spyral rows) straight
    # from the device, 32 (72 + 8) B/row over PCIe -- what a `SimulationWriter.write` consumer gets without any decode
    f64_s, f64_steps = None, args.steps
    if not args.no_e2e and not args.float64_rows and args.e2e_engines > 1:
        stream_e2e(2, 2000, float64_rows=True, engines=2)  # (sizes the pinned float64 buffers)
        barrier()
        t0 = time.perf_counter()
        stream_e2e(f64_steps, 3000, float64_rows=True, engines=2)
        torch.cuda.synchronize()
        f64_s = time.perf_counter() - t0
        barrier()
    clocks = sampler.stop()
    # e2e_decoded: the same call plus the decode of the wire format into the arrays `SimulationWriter.write` receives
    # (float64 [N, 3] + int64 [N]; or the float64 [M, 8] Spyral rows), on one host thread; one step, rank-local
    decoded_s = None
    if not args.no_e2e and not args.float64_rows:
        warm = batch_e2e(998)  # (untimed: the decoder is JIT-compiled on first use)
        _ = (warm.rows, warm.row_labels) if args.spyral else (warm.cloud, warm.labels)
        del warm, _
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        b = batch_e2e(999)
        if args.spyral:
            _ = b.rows, b.row_labels
        else:
            _ = b.cloud, b.labels
        decoded_s = time.perf_counter() - t0
        del b, _

    dev_s = reduce_max(dist, dev_ms / 1e3, local)
    e2e_s = reduce_max(dist, e2e_s, local) if not args.no_e2e else float("nan")
    e2e_sync_s = e2e_s
    if f64_s is not None:
        f64_s = reduce_max(dist, f64_s, local)
    if piped_s is not None:  # the headline e2e is the pipelined call; its bytes are counted from its own batches
        e2e_s = reduce_max(dist, piped_s, local)
        e2e_points, e2e_rows, e2e_big = p_points, p_rows, p_big
    total_events = B * world * args.steps
    electrons = reduce_sum(dist, stats_sum["n_primary_electrons"], local)
    points = reduce_sum(dist, stats_sum["n_points"], local)
    deposits = reduce_sum(dist, stats_sum["n_deposits"], local)
    # bytes this rank brought to the host per step of the e2e loop (rows + CSR offsets), summed over the ranks
    row_bytes = (e2e_rows * (72 if args.float64_rows else 13) if args.spyral
                 else e2e_points * (32 if args.float64_rows else 8 if e2e_packed else 11) + 16 * e2e_big
                 + (1024 * B * args.steps if e2e_packed and not args.float64_rows else 0))
    d2h_local = 0.0 if args.no_e2e else row_bytes / max(1, args.steps) + (B + 1) * 8 * (2 if args.spyral else 1)
    d2h_total = reduce_sum(dist, d2h_local, local)

    if rank != 0:
        return
    peak, peak_src = measured_peak_hbm()
    # dominant kernel by device time (CUDA events recorded by the library around each stage, on its own stream)
    stage_ms = {"track_kernel": stats_sum["ms_tracks"], "point_scan+point_order": stats_sum["ms_order"],
                "deposit_kernel": stats_sum["ms_deposit"],
                "finalize (order+offsets+emit" + (", Spyral rows)" if args.spyral else ")"): stats_sum["ms_finalize"]}  # fmt: skip
    dominant = max(stage_ms, key=stage_ms.get)
    n_ev_rank = B * args.steps
    n_out = stats_sum["n_points"] / n_ev_rank
    bytes_per_event = 8 * (4 * K + 3) + 32 * n_out
    launches_dom = stats_sum["n_track_launches"] if dominant == "track_kernel" else stats_sum["n_group_launches"]
    events_per_launch = n_ev_rank / launches_dom
    avg_launch_ms = stage_ms[dominant] / launches_dom
    achieved = bytes_per_event * events_per_launch / (avg_launch_ms * 1e-3) / 1e9
    # DRAM traffic of the same kernel from the committed `ncu --set full` capture (profiles/traffic.json, written by
    # tools/ncu_summary.py): dram__bytes_read.sum + dram__bytes_write.sum per launch, scaled to this launch size
    traffic, traffic_note = None, "no ncu capture committed for this kernel"
    tj = ROOT / "profiles" / "traffic.json"
    if tj.exists():
        try:
            rec = json.loads(tj.read_text()).get(dominant)
            if rec and rec.get("workload") == args.workload:
                traffic = round(rec["dram_bytes_per_launch"] * events_per_launch / rec["events_per_launch"] / 1e9, 4)
                traffic_note = (f"GB per launch; {rec['source']}: {rec['dram_bytes_per_launch'] / 1e9:.3f} GB for "
                                f"{rec['events_per_launch']} events; issue slots busy {rec.get('issue_active_pct')} %")
        except Exception as exc:  # a malformed file must not break the benchmark
            traffic_note = f"profiles/traffic.json unreadable: {exc}"
    # The path is bound by instruction issue, not by HBM (SURVEY.md 8d): the roofline of the dominant kernel is its
    # issued warp instructions per second (count from the committed ncu capture, scaled to this launch size, over the
    # launch duration measured live) against 148 SMs x 4 schedulers x 1 warp instruction per clock; the HBM figure of
    # the whole step (algorithmic bytes over step time against the measured copy bandwidth) stands beside it.
    rec = None
    if tj.exists():
        try:
            rec = json.loads(tj.read_text()).get(dominant if dominant in ("track_kernel", "deposit_kernel") else "")
        except Exception:
            rec = None
    step_bytes = bytes_per_event * n_ev_rank / args.steps
    hbm = {"achieved": round(step_bytes / (dev_ms / args.steps * 1e-3) / 1e9, 2), "peak": peak, "unit": "GB/s",
           "frac": round(step_bytes / (dev_ms / args.steps * 1e-3) / 1e9 / peak, 5), "peak_source": peak_src,
           "what": "algorithmic bytes of the whole step (8 (4K + 3) + 32 N_out per event) over the step time"}  # fmt: skip
    sm_mhz = clocks.get("sm_max_mhz") or 1965.0
    issue_peak = 148 * 4 * sm_mhz * 1e6 / 1e9  # G warp instructions / s
    if rec and rec.get("workload") == args.workload and rec.get("warp_inst_per_launch"):
        inst = rec["warp_inst_per_launch"] * events_per_launch / rec["events_per_launch"]
        issue_achieved = inst / (avg_launch_ms * 1e-3) / 1e9
        roofline = {
            "kernel": dominant, "bound": "issue", "achieved": round(issue_achieved, 2), "peak": round(issue_peak, 1),
            "unit": "G warp-instructions/s", "frac": round(issue_achieved / issue_peak, 4),
            "peak_source": f"148 SMs x 4 schedulers x {sm_mhz:.0f} MHz", "traffic": traffic, "traffic_note": traffic_note,
            "instructions_note": f"{rec['warp_inst_per_launch']:.4g} warp instructions per {rec['events_per_launch']}-event launch "
                                 f"({rec['source']}; ncu issue-slot utilisation there: {rec.get('issue_active_pct')} %)",
            "events_per_launch": round(events_per_launch, 1), "avg_launch_ms": round(avg_launch_ms, 4), "hbm": hbm,
            "stage_ms_per_step": {k: round(v / args.steps, 3) for k, v in stage_ms.items()},
        }  # fmt: skip
    else:
        roofline = {
            "kernel": dominant, "bound": "hbm", "achieved": round(achieved, 3), "peak": peak, "unit": "GB/s",
            "frac": round(achieved / peak, 6), "traffic": traffic, "traffic_note": traffic_note, "peak_source": peak_src,
            "bytes_per_event": round(bytes_per_event, 1), "events_per_launch": round(events_per_launch, 1),
            "avg_launch_ms": round(avg_launch_ms, 4), "hbm": hbm,
            "note": "no committed ncu instruction count for this kernel / workload: algorithmic bytes of the path over "
                    "the kernel's time; the path is instruction-issue bound, not HBM bound (SURVEY.md 8d)",
            "stage_ms_per_step": {k: round(v / args.steps, 3) for k, v in stage_ms.items()},
        }  # fmt: skip
    out = {
        "metric": "detector-simulated events/s", "value": round(total_events / dev_s, 1), "unit": "events/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(dev_s / args.steps * 1e3, 3),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {
            "workload": f"{args.workload}: {WORKLOADS[args.workload]['desc']}", "events_per_gpu_per_step": B,
            "nuclei_per_event": K, "tracks": indices, "l2": "flushed between steps (256 MiB device write)",
            "dedx": "analytic Bethe+Lindhard table (not CATIMA)", "parallelism": f"event-range shards x{world}",
            "numa": f"rank 0 bound to {len(numa_cpus)} CPUs next to its GPU" if numa_cpus else "no binding",
            "output": "raw cloud [pad, tb, e] + Spyral rows (response, threshold, z-sort)" if args.spyral else "raw cloud [pad, tb, e]",
        },
        "electrons_per_s": round(electrons / dev_s, 1), "cloud_points_per_s": round(points / dev_s, 1),
        "pixel_deposits_per_s": round(deposits / dev_s, 1),
        "per_event": {"cloud_points": round(n_out, 1), "active_points": round(stats_sum["n_active_points"] / n_ev_rank, 1),
                      "trajectory_points": round(stats_sum["n_trajectory_points"] / n_ev_rank, 1),
                      "primary_electrons": round(stats_sum["n_primary_electrons"] / n_ev_rank, 1),
                      "table_flushes": round(stats_sum["n_table_flushes"] / n_ev_rank, 4),
                      "rhs_evals_per_track": round((6 * stats_sum["n_rk_steps"] + stats_sum["n_tracks"]) / max(1, stats_sum["n_tracks"]), 1)},
        "wall_s_device_loop": round(wall_dev, 3),
        "e2e": {"value": None if args.no_e2e else round(total_events / e2e_s, 1), "unit": "events/s",
                "h2d_bytes_per_step": int(momenta.nbytes + vertices.nbytes) * world,
                "result": ("Spyral rows float64[M,8] + labels" if args.spyral and args.float64_rows else
                           "Spyral rows (ADC threshold, z-sorted) as typed columns: pad int16, time bucket uint32 Q16.16, "
                           "electrons uint32 + uint16, label int8; the host rebuilds the 8 float64 columns bit for bit" if args.spyral else
                           "cloud float64[N,3] + int64 labels" if args.float64_rows else
                           "packed typed columns: pad id + track rank uint16, wiggle uint16, electrons uint32 + list of the "
                           "counts >= 2^32, rows per (event, time bucket) uint16 [B, 512]: 8 B/row + 1 KB/event, lossless" if e2e_packed else
                           "typed columns: pad int16, time bucket uint32 Q16.16, electrons uint32 + list of the counts >= 2^32, label int8"),
                "d2h_bytes_per_step": int(d2h_total),
                "call": (f"simulate_stream, {args.e2e_engines} engines per GPU: steps pipelined (the copy of one step to the "
                         "host overlaps the kernels of the next); inputs are read from pinned host memory and results "
                         "land in pinned host memory every step; working set per step >> L2" if piped_s is not None
                         else "simulate_batch, one call after the other; L2 flushed between steps")},
        "e2e_sync": None if args.no_e2e else {
            "value": round(total_events / e2e_sync_s, 1), "unit": "events/s",
            "what": "simulate_batch, one synchronous call per step, L2 flushed between steps"},
        "e2e_float64": None if f64_s is None else {
            "value": round(B * world * f64_steps / f64_s, 1), "unit": "events/s", "steps": f64_steps,
            "what": ("the same pipelined call returning the reference's own arrays, no decode on the host: "
                     + ("Spyral rows float64 [M, 8] + int64 labels, 80 B/row" if args.spyral else
                        "cloud float64 [N, 3] + int64 labels, 32 B/row") + " over PCIe (two engines)")},
        "e2e_decoded": None if decoded_s is None else {
            "value": round(B / decoded_s, 1), "unit": "events/s per rank",
            "what": "one e2e step plus the host-side decode of the typed columns into the float64 / int64 arrays of the "
                    "reference's writer protocol (raw cloud: one pass over the rows on all host threads, numba; "
                    "Spyral rows: numpy, one thread)"},
        "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline,
    }  # fmt: skip
    if world == 1 and not args.no_cpu:
        out["cpu_baseline"] = cpu_baseline(args, momenta, vertices)
    if dump is not None:
        write_dump(args.dump_outputs, dump)
    print(json.dumps(out), flush=True)
    if dist is not None:
        dist.destroy_process_group()


def run_pipeline(args):
    """BASELINE config 5 end to end: kinematics -> detector simulation -> host, sharded by event range.

    `--events-total` events (default 10 M) of `--workload` (default c16dd_sweep) are cut into chunks of `--events`;
    rank r of N takes a contiguous range of chunks (one process per GPU, no collective on the data path).  Per chunk:
    the vectorised `KinematicsPipeline.run_batch` (two prefetch threads; a chunk's seed depends on the chunk alone, so
    the events do not depend on N), `simulate_stream` (pipelined `simulate_batch`) with host inputs and the typed columns back in pinned host memory,
    and a gather step that keeps the CSR offsets and per-chunk totals.  The real bulk writer (`ParquetCloudWriter`, zstd) is timed on the
    first `--writer-chunks` chunks of rank 0 into a scratch directory and reported beside it: a full 10 M-event cloud is
    ~0.9 TB as float64 rows (0.3 TB as typed columns), more than the box can hold or write in minutes.
    """
    import threading

    import torch

    from attpc_engine_b200 import nuclear_map
    from attpc_engine_b200.detector.engine import engine_for
    from attpc_engine_b200.detector.sharding import shard_range
    from attpc_engine_b200.detector.simulator import _nuclei_for

    local_env = int(os.environ.get("LOCAL_RANK", "0"))
    if int(os.environ.get("WORLD_SIZE", "1")) > 1 and not args.no_numa:
        from attpc_engine_b200.detector.sharding import bind_to_gpu_numa_node

        bind_to_gpu_numa_node(local_env)
    rank, world, local, dist = dist_setup(args.gpus)
    torch.cuda.set_device(local)
    name = args.workload
    B = args.events
    n_chunks = -(-args.events_total // B)
    c0, c1 = shard_range(n_chunks, rank, world)
    config, m0, v0, zs, as_, indices = build_workload(name, 8)
    K = m0.shape[1]

    def kinematics(c):
        pipeline, _ = make_pipeline(name)  # (cheap: tables are cached per process)
        pipeline.seed(workload_seed(name, 1000 + c))
        n = min(B, args.events_total - c * B)
        t0 = time.perf_counter()
        vertices, momenta = pipeline.run_batch(n)
        return c, momenta, vertices, time.perf_counter() - t0

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()

    from concurrent.futures import ThreadPoolExecutor

    from attpc_engine_b200.detector import simulate_stream

    # warm-up: engines built, buffers sized, kernels loaded
    _, m, v, _ = kinematics(c0)
    warm = [(m, v, c0 * B)] * max(args.e2e_engines, args.warmup)
    for _ in simulate_stream(warm, zs, as_, config, 1, indices, devices=[local], engines_per_device=args.e2e_engines,
                             copy=False, columns=True):  # fmt: skip
        pass
    barrier()
    wall0 = time.perf_counter()
    # kinematics of the next chunks on two prefetch threads, the chunks through the pipelined public call
    pool = ThreadPoolExecutor(max_workers=2)
    chunks = list(range(c0, c1))
    futures, submitted, kin_lock = {}, [0], threading.Lock()
    t_kin_box = [0.0]

    def reader(k):
        def read():
            with kin_lock:
                while submitted[0] < min(len(chunks), k + 5):
                    futures[submitted[0]] = pool.submit(kinematics, chunks[submitted[0]])
                    submitted[0] += 1
                fut = futures.pop(k)
            c, momenta, vertices, dt = fut.result()
            t_kin_box[0] += dt
            return momenta, vertices, c * B

        read.thread_safe = True
        return read

    t_gather, events, points, electrons = 0.0, 0, 0, 0
    check = np.zeros(2, dtype=np.uint64)
    for _, batch in simulate_stream([reader(k) for k in range(len(chunks))], zs, as_, config, 20260101, indices,
                                    devices=[local], engines_per_device=args.e2e_engines, copy=False, columns=True):  # fmt: skip
        t1 = time.perf_counter()
        # gather: what a shard hands to the collector -- the CSR offsets and a checksum over the head of two columns
        # (reading every byte is the writer's job: see writer_sample)
        head = batch.packed["pad_rank"] if batch.packed is not None else batch.columns["pad"]
        check[0] += np.uint64(int(np.add.reduce(head[: 1 << 20], dtype=np.int64)) & (2**63 - 1))
        check[1] += np.uint64(int(batch.offsets[-1]))
        t_gather += time.perf_counter() - t1
        events += len(batch)
        points += batch.stats["n_points"]
        electrons += batch.stats["n_primary_electrons"]
    pool.shutdown()
    t_kin = t_kin_box[0]
    barrier()
    wall = time.perf_counter() - wall0
    wall = reduce_max(dist, wall, local)
    total_events = reduce_sum(dist, events, local)
    total_points = reduce_sum(dist, points, local)
    total_electrons = reduce_sum(dist, electrons, local)
    if rank != 0:
        return
    # the real bulk writer on a bounded sample (rank 0)
    writer_info = None
    if args.writer_chunks > 0:
        from attpc_engine_b200.detector import ParquetCloudWriter, simulate_batch

        tmp = Path(tempfile.mkdtemp(prefix="attpc_bench_"))
        try:
            w = ParquetCloudWriter(tmp)
            n_w = min(args.writer_chunks, c1 - c0)
            ev_w = rows_w = 0
            t_w = 0.0
            for c in range(c0, c0 + n_w):
                _, momenta, vertices, _ = kinematics(c)
                batch = simulate_batch(momenta, vertices, zs, as_, config, 20260101, indices, first_event=c * B,
                                       device=local, copy=False, columns=True)  # fmt: skip
                t0 = time.perf_counter()
                w.write_batch(batch, config)
                t_w += time.perf_counter() - t0
                ev_w += len(batch)
                rows_w += batch.stats["n_points"]
            t0 = time.perf_counter()
            w.close()
            t_w += time.perf_counter() - t0
            size = sum(f.stat().st_size for f in tmp.glob("*.parquet"))
            writer_info = {"writer": "ParquetCloudWriter (zstd), one process", "events": ev_w, "rows": int(rows_w),
                           "seconds": round(t_w, 3), "events_per_s": round(ev_w / t_w, 1),
                           "bytes_written": int(size), "bytes_per_event": round(size / max(1, ev_w), 1)}  # fmt: skip
        finally:
            shutil.rmtree(tmp, ignore_errors=True)
    out = {
        "metric": "detector-simulated events/s (pipeline: kinematics -> simulate -> host gather)",
        "value": round(total_events / wall, 1), "unit": "events/s", "n_gpus": world, "higher_is_better": True,
        "scaling": "strong", "dtype": "f64", "data": "synthetic", "mode": "pipeline",
        "config": {"workload": f"{name}: {WORKLOADS[name]['desc']}", "events_total": int(total_events),
                   "events_per_chunk": B, "chunks_per_rank": c1 - c0, "parallelism": f"event-range shards x{world}",
                   "result": "typed columns in pinned host memory, per-chunk totals gathered"},
        "wall_s": round(wall, 3), "cloud_points": int(total_points), "electrons_per_s": round(total_electrons / wall, 1),
        "rank0_seconds": {"kinematics (2 prefetch threads, summed)": round(t_kin, 3), "gather": round(t_gather, 3)},
        "call": f"simulate_stream, {args.e2e_engines} engines per GPU (host in, typed columns in pinned host memory out)",
        "checksum": [int(check[0]), int(check[1])], "writer_sample": writer_info,
    }  # fmt: skip
    print(json.dumps(out), flush=True)
    if dist is not None:
        dist.destroy_process_group()


def run_threads(args):
    """e2e with ONE process and one thread + engine per GPU (the `run_simulation(devices=[...])` arrangement), as a
    counterpart to the one-process-per-GPU launch: does the host-side limit of a multi-GPU box depend on it?"""
    import threading

    import torch

    from attpc_engine_b200 import nuclear_map
    from attpc_engine_b200.detector.engine import engine_for
    from attpc_engine_b200.detector.simulator import _nuclei_for

    G, B = args.thread_gpus, args.events
    config, momenta, vertices, zs, as_, indices = build_workload(args.workload, B)
    nuclei = _nuclei_for(zs, as_, indices, nuclear_map)
    engines = [engine_for(config, nuclei, device=g, instance=g, max_events_per_launch=args.launch_events,
                          copy_events_per_launch=args.copy_events) for g in range(G)]  # fmt: skip
    pins = [(torch.from_numpy(momenta).pin_memory(), torch.from_numpy(vertices).pin_memory()) for _ in range(G)]
    barrier = threading.Barrier(G + 1)
    spans, errors = [None] * G, []

    def worker(g):
        try:
            torch.cuda.set_device(g)
            m, v = pins[g]
            for i in range(args.warmup):
                engines[g].simulate_batch(m.numpy(), v.numpy(), zs, as_, indices, seed=i, first_event=g * B, copy=False,
                                          columns=not args.float64_rows)  # fmt: skip
            barrier.wait()
            t0 = time.perf_counter()
            pts = 0
            for i in range(args.steps):
                st = engines[g].simulate_batch(m.numpy(), v.numpy(), zs, as_, indices, seed=100 + i, first_event=g * B,
                                               copy=False, columns=not args.float64_rows).stats  # fmt: skip
                pts += st["n_points"]
            spans[g] = (t0, time.perf_counter(), pts)
        except BaseException as exc:  # noqa: BLE001
            errors.append(exc)
            barrier.abort()

    threads = [threading.Thread(target=worker, args=(g,)) for g in range(G)]
    for t in threads:
        t.start()
    barrier.wait()
    for t in threads:
        t.join()
    if errors:
        raise errors[0]
    wall = max(s[1] for s in spans) - min(s[0] for s in spans)
    points = sum(s[2] for s in spans)
    out = {"metric": "detector-simulated events/s", "mode": "one process, one thread per GPU", "n_gpus": G,
           "e2e": {"value": round(G * B * args.steps / wall, 1), "unit": "events/s",
                   "d2h_bytes_per_step": int(points / args.steps * (32 if args.float64_rows else 11))},
           "d2h_GBps": round(points * (32 if args.float64_rows else 11) / wall / 1e9, 2), "steps": args.steps,
           "config": {"workload": args.workload, "events_per_gpu_per_step": B}}  # fmt: skip
    print(json.dumps(out), flush=True)


def cpu_baseline(args, momenta, vertices):
    arm = CpuArm(args.workload, args.cpu_cores or None)
    n = min(len(momenta), max(64, args.cpu_events_per_core * arm.cores))
    arm.run(momenta[: arm.cores], vertices[: arm.cores])  # every worker has imported and JIT-compiled before timing
    res = arm.run(momenta[:n], vertices[:n])
    arm.close()
    return {"value": round(res["events"] / res["wall_s"], 2), "unit": "events/s", "cores": arm.cores, "kind": "port",
            "sample": f"first {n} events of the same workload, {arm.cores} processes, numba warm-up excluded",
            "events_per_s_per_core": round(res["events"] / res["core_s"], 2),
            "electrons_per_s": round(res["electrons"] / res["wall_s"], 1)}  # fmt: skip


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    arm = CpuArm(args.workload, args.cpu_cores or None)
    n = max(64, args.cpu_events_per_core * arm.cores)
    config, momenta, vertices, zs, as_, indices = build_workload(args.workload, n)
    for _ in range(args.warmup):
        arm.run(momenta[: arm.cores], vertices[: arm.cores])
    wall = events = electrons = 0.0
    core_s = 0.0
    for i in range(args.steps):
        res = arm.run(momenta, vertices, first=i * n)
        wall += res["wall_s"]
        events += res["events"]
        electrons += res["electrons"]
        core_s += res["core_s"]
    arm.close()
    value = round(events / wall, 2)
    sample = f"{n} events per step of the same workload, {arm.cores} processes"
    out = {
        "impl": "reference", "metric": "detector-simulated events/s", "value": value, "unit": "events/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(wall / args.steps * 1e3, 1),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"{args.workload}: {WORKLOADS[args.workload]['desc']}", "events_per_step": n,
                   "dedx": "analytic Bethe+Lindhard table (not CATIMA)"},
        "electrons_per_s": round(electrons / wall, 1),
        "cpu_baseline": {"value": value, "unit": "events/s", "cores": arm.cores, "kind": "port", "sample": sample,
                         "events_per_s_per_core": round(events / core_s, 2)},
        "e2e": {"value": value, "unit": "events/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }  # fmt: skip
    print(json.dumps(out), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c16dd", choices=sorted(WORKLOADS))
    ap.add_argument("--events", type=int, default=32768, help="events per GPU per step")
    ap.add_argument("--launch-events", type=int, default=0, help="events per track-kernel launch (0 = library default)")
    ap.add_argument("--copy-events", type=int, default=0, help="events per host-copy chunk (0 = library default)")
    ap.add_argument("--tune", action="append", default=[], metavar="KEY=INT",
                    help="engine tuning knob, e.g. table_spill_keys=3000 or unit_points=512 (results do not depend on them)")
    ap.add_argument("--cpu-cores", type=int, default=0)
    ap.add_argument("--cpu-events-per-core", type=int, default=64)
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-numa", action="store_true", help="multi-GPU: do not bind each rank to the CPUs next to its GPU")
    ap.add_argument("--no-e2e", action="store_true", help="profiling aid: only the device-resident steps")
    ap.add_argument("--e2e-engines", type=int, default=3,
                    help="engines per GPU of the pipelined e2e call (simulate_stream); 1 = synchronous calls only")
    ap.add_argument("--spyral", action="store_true", help="also produce the Spyral 8-column rows (full pad-plane response)")
    ap.add_argument("--pipeline", action="store_true",
                    help="BASELINE config 5: kinematics -> simulate -> host for --events-total events, sharded over the ranks")
    ap.add_argument("--events-total", type=int, default=10_000_000, help="--pipeline: events of the whole job")
    ap.add_argument("--writer-chunks", type=int, default=1, help="--pipeline: chunks also written with ParquetCloudWriter (rank 0)")
    ap.add_argument("--thread-gpus", type=int, default=0,
                    help="e2e only: ONE process with a thread and an engine per GPU (0 = off)")
    ap.add_argument("--float64-rows", action="store_true",
                    help="e2e: bring the cloud back as float64[N,3] + int64 labels (32 B/row) instead of typed columns")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed device-resident step computed (rank 0) as DIR/<name>.npy, float64, "
                         "at most 64 MB: points_per_event, and sample_events / cloud / labels of a seeded event sample")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl == "reference" or args.thread_gpus > 0 or args.pipeline):
        ap.error("--dump-outputs applies to the device-resident steps of the default mode")
    if "NUMBA_CACHE_DIR" not in os.environ:  # numba's on-disk cache (the column decoder) stays out of the tree
        os.environ["NUMBA_CACHE_DIR"] = tempfile.mkdtemp(prefix="attpc_bench_numba_")
        atexit.register(shutil.rmtree, os.environ["NUMBA_CACHE_DIR"], ignore_errors=True)
    if args.impl == "reference":
        run_reference(args)
    elif args.thread_gpus > 0:
        run_threads(args)
    elif args.pipeline:
        if args.workload == "c16dd":
            args.workload = "c16dd_sweep"
        run_pipeline(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
