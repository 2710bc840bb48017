"""Cost of longitudinal diffusion: device-resident steps and end-to-end `simulate_stream` at D_L in {0, 0.1, 0.277} V.

    python tools/longitudinal_bench.py --out profiles/r03_longitudinal_b200.json [--steps 10] [--warmup 3]

Device-resident: 32768-event steps of `bench.build_workload` through `Engine.simulate_device` (inputs on the GPU,
results left there), L2 overwritten between steps as bench.py does; reports events/s, the stage times of the library's
CUDA events (ms_order = point ordering, and with D_L > 0 the split into sub-points; ms_deposit = deposit kernel alone;
ms_finalize), deposits and keys per event, and the device time per pixel deposit.  End to end: the same steps through
`simulate_stream` (two engines, packed typed columns to pinned host memory) for c16dd.  The card's name and power limit
are read in the same run.
"""

import argparse
import copy
import dataclasses
import gc
import json
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

D_LS = (0.0, 0.1, 0.277)
EVENTS = 32768


def with_dl(config, d_l):
    out = copy.copy(config)
    out.__dict__.pop("_b200_engines", None)
    out.det_params = dataclasses.replace(config.det_params, longitudinal_diffusion=d_l)
    return out


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)  # fmt: skip
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def device_leg(name, d_l, steps, warmup):
    import torch

    import bench
    from attpc_engine_b200 import nuclear_map
    from attpc_engine_b200.detector.engine import engine_for
    from attpc_engine_b200.detector.simulator import _nuclei_for

    config, momenta, vertices, zs, as_, indices = bench.build_workload(name, EVENTS)
    config = with_dl(config, d_l)
    eng = engine_for(config, _nuclei_for(zs, as_, indices, nuclear_map))
    mom = torch.from_numpy(momenta).cuda()
    vtx = torch.from_numpy(vertices).cuda()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    K = momenta.shape[1]
    for i in range(warmup):
        eng.simulate_device(mom.data_ptr(), vtx.data_ptr(), EVENTS, K, zs, as_, indices, seed=20260101 + i)
    tot = {}
    for i in range(steps):
        flush.zero_()
        torch.cuda.synchronize()
        st = eng.simulate_device(mom.data_ptr(), vtx.data_ptr(), EVENTS, K, zs, as_, indices, seed=20260201 + i).stats
        for k in ("ms_total", "ms_order", "ms_deposit", "ms_finalize", "ms_tracks", "n_deposits", "n_keys",
                  "n_active_points", "n_retries", "n_kernel_launches"):  # fmt: skip
            tot[k] = tot.get(k, 0) + st[k]
    n_ev = steps * EVENTS
    out = {
        "workload": name, "longitudinal_diffusion_V": d_l, "events_per_step": EVENTS, "steps": steps,
        "events_per_s": round(n_ev / (tot["ms_total"] / 1e3), 1),
        "ms_per_step": {k: round(tot[k] / steps, 3) for k in ("ms_total", "ms_tracks", "ms_order", "ms_deposit", "ms_finalize")},
        "per_event": {k: round(tot[k] / n_ev, 2) for k in ("n_active_points", "n_deposits", "n_keys")},
        "ns_per_deposit": round(tot["ms_deposit"] * 1e6 / tot["n_deposits"], 5),
        "ns_per_deposit_incl_order": round((tot["ms_deposit"] + tot["ms_order"]) * 1e6 / tot["n_deposits"], 5),
        "kernel_launches_per_step": tot["n_kernel_launches"] / steps, "retries_in_timed_steps": tot["n_retries"],
    }  # fmt: skip
    del eng, config, mom, vtx, flush
    gc.collect()
    torch.cuda.empty_cache()
    return out


def stream_leg(name, d_l, steps, warmup):
    import bench
    from attpc_engine_b200.detector import simulate_stream

    config, momenta, vertices, zs, as_, indices = bench.build_workload(name, EVENTS)
    config = with_dl(config, d_l)

    def run(n, step0):
        rows = 0
        batches = [(momenta, vertices, (step0 + k) * EVENTS) for k in range(n)]
        for _, b in simulate_stream(batches, zs, as_, config, 20260101, indices, engines_per_device=2, copy=False,
                                    columns=True):  # fmt: skip
            rows += b.stats["n_points"]
        return rows

    run(max(warmup, 2), 0)
    t0 = time.perf_counter()
    rows = run(steps, 100)
    dt = time.perf_counter() - t0
    return {"workload": name, "longitudinal_diffusion_V": d_l, "events": steps * EVENTS,
            "events_per_s": round(steps * EVENTS / dt, 1), "rows_per_event": round(rows / (steps * EVENTS), 2),
            "call": "simulate_stream, 2 engines, packed typed columns in pinned host memory"}  # fmt: skip


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--out", required=True, help="JSON file to write")
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    out = {"gpu": card(), "device_resident": [], "end_to_end": []}
    for name in ("c16dd", "c12aa"):
        for d_l in D_LS:
            r = device_leg(name, d_l, args.steps, args.warmup)
            print(json.dumps(r), flush=True)
            out["device_resident"].append(r)
    for d_l in D_LS:
        r = stream_leg("c16dd", d_l, args.steps, args.warmup)
        print(json.dumps(r), flush=True)
        out["end_to_end"].append(r)
    base = {r["workload"]: r["ns_per_deposit"] for r in out["device_resident"] if r["longitudinal_diffusion_V"] == 0.0}
    out["deposit_time_ratio_vs_off"] = {
        f'{r["workload"]}@{r["longitudinal_diffusion_V"]}': round(r["ns_per_deposit"] / base[r["workload"]], 3)
        for r in out["device_resident"]
    }
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(out, indent=1) + "\n")
    print(json.dumps(out["deposit_time_ratio_vs_off"]), flush=True)


if __name__ == "__main__":
    main()
