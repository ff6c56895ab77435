"""Training steps on random hourly windows of the 3-year 34-station table: materialising the windows plus
Trainer.step (a) against Trainer.step_table (b), on one GPU.  Prints one JSON line.

    python scripts/train_table_time.py [--out FILE] [--batches 512 4096]

Workload: the seeded [26304, 34, 13] table of scripts/forecast_time.py, the shipped 34-station model, and B windows of
168 hours drawn at random (seeded, without repeats) from the 26,134 hourly windows with 3 label hours after them.
  (a) x = table[starts[:, None] + arange(168)], y = its targets (two gathers), trainer.step(x, y)
  (b) trainer.step_table(table, starts)
Each route has its own trainer from the same checkpoint.  Both are warmed up, then timed alternately with CUDA events,
each timed window at least --min-seconds long; the median window is reported.  Peak device memory of a route: the
allocator's peak during one step above what was allocated before it.  Then, in a separate pass under torch.profiler,
one step of each route gives the time of every kernel (ms per step); the dGI row reduction's bandwidth is its bytes
(every DG row read once, every span row written once) over its time.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import windgnn_b200  # noqa: E402
from windgnn_b200 import train  # noqa: E402

TTOT, S, L, HORIZONS, LABEL = 26304, 34, 168, 3, 11
H = 3 * S
DEV = torch.device("cuda:0")


def setup():
    golden = os.path.join(ROOT, "tests", "golden")
    sd = torch.load(os.path.join(golden, "wind_gnn_34.pth"), map_location="cpu", weights_only=True)
    adj = torch.from_numpy(np.load(os.path.join(golden, "adj_ref_34.npy")).astype(np.float32)).to(DEV)
    g = torch.Generator(device=DEV).manual_seed(2024)
    table = torch.rand((TTOT, S, 13), generator=g, device=DEV)
    return sd, adj, table


def trainer(sd, adj):
    model = windgnn_b200.GCN_GRU(13, 13, 13, 13 * S, H)
    model.load_state_dict(sd, strict=True)
    return train.Trainer(model.to(DEV).train(), adj)


def routes(sd, adj, table, starts):
    rows = starts.to(DEV)[:, None] + torch.arange(L, device=DEV)
    lab = rows[:, :, None] + 1 + torch.arange(HORIZONS, device=DEV)
    ta, tb = trainer(sd, adj), trainer(sd, adj)

    def materialised():
        x = table[rows]
        y = table[lab, :, LABEL].reshape(starts.numel(), L, HORIZONS * S)
        return ta.step(x, y)

    def table_windows():
        return tb.step_table(table, starts, seq_length=L, label_feature=LABEL, horizons=HORIZONS)

    return {"materialised": materialised, "table": table_windows}


def time_calls(fn, n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / n


def peak_bytes(fn):
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    base = torch.cuda.memory_allocated(DEV)
    torch.cuda.reset_peak_memory_stats(DEV)
    out = fn()
    torch.cuda.synchronize()
    del out
    return torch.cuda.max_memory_allocated(DEV) - base


def card():
    name = torch.cuda.get_device_name(DEV)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        q = f"unavailable ({type(e).__name__})"
    return name, q


def kernel_ms(fn):
    """ms per kernel name in one step (torch.profiler, CUDA activities)."""
    from torch.profiler import ProfilerActivity, profile

    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = e.cuda_time_total
        if t > 0:
            out[e.key[:90]] = round(t / 1e3, 4)
    return dict(sorted(out.items(), key=lambda kv: -kv[1]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--min-seconds", type=float, default=1.0)
    ap.add_argument("--reps", type=int, default=3, help="timed windows per route (alternating)")
    ap.add_argument("--batches", type=int, nargs="+", default=[512, 4096])
    ap.add_argument("--out", help="also write the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("train_table_time.py needs a CUDA device")
    sd, adj, table = setup()
    gpu, power = card()
    all_starts = windgnn_b200.window_starts(TTOT, L, 1, HORIZONS)
    res = {"workload": f"training steps: table {TTOT} x {S} x 13, B random hourly windows of {L} h "
                       f"(of {all_starts.numel()}), shipped 34-station model",
           "gpu": gpu, "power_limit_and_max_sm_clock": power}
    rng = np.random.default_rng(7)
    for B in args.batches:
        starts = all_starts[torch.from_numpy(rng.choice(all_starts.numel(), size=B, replace=False))]
        span = int(starts.max()) + L - int(starts.min())
        fns = routes(sd, adj, table, starts)
        la, lb = fns["materialised"](), fns["table"]()   # first step from the same checkpoint
        torch.cuda.synchronize()
        first = {"loss_materialised": la.item(), "loss_table": lb.item()}
        mem = {k: peak_bytes(fn) for k, fn in fns.items()}
        n_calls = {}
        for k, fn in fns.items():   # warm-up, then calls per timed window
            fn()
            t = time_calls(fn, 2)
            n_calls[k] = max(2, int(np.ceil(args.min_seconds * 1.1e3 / t)))
        ms = {k: [] for k in fns}
        for _ in range(args.reps):
            for k, fn in fns.items():
                ms[k].append(time_calls(fn, n_calls[k]))
        leg = {"windows": B, "span_rows": span, "window_rows": B * L, **first}
        for k in fns:
            m = float(np.median(ms[k]))
            leg[k] = {"ms_per_step": round(m, 3), "windows_per_s": round(B / m * 1e3),
                      "steps_per_window": n_calls[k], "ms_all_windows": [round(v, 3) for v in ms[k]],
                      "peak_device_mb": round(mem[k] / 2**20, 1)}
        leg["speedup"] = round(leg["materialised"]["ms_per_step"] / leg["table"]["ms_per_step"], 2)
        # per-stage kernel times, a separate pass under the profiler
        for k, fn in fns.items():
            leg[k]["kernels_ms"] = kernel_ms(fn)
        dgi = [v for n, v in leg["table"]["kernels_ms"].items() if "dgi_rows_kernel" in n]
        if dgi:
            G4, LD4 = (3 * H + 3) // 4 * 4, (4 * H + 3) // 4 * 4
            nbytes = B * L * G4 * 4 + span * LD4 * 4
            leg["dgi_rows"] = {"ms": dgi[0], "bytes": nbytes, "gb_per_s": round(nbytes / (dgi[0] * 1e-3) / 1e9, 1)}
        res[f"B{B}"] = leg
        del fns
    res["table_mb"] = round(table.numel() * 4 / 2**20, 1)
    line = json.dumps(res)
    print(line, flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
