"""Rolling forecasts of the 3-year 34-station table: every hourly window through the forward on materialised windows
(a) against GCN_GRU.forecast (b), FP32 and tensor path, on one GPU.  Prints one JSON line.

    python scripts/forecast_time.py [--out FILE] [--profile FILE]

Workload: a seeded [26304, 34, 13] table (3 years of hours, the shipped 34-station model) and all 26,134 windows of
168 hours that have 3 label hours after them.
  (a) x = table[starts[:, None] + arange(168)] (a gather, 7.8 GB), ops.gcn_gru_forward(x)[:, -1]
  (b) model.forecast(adj, table, starts)
Both routes are warmed up, then timed alternately with CUDA events, each timed window at least --min-seconds long;
the median window is reported.  The outputs must be bit-identical.  Peak device memory of a route: the allocator's
peak during one call above what was allocated before it, workspaces released first (so it includes the route's
workspace).  --profile FILE: a torch.profiler CUDA-kernel table of one call of each route, in a run of its own.
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
from windgnn_b200 import ops  # noqa: E402

TTOT, S, L, HORIZONS = 26304, 34, 168, 3
DEV = torch.device("cuda:0")


def setup():
    golden = os.path.join(ROOT, "tests", "golden")
    sd = torch.load(os.path.join(golden, "wind_gnn_34.pth"), map_location="cpu", weights_only=True)
    model = windgnn_b200.GCN_GRU(13, 13, 13, 13 * S, 3 * S)
    model.load_state_dict(sd, strict=True)
    model = model.to(DEV).eval()
    adj = torch.from_numpy(np.load(os.path.join(golden, "adj_ref_34.npy")).astype(np.float32)).to(DEV)
    g = torch.Generator(device=DEV).manual_seed(2024)
    table = torch.rand((TTOT, S, 13), generator=g, device=DEV)
    starts = windgnn_b200.window_starts(TTOT, L, 1, HORIZONS)
    return model, adj, table, starts


def routes(model, adj, table, starts, flags):
    params = [p.detach() for p in (model.conv1.weight, model.conv1.bias, model.conv2.weight, model.conv2.bias,
                                   model.gru.weight_ih_l0, model.gru.weight_hh_l0, model.gru.bias_ih_l0,
                                   model.gru.bias_hh_l0)]
    idx = starts.to(DEV)[:, None] + torch.arange(L, device=DEV)

    def materialised():
        x = table[idx]
        return ops.gcn_gru_forward(adj, x, *params, 0, flags)[:, -1]

    def forecast():
        model.precision = "tensor" if flags else "fp32"
        return model.forecast(adj, table, starts, seq_length=L)

    return {"materialised": materialised, "forecast": forecast}


def time_calls(fn, n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / n


def peak_bytes(fn):
    ops.release_workspaces()
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


def profile(path, model, adj, table, starts):
    from torch.profiler import ProfilerActivity, profile as tprofile

    with open(path, "w") as f:
        for flags, prec in ((0, "fp32"), (1, "tensor")):
            for name, fn in routes(model, adj, table, starts, flags).items():
                fn()
                torch.cuda.synchronize()
                with tprofile(activities=[ProfilerActivity.CUDA]) as prof:
                    fn()
                    torch.cuda.synchronize()
                f.write(f"==== {name} {prec}: one call, {starts.numel()} windows\n")
                f.write(prof.key_averages().table(sort_by="cuda_time_total", row_limit=15) + "\n")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--min-seconds", type=float, default=1.0)
    ap.add_argument("--reps", type=int, default=3, help="timed windows per route (alternating)")
    ap.add_argument("--out", help="also write the JSON line to this file")
    ap.add_argument("--profile", metavar="FILE", help="write a torch.profiler kernel table instead of timing")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("forecast_time.py needs a CUDA device")
    model, adj, table, starts = setup()
    if args.profile:
        profile(args.profile, model, adj, table, starts)
        return
    N = starts.numel()
    gpu, power = card()
    res = {"workload": f"rolling forecasts: table {TTOT} x {S} x 13, {N} windows of {L} h (stride 1)",
           "gpu": gpu, "power_limit_and_max_sm_clock": power}
    for flags, prec in ((0, "fp32"), (1, "tensor")):
        fns = routes(model, adj, table, starts, flags)
        a, b = fns["materialised"](), fns["forecast"]()
        torch.cuda.synchronize()
        assert torch.equal(a, b), f"{prec}: forecast differs from the forward's last step"
        del a, b
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
        leg = {}
        for k in fns:
            m = float(np.median(ms[k]))
            leg[k] = {"ms_per_call": round(m, 3), "windows_per_s": round(N / m * 1e3),
                      "calls_per_window": n_calls[k], "ms_all_windows": [round(v, 3) for v in ms[k]],
                      "peak_device_mb": round(mem[k] / 2**20, 1)}
        leg["speedup"] = round(leg["materialised"]["ms_per_call"] / leg["forecast"]["ms_per_call"], 2)
        leg["bit_identical"] = True
        res[prec] = leg
    res["table_mb"] = round(table.numel() * 4 / 2**20, 1)
    line = json.dumps(res)
    print(line, flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
