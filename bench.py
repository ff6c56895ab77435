#!/usr/bin/env python
"""Benchmark of the WindGNN GCN-GRU forward hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

One "step" = one forward of the workload (BASELINE.json configs[1]: the shipped 34-station checkpoint,
batch 4096 windows of 168 hours) per GPU; exactly K steps are timed, after max(W, 3) untimed ones.  At
about 5 ms per step, K >= 400 gives a timed region of 2 s (sustained clocks, >= 20 nvidia-smi samples inside
it).  With N > 1 (launched through ``torch.distributed.run``) every rank runs the same per-GPU batch on
its own device (weak scaling: the sequence batch is sharded, no collective on the data path).

Prints ONE JSON line (rank 0):
  value         sequences/s with the inputs resident in HBM (CUDA events, max over ranks)
  e2e           the same through the host-buffer entry point (pinned host input, H2D + compute + D2H inside
                the timed region) + the measured concurrent H2D ceiling of the box it is bounded by
  roofline      the dominant kernel (the input-projection FFMA GEMM) against the FP32 FFMA peak measured
                live on the same GPU (and the nominal peak), its algorithmic bytes and the ncu DRAM traffic
                of the committed capture of THIS workload (profiles/r02_ncu_summary.json)
  cpu_baseline  the reference's own classes (oracle/_ref, kind "reference"; the oracle's torch port,
                kind "port", if oracle/_ref is absent) on this box's host cores
  gpu_eager     the reference's own classes in PyTorch eager on the same B200 (cuBLAS + cuDNN GRU): batched
                through its sub-modules, and as written (one window per call, src/main.py:101-102)
  tensor_path   the opt-in tensor-core path on the same workload (device-resident and end to end)
  scaled        BASELINE.json configs[0] (7 stations), configs[2] (2^20 windows, sharded) and configs[3]
                (4096-station kNN graph) as sub-objects: value, ms, FP32 fraction
  train_step    BASELINE.json configs[4]

``--impl reference`` times the reference's CPU forward alone on the full configs[1] step (4096 windows
per step), all host threads.

``--dump-outputs DIR`` writes what the timed path returned in its last timed step (rank 0) as
DIR/<name>.npy, float32.  The inputs are seeded, so two builds run with the same arguments can be
compared output for output.  An output above 64 MB is cut to a fixed sample of windows (see dump_output).
"""

from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")
METRIC = "gcn_gru_forward_sequences_per_s"
UNIT = "sequences/s"
NCU_SUMMARY = os.path.join(ROOT, "profiles", "r02_ncu_summary.json")   # capture of THIS workload (B=4096, S=34)

# workload = BASELINE.json configs[1]
S, T, F, B_PER_GPU = 34, 168, 13, 4096
H, I = 3 * S, 13 * S


def flop_per_seq(S_, T_, Fi, Fh, Fo, H_, nnz=None):
    """Algorithmic FLOPs of one sequence (SURVEY.md 8(d)): matmul multiply-adds x 2 only."""
    a = S_ * S_ if nnz is None else nnz
    gcn = 2 * (a * Fi + S_ * Fi * Fh) + 2 * (a * Fh + S_ * Fh * Fo)
    return T_ * (gcn + 2 * (S_ * Fo) * 3 * H_ + 2 * H_ * 3 * H_)


def bytes_per_seq(S_, T_, Fi, H_):
    """Mandatory HBM traffic of one sequence: input read once + output written once."""
    return T_ * S_ * Fi * 4 + T_ * H_ * 4


FLOP_IH = 2 * I * 3 * H
FLOP_PER_SEQ = flop_per_seq(S, T, F, F, F, H)        # 69,892,032
BYTES_PER_SEQ = bytes_per_seq(S, T, F, H)            # 365,568


def load_workload(S_=34):
    sd = torch.load(os.path.join(GOLDEN, f"wind_gnn_{S_}.pth"), map_location="cpu", weights_only=True)
    with open(os.path.join(GOLDEN, "coords.json")) as f:
        c = json.load(f)
    idx = list(range(7)) if S_ == 7 else [i for i, n in enumerate(c["names"]) if n != "Enchant 2 AGCM"]
    latlon = np.array([[c["lat"][i], c["lon"][i]] for i in idx], dtype=np.float64)
    return sd, latlon


DUMP_MAX_BYTES = 64_000_000


def dump_output(out_dir: str, name: str, y: torch.Tensor) -> None:
    """Save `y` [B, ...] as out_dir/<name>.npy in float32.  If it is larger than DUMP_MAX_BYTES, only the
    windows rows = sorted(default_rng(0).choice(B, n, replace=False)) are saved, n as many as fit: the
    same rows for the same B, whichever build wrote the file."""
    y = y.detach()
    n = min(y.shape[0], DUMP_MAX_BYTES // (4 * max(1, math.prod(y.shape[1:]))))
    if n < y.shape[0]:
        rows = np.sort(np.random.default_rng(0).choice(y.shape[0], n, replace=False))
        y = y[torch.from_numpy(rows).to(y.device)]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, f"{name}.npy"), y.to(torch.float32).cpu().numpy())


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region: one streaming
    `nvidia-smi -lms 20` process started ahead of time; `mark_start()` / `mark_stop()` bracket the
    region and only samples stamped inside it are summarised."""

    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.t0 = self.t1 = None
        self.rows = []

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index),
                 "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            time.sleep(0.5)  # let it start streaming before the timed region begins
        except OSError:
            self.proc = None
        return self

    def mark_start(self):
        self.t0 = time.time()

    def mark_stop(self):
        self.t1 = time.time()

    def __exit__(self, *a):
        self.rows = []
        if self.proc is None:
            return
        time.sleep(0.05)
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=10)
        except subprocess.TimeoutExpired:
            self.proc.kill()
            out, _ = self.proc.communicate()
        import datetime

        for line in out.splitlines():
            parts = [v.strip() for v in line.split(",")]
            if len(parts) < 8:
                continue
            try:
                ts = datetime.datetime.strptime(parts[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
            except ValueError:
                continue
            self.rows.append((ts, parts[1:]))

    def summary(self):
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        lo = (self.t0 or 0) - 0.02
        hi = (self.t1 or 1e18) + 0.02
        inside = [r for ts, r in self.rows if lo <= ts <= hi]
        where = "timed region"
        if not inside:  # region shorter than the sampling period: fall back to the nearest samples
            inside = [r for _, r in sorted(self.rows, key=lambda x: abs(x[0] - (self.t0 or 0)))[:3]]
            where = "nearest to timed region"
        sm, mx, pw, reasons = [], [], [], set()
        for r in inside:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
                pw.append(float(r[2]))
            except (ValueError, IndexError):
                continue
            for n, v in zip(names, r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_min_mhz": float(min(sm)), "sm_max_mhz": float(max(mx)),
                "power_w_median": float(np.median(pw)), "reasons": sorted(reasons), "samples": len(sm),
                "window": where, "seconds": (self.t1 or 0) - (self.t0 or 0)}


def ncu_traffic_bytes(kernel_name: str, algorithmic_bytes: float):
    """dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of `kernel_name`, from the committed
    ncu capture of this very workload (profiles/r02_ncu_summary.json, written by
    scripts/make_profile_summary.py from `ncu --set full` of scripts/profile_step.py at B=4096, S=34).
    The kernel is matched by its full demangled base name; a capture whose traffic is not within
    [0.5, 3] x the algorithmic bytes is rejected (it would be another workload's launch).
    Returns (bytes or None, note)."""
    summ = {"kernels": []}
    for path in (NCU_SUMMARY, NCU_SUMMARY.replace("r02_", "r02_tensor_")):   # FP32-path / tensor-path captures
        try:
            with open(path) as f:
                part = json.load(f)
            summ["kernels"] += part.get("kernels", [])
            summ.setdefault("command", part.get("command", ""))
        except (OSError, ValueError):
            continue
    if not summ["kernels"]:
        return None, "no committed capture (profiles/r02_ncu_summary.json)"
    scale = {"Gbyte": 1e9, "Mbyte": 1e6, "Kbyte": 1e3, "byte": 1.0}
    for k in summ.get("kernels", []):
        base = k["kernel"].split("(")[0].replace("void ", "").replace("wg::", "").strip()
        if base != kernel_name:
            continue
        try:
            t = (k["dram__bytes_read.sum"] * scale[k["dram__bytes_read.sum.unit"]]
                 + k["dram__bytes_write.sum"] * scale[k["dram__bytes_write.sum.unit"]])
        except KeyError:
            continue
        if not 0.5 <= t / algorithmic_bytes <= 3.0:
            return None, f"capture rejected: {t:.3e} B is not within [0.5, 3] x algorithmic {algorithmic_bytes:.3e} B"
        return t, f"profiles/r02_ncu_summary.json ({summ.get('command', '')})"
    return None, f"kernel {kernel_name} not in profiles/r02_ncu_summary.json"


# --------------------------------------------------------------------------------------------------
# the reference's own forward (oracle/_ref when built, else the oracle's torch port)
# --------------------------------------------------------------------------------------------------
def reference_callable(sd, dims, device):
    """Returns (batched_fn(adj, x), as_written_fn(adj, x) or None, kind)."""
    from oracle.ref_loader import reference_forward_as_written, reference_forward_batched, reference_model

    model = reference_model(sd, dims, device)
    if model is not None:
        return (lambda adj, x: reference_forward_batched(model, adj, x),
                lambda adj, x: reference_forward_as_written(model, adj, x), "reference")
    if str(device) != "cpu":
        return None, None, "unavailable"
    from oracle import gcn_gru_forward_torch

    return (lambda adj, x: gcn_gru_forward_torch(adj, x, sd)), None, "port"


def cpu_reference_seq_per_s(sd, adj32, n_seq: int, min_seconds: float, max_reps: int, seed: int = 0):
    """The reference forward on all host threads.  Returns (sequences/s, threads, reps, seconds, kind)."""
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    fn, _, kind = reference_callable(sd, (F, F, F, I, H), "cpu")
    x = torch.rand((n_seq, T, S, F), generator=torch.Generator().manual_seed(seed))
    fn(adj32, x[: max(1, n_seq // 8)])  # warm-up (thread pool, allocator)
    reps, t0 = 0, time.perf_counter()
    while True:
        fn(adj32, x)
        reps += 1
        dt = time.perf_counter() - t0
        if dt >= min_seconds or reps >= max_reps:
            break
    return n_seq * reps / dt, threads, reps, dt, kind


def run_reference(args, rank: int):
    """Reference arm: the reference's own CPU forward of the path on the box's host cores (rank 0 only),
    on the full configs[1] step (4096 windows per step)."""
    if rank != 0:
        return
    sd, latlon = load_workload()
    from oracle import dense_graph_f64

    adj32 = torch.from_numpy(dense_graph_f64(latlon).astype(np.float32))
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    fn, _, kind = reference_callable(sd, (F, F, F, I, H), "cpu")
    n_seq = args.ref_seqs
    x = torch.rand((n_seq, T, S, F), generator=torch.Generator().manual_seed(0))
    for _ in range(max(1, min(args.warmup, 2))):
        fn(adj32, x[: min(256, n_seq)])
    t0 = time.perf_counter()
    for _ in range(args.steps):
        y = fn(adj32, x)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_output(args.dump_outputs, "y", y)
    value = n_seq * args.steps / dt
    what = ("the reference's own GraphConvLayer / nn.GRU modules (oracle/_ref, unmodified), batched through its "
            "sub-modules" if kind == "reference" else "the oracle's torch-CPU port (oracle/_ref absent)")
    sample = f"{n_seq} of the {B_PER_GPU} sequences of each step, {args.steps} steps, {what}, fp32, {threads} threads"
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "34-station GCN-GRU forward (wind_gnn_34.pth), T=168, batch 4096 per step "
                               "(BASELINE.json configs[1]), CPU", "S": S, "T": T, "batch_per_step": n_seq,
                   "same_config": n_seq == B_PER_GPU},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }), flush=True)


# --------------------------------------------------------------------------------------------------
# helpers shared by the GPU legs
# --------------------------------------------------------------------------------------------------
class Ctx:
    def __init__(self, rank, world, local_rank):
        self.rank, self.world, self.local_rank = rank, world, local_rank
        self.dev = torch.device("cuda", local_rank)
        self.dist = None

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()
        torch.cuda.synchronize(self.dev)

    def max_over_ranks(self, v: float) -> float:
        from windgnn_b200.shard import max_over_ranks

        return max_over_ranks(v, self.dev)


def timed_events(ctx: Ctx, fn, steps: int, warmup: int, clocks: ClockSampler | None = None) -> float:
    """`warmup` untimed calls, then `steps` timed calls between a barrier + synchronize on both sides;
    CUDA events on the launching stream; returns the max over ranks in ms."""
    for _ in range(warmup):
        fn()
    ctx.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ctx.barrier()
    if clocks is not None:
        clocks.mark_start()
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    ctx.barrier()
    if clocks is not None:
        clocks.mark_stop()
    return ctx.max_over_ranks(e0.elapsed_time(e1))


def scaled_leg(ctx: Ctx, which: str, steps: int, warmup: int, lib_peak: float, batch4096: int = 256,
               dump_dir: str | None = None):
    """One of the other BASELINE configs as a sub-object (device-resident throughput; parity for these shapes
    is in tests/test_parity_gpu.py).
      fwd7     configs[0]: shipped 7-station checkpoint, 4096 windows per GPU (weak)
      fwd34_1m configs[2]: 2^20 windows in total, rank r owns a contiguous 1/world of them, streamed through the
               library in resident pieces of <= 131072 windows (one synthetic piece reused) (strong)
      fwd4096  configs[3]: 4096-station kNN(8) graph, GCN_GRU(13,128,13,53248,128), T=24, 256 windows per GPU (weak)
    With `dump_dir`, rank 0 saves the output of the last timed step (fwd34_1m: of its last piece) there."""
    import windgnn_b200
    from windgnn_b200.shard import shard_range

    dev, rank, world = ctx.dev, ctx.rank, ctx.world
    gen = torch.Generator(device=dev).manual_seed(99 + rank)
    last = {}
    if which == "fwd34_1m":
        sd, latlon = load_workload()
        model = windgnn_b200.GCN_GRU(F, F, F, I, H)
        model.load_state_dict(sd, strict=True)
        adj = windgnn_b200.build_graph_from_latlon(latlon, device=dev, dtype=torch.float32)
        total = 1 << 20
        lo, hi = shard_range(total, rank, world)
        piece = min(hi - lo, 131072)
        n_pieces = (hi - lo + piece - 1) // piece
        x = torch.rand((piece, T, S, F), generator=gen, device=dev)
        Sx, Tx, fl, by, scaling, units = S, T, FLOP_PER_SEQ, BYTES_PER_SEQ, "strong", total
        name = ("34-station forward (wind_gnn_34.pth), T=168, 2^20 windows sharded contiguously over the GPUs, "
                f"{n_pieces} resident piece(s) of {piece} per GPU (BASELINE.json configs[2])")

        def step():
            for _ in range(n_pieces):
                last["y"] = model(adj, x)
    elif which == "fwd7":
        sd, latlon = load_workload(7)
        model = windgnn_b200.GCN_GRU(F, F, F, 13 * 7, 21)
        model.load_state_dict(sd, strict=True)
        adj = windgnn_b200.build_graph_from_latlon(latlon, device=dev, dtype=torch.float32)
        B7 = 4096
        x = torch.rand((B7, T, 7, F), generator=gen, device=dev)
        Sx, Tx, scaling, units = 7, T, "weak", world * B7
        fl, by = flop_per_seq(7, T, F, F, F, 21), bytes_per_seq(7, T, F, 21)
        name = "7-station forward (wind_gnn_7.pth), T=168, 4096 windows per GPU (BASELINE.json configs[0], batched)"

        def step():
            last["y"] = model(adj, x)
    else:
        S4, Fh4, H4, T4, B4 = 4096, 128, 128, 24, batch4096
        torch.manual_seed(4)
        model = windgnn_b200.GCN_GRU(F, Fh4, F, F * S4, H4)
        with torch.no_grad():
            model.conv1.weight.mul_(0.05)
            model.conv2.weight.mul_(0.05)
        ll = windgnn_b200.synthetic_coordinates(S4, seed=0, device=dev).cpu().numpy()
        adj = windgnn_b200.knn_graph_csr_from_latlon(ll, k=8, device=dev)   # CSR straight from the kNN builder
        nnz = adj.nnz
        x = torch.rand((B4, T4, S4, F), generator=gen, device=dev)
        Sx, Tx, scaling, units = S4, T4, "weak", world * B4
        fl, by = flop_per_seq(S4, T4, F, Fh4, F, H4, nnz=nnz), bytes_per_seq(S4, T4, F, H4)
        name = (f"synthetic 4096-station kNN(k=8) graph (nnz {nnz}, CSR from the GPU builder), "
                f"GCN_GRU(13,128,13,53248,128), T=24, {B4} windows per GPU (BASELINE.json configs[3], SURVEY 8(d) "
                "variant C)")

        def step():
            last["y"] = model(adj, x)
    model = model.to(dev).eval()
    with torch.no_grad():
        ms = timed_events(ctx, step, steps, warmup)
    if dump_dir and rank == 0:
        dump_output(dump_dir, "y", last["y"])
    value = units * steps / (ms * 1e-3)
    tfl = fl * value / world / 1e12
    tensor = None
    if which == "fwd4096":   # the same configuration on the tensor path (projection + recurrence on tcgen05)
        model.precision = "tensor"
        with torch.no_grad():
            ms_t = timed_events(ctx, step, steps, warmup)
        model.precision = "fp32"
        tensor = {"value": units * steps / (ms_t * 1e-3), "ms_per_step": ms_t / steps,
                  "precision": "tensor (tcgen05 projection and recurrence, split fp16 operands); the CSR GCN stays FP32"}
    out = {"workload": name, "value": value, "unit": UNIT, "ms_per_step": ms / steps, "steps": steps, "warmup": warmup,
           "scaling": scaling, "S": Sx, "T": Tx, "station_sequence_predictions_per_s": value * Sx,
           "tflops_per_gpu": tfl, "frac_fp32": tfl / lib_peak if lib_peak > 0 else None,
           "hbm_gbs_algorithmic_per_gpu": by * value / world / 1e9, "flop_per_seq": fl}
    if tensor is not None:
        out["tensor_path"] = tensor
    del x, model, adj, last
    torch.cuda.empty_cache()
    return out


def h2d_ceiling(ctx: Ctx, xh: torch.Tensor, oh: torch.Tensor, reps: int = 4):
    """What the host can deliver: every rank copies its pinned step input host->device (and, concurrently on a
    second stream, a step output device->host) `reps` times, no compute; aggregate GB/s over all ranks."""
    dev = ctx.dev
    xd = torch.empty(xh.shape, dtype=xh.dtype, device=dev)
    od = torch.empty(oh.shape, dtype=oh.dtype, device=dev)
    s_in, s_out = torch.cuda.Stream(dev), torch.cuda.Stream(dev)

    def run(duplex: bool):
        ctx.barrier()
        t0 = time.perf_counter()
        for _ in range(reps):
            with torch.cuda.stream(s_in):
                xd.copy_(xh, non_blocking=True)
            if duplex:
                with torch.cuda.stream(s_out):
                    oh.copy_(od, non_blocking=True)
        s_in.synchronize()
        s_out.synchronize()
        return ctx.max_over_ranks(time.perf_counter() - t0)

    run(False)
    dt_h2d = run(False)
    dt_dup = run(True)
    nb = xh.numel() * 4
    del xd, od
    return {"h2d_gbs_aggregate": ctx.world * nb * reps / dt_h2d / 1e9,
            "h2d_gbs_aggregate_with_concurrent_d2h": ctx.world * nb * reps / dt_dup / 1e9,
            "step_ms_floor": 1e3 * dt_dup / reps,
            "what": f"{ctx.world} rank(s) x {reps} x cudaMemcpyAsync of the {nb / 1e9:.2f} GB step input from pinned "
                    "host memory, concurrently, no compute (second figure: with the step output going back on "
                    "another stream)"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20, help="timed steps (one forward of the batch each)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=B_PER_GPU, help="sequences per GPU per step")
    ap.add_argument("--min-seconds", type=float, default=2.0,
                    help="minimum length of the timed region of the host-buffer (e2e) leg")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-tensor-path", action="store_true")
    ap.add_argument("--no-gpu-eager", action="store_true")
    ap.add_argument("--no-scaled", action="store_true")
    ap.add_argument("--no-train-step", action="store_true")
    ap.add_argument("--precision", default="fp32", choices=["fp32", "tensor", "tf32x3"],
                    help="fp32: every contraction as FP32 FMA; tensor: projection and recurrence on tcgen05 (split fp16 operands)")
    ap.add_argument("--ref-seqs", type=int, default=B_PER_GPU,
                    help="sequences per step of the reference arm (default: the full configs[1] step)")
    ap.add_argument("--workload", default="fwd34", choices=["fwd34", "fwd34_1m", "fwd4096", "fwd7"],
                    help="fwd34: BASELINE configs[1] (default, the contract line, carries the others as `scaled`); "
                         "the other names print that config alone")
    ap.add_argument("--train-batch", type=int, default=512,
                    help="windows per GPU of the training-step measurement (BASELINE.json configs[4]: 4096 over 8 GPUs)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="save the output of the last timed step as DIR/y.npy (float32; above 64 MB a fixed sample "
                         "of windows)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference(args, rank)
        return

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — windgnn_b200 has no CPU fallback")
    import windgnn_b200
    from windgnn_b200 import _lib

    lib = _lib.load()
    torch.cuda.set_device(local_rank)
    ctx = Ctx(rank, world, local_rank)
    dev = ctx.dev
    if world > 1:
        import torch.distributed as dist

        # keep stdout to the one JSON line: NCCL prints its version banner there at VERSION level
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"
        dist.init_process_group("nccl", device_id=dev)
        ctx.dist = dist

    warmup = max(args.warmup, 3)
    steps = args.steps
    Bg = args.batch
    ffma_peak = lib.wg_measure_ffma_tflops(local_rank, 10)

    if args.workload != "fwd34":
        leg = scaled_leg(ctx, args.workload, steps, warmup, ffma_peak, Bg if Bg != B_PER_GPU else 256, args.dump_outputs)
        if rank == 0:
            print(json.dumps({
                "metric": METRIC, "value": leg["value"], "unit": UNIT, "n_gpus": world, "steps": steps,
                "warmup": warmup, "ms_per_step": leg["ms_per_step"], "higher_is_better": True,
                "scaling": leg["scaling"], "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": leg["workload"], "S": leg["S"], "T": leg["T"],
                           "l2_policy": "inputs larger than L2"},
                "roofline": {"bound": "fp32", "achieved": leg["tflops_per_gpu"], "peak": ffma_peak, "unit": "TFLOP/s",
                             "frac": leg["frac_fp32"], "scope": "whole path, per GPU, algorithmic FLOPs"},
                "scaled": {args.workload: leg}}), flush=True)
        if ctx.dist is not None:
            ctx.dist.barrier()
            ctx.dist.destroy_process_group()
        return

    sd, latlon = load_workload()
    model = windgnn_b200.GCN_GRU(F, F, F, I, H)
    model.load_state_dict(sd, strict=True)
    model = model.to(dev).eval()
    model.precision = args.precision
    flags = model._flags()
    adj = windgnn_b200.build_graph_from_latlon(latlon, device=dev, dtype=torch.float32)
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    x = torch.rand((Bg, T, S, F), generator=gen, device=dev)  # 1.22 GB at B=4096: larger than the 126 MB L2

    # ---------------- device-resident throughput (`value`) ----------------
    holder = {}

    def one_step():
        holder["y"] = model(adj, x)

    with torch.no_grad():
        with ClockSampler(local_rank) as clocks:
            ms = timed_events(ctx, one_step, steps, warmup, clocks)
    y = holder["y"]
    if args.dump_outputs and rank == 0:
        dump_output(args.dump_outputs, "y", y)
    value = world * Bg * steps / (ms * 1e-3)
    n_chunks = (Bg + 148 * 32 - 1) // (148 * 32)
    launches_per_pass = 1 + 3 * n_chunks  # pack + (gcn, inproj, recur) per internal chunk

    # ---------------- the opt-in tensor-core path, same workload, same timing rules ----------------
    tensor_path = None
    if args.precision == "fp32" and not args.no_tensor_path:
        model.precision = "tensor"
        try:
            with torch.no_grad():
                def tc_step():
                    holder["yt"] = model(adj, x)

                ms_t = timed_events(ctx, tc_step, steps, 2)
            yt = holder["yt"]
            err = float((yt - y).abs().max() / y.abs().max())
            tensor_path = {"precision": "tensor-core path (tcgen05, error-compensated split operands, fp32 accumulate)",
                           "value": world * Bg * steps / (ms_t * 1e-3), "unit": UNIT,
                           "ms_per_pass": ms_t / steps,
                           "max_abs_diff_vs_fp32_path_normalised": err, "parity_bar": 1e-5}
            del yt
            holder.pop("yt", None)
        finally:
            model.precision = args.precision
    ctx.barrier()

    # ---------------- the reference's own call pattern: one window per call (src/main.py:101-103) ----------
    batch1 = None
    if rank == 0:
        with torch.no_grad():
            x1 = x[:1]
            for _ in range(5):
                model(adj, x1)
            torch.cuda.synchronize(dev)
            b0e, b1e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            b0e.record()
            for _ in range(50):
                model(adj, x1)
            b1e.record()
            torch.cuda.synchronize(dev)
        batch1 = {"gpu_ms_per_window": b0e.elapsed_time(b1e) / 50,
                  "what": "model(adj_matrix, batch_x) with batch_x [1,168,34,13] resident on the GPU, 50 calls back to back"}
    ctx.barrier()

    # ---------------- PyTorch eager on the same B200: the reference's own classes (cuBLAS + cuDNN GRU) ----------
    gpu_eager = None
    if rank == 0 and not args.no_gpu_eager:
        try:
            fn_b, fn_w, kind = reference_callable(sd, (F, F, F, I, H), dev)
            if fn_b is None:
                gpu_eager = {"unavailable": "oracle/_ref not built (the reference classes are needed on the GPU)"}
            else:
                def eager_batched():
                    for _ in range(2):
                        ye = fn_b(adj, x)
                    torch.cuda.synchronize(dev)
                    g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    reps_e = 5
                    g0.record()
                    for _ in range(reps_e):
                        ye = fn_b(adj, x)
                    g1.record()
                    torch.cuda.synchronize(dev)
                    return g0.elapsed_time(g1) / reps_e, float((ye - y).abs().max() / ye.abs().max())

                with torch.no_grad():
                    # PyTorch's defaults, i.e. what `python src/main.py` gets on this GPU: fp32 matmuls, but the
                    # cuDNN GRU is allowed TF32 (torch.backends.cudnn.allow_tf32 defaults to True)
                    ms_d, err_d = eager_batched()
                    for _ in range(3):
                        fn_w(adj, x[:4])
                    torch.cuda.synchronize(dev)
                    g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    g0.record()
                    fn_w(adj, x[:64])
                    g1.record()
                    torch.cuda.synchronize(dev)
                    ms_w = g0.elapsed_time(g1) / 64
                    # strict fp32 (the precision this library's FP32 path is held to)
                    prev = torch.backends.cudnn.allow_tf32
                    torch.backends.cudnn.allow_tf32 = False
                    try:
                        ms_e, err_e = eager_batched()
                    finally:
                        torch.backends.cudnn.allow_tf32 = prev
                gpu_eager = {"kind": kind, "value": Bg / (ms_e * 1e-3), "unit": UNIT, "ms_per_pass": ms_e,
                             "batch": Bg, "ours_vs_eager_normalised_max_diff": err_e,
                             "pytorch_defaults": {"value": Bg / (ms_d * 1e-3), "ms_per_pass": ms_d,
                                                  "ours_vs_eager_normalised_max_diff": err_d,
                                                  "note": "torch.backends.cudnn.allow_tf32 = True (default): the cuDNN GRU "
                                                          "may use TF32"},
                             "as_written_ms_per_window": ms_w,
                             "what": "the reference's GraphConvLayer / nn.GRU modules (oracle/_ref, unmodified) in PyTorch "
                                     "eager on this GPU (cuBLAS + cuDNN GRU), strict fp32 (cudnn.allow_tf32 = False): batched "
                                     "through its sub-modules at the bench batch; `as_written` = one model(adj_matrix, batch_x) "
                                     "call per window (main.py:101-102) with PyTorch's defaults"}
            torch.cuda.empty_cache()
        except Exception as e:  # the comparator must never take the bench line down
            gpu_eager = {"unavailable": f"{type(e).__name__}: {e}"[:300]}
    ctx.barrier()

    # ---------------- training step (BASELINE.json configs[4]): fwd + MSE + bwd + all-reduce + Adam ----------
    train_step = None
    if not args.no_train_step:
        from windgnn_b200 import train as wtrain

        tmodel = windgnn_b200.GCN_GRU(F, F, F, I, H)
        tmodel.load_state_dict(sd, strict=True)
        tmodel = tmodel.to(dev).train()
        trainer = wtrain.Trainer(tmodel, adj, lr=1e-3)   # main.py:45,52
        Bt = args.train_batch
        xt = x[:Bt] if Bt <= Bg else torch.rand((Bt, T, S, F), generator=gen, device=dev)
        yt_ = torch.rand((Bt, T, H), generator=gen, device=dev)
        hold_t = {}

        def tstep():
            hold_t["l"] = trainer.step(xt, yt_)

        tr_steps = max(steps, 50)
        ms_tr = timed_events(ctx, tstep, tr_steps, warmup)
        train_step = {"metric": "gcn_gru_train_step_sequences_per_s", "value": world * Bt * tr_steps / (ms_tr * 1e-3),
                      "unit": UNIT, "ms_per_step": ms_tr / tr_steps, "steps": tr_steps, "batch_per_gpu": Bt,
                      "global_batch": Bt * world, "loss_after": float(hold_t["l"].item()),
                      "what": "forward (gates saved) + MSE + BPTT/GEMM/GCN backward + "
                              + ("NCCL sum all-reduce of one flat 167,440-float gradient bucket + " if world > 1 else "")
                              + "fused Adam, all inside the timed region; FP32",
                      "gpu_launches_per_step": 22 + (1 if world > 1 else 0)}
        del trainer, tmodel, xt, yt_
    ctx.barrier()

    # ---------------- per-kernel timing for the roofline (rank 0's GPU, same stream) -------------
    dims = (T, S, F, F, F, H)
    stage_ms = {}
    if rank == 0:
        Bc = min(Bg, 148 * 32)
        nbytes = lib.wg_gcn_gru_workspace_bytes(Bc, *dims, Bc, flags)
        ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        out = torch.empty((Bc, T, H), device=dev)
        p = [t.detach().contiguous() for t in (
            model.conv1.weight, model.conv1.bias, model.conv2.weight, model.conv2.bias,
            model.gru.weight_ih_l0, model.gru.weight_hh_l0, model.gru.bias_ih_l0, model.gru.bias_hh_l0)]
        st = torch.cuda.current_stream(dev).cuda_stream
        xs = x[:Bc]
        calls = {
            "pack": lambda: lib.wg_stage_pack_f32(*(t.data_ptr() for t in p[4:]), *dims, Bc, flags, ws.data_ptr(), nbytes, local_rank, st),
            "gcn": lambda: lib.wg_stage_gcn_f32(adj.data_ptr(), xs.data_ptr(), *(t.data_ptr() for t in p[:4]), Bc, *dims, Bc, flags, ws.data_ptr(), nbytes, local_rank, st),
            "inproj": lambda: lib.wg_stage_inproj_f32(Bc, *dims, Bc, flags, ws.data_ptr(), nbytes, local_rank, st),
            "recur": lambda: lib.wg_stage_recur_f32(out.data_ptr(), Bc, *dims, Bc, flags, ws.data_ptr(), nbytes, local_rank, st),
        }
        for name in ("pack", "gcn", "inproj", "recur"):
            for _ in range(3):
                _lib.check(calls[name]())
            torch.cuda.synchronize(dev)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            reps = 20
            a.record()
            for _ in range(reps):
                _lib.check(calls[name]())
            b.record()
            torch.cuda.synchronize(dev)
            stage_ms[name] = a.elapsed_time(b) / reps
        del ws, out
    ctx.barrier()

    # ---------------- end-to-end through the host-buffer entry point ----------------
    e2e = None
    if not args.no_e2e:
        xh = torch.empty((Bg, T, S, F), dtype=torch.float32, pin_memory=True)
        xh.copy_(x)
        oh = torch.empty((Bg, T, H), dtype=torch.float32, pin_memory=True)
        model.chunk = 256  # pipeline granularity: H2D / compute (two lanes) / D2H of consecutive chunks overlap

        def e2e_run(n):
            ctx.barrier()
            t0 = time.perf_counter()
            for _ in range(n):
                model.forward_host(adj, xh, oh)  # blocks until `oh` is complete
            torch.cuda.synchronize(dev)
            return ctx.max_over_ranks(time.perf_counter() - t0)

        with torch.no_grad():
            dt2 = e2e_run(2)   # warm-up, and the estimate the step count is sized from
            e2e_steps = max(steps, min(200, math.ceil(args.min_seconds / (dt2 / 2))))
            dt = e2e_run(e2e_steps)
            e2e = {"value": world * Bg * e2e_steps / dt, "unit": UNIT,
                   "h2d_bytes_per_step": Bg * T * S * F * 4, "d2h_bytes_per_step": Bg * T * H * 4,
                   "steps": e2e_steps, "ms_per_step": 1e3 * dt / e2e_steps, "pipeline_chunk": 256, "compute_lanes": 2,
                   "timing": "host wall clock around the blocking calls (the public API returns when the host output "
                             "buffer is complete), max over ranks"}
            # what the reference's evaluation loop needs (main.py:101-116): de-normalised last step only
            ph = torch.empty((Bg, H), dtype=torch.float32, pin_memory=True)
            ctx.barrier()
            t0 = time.perf_counter()
            for _ in range(max(3, e2e_steps // 4)):
                model.forward_host(adj, xh, ph, last_step_range=(0.0, 83.6))
            torch.cuda.synchronize(dev)
            dtp = ctx.max_over_ranks(time.perf_counter() - t0) / max(3, e2e_steps // 4)
            e2e["last_step_only"] = {"value": world * Bg / dtp, "ms_per_step": 1e3 * dtp, "d2h_bytes_per_step": Bg * H * 4,
                                     "what": "wg_gcn_gru_predict_host_f32: only the de-normalised last timestep "
                                             "[B, 3S] returns to the host"}
            del ph
            if tensor_path is not None:
                model.precision = "tensor"
                try:
                    e2e_run(2)
                    dtt = e2e_run(e2e_steps)
                    tensor_path["e2e_value"] = world * Bg * e2e_steps / dtt
                    tensor_path["e2e_ms_per_step"] = 1e3 * dtt / e2e_steps
                finally:
                    model.precision = args.precision
            ceil_ = h2d_ceiling(ctx, xh, oh)
            ceil_["seq_per_s_ceiling"] = world * Bg / (ceil_["step_ms_floor"] * 1e-3)
            ceil_["e2e_frac_of_ceiling"] = e2e["value"] / ceil_["seq_per_s_ceiling"]
            e2e["h2d_ceiling"] = ceil_
        model.chunk = 0
        del xh, oh
    ctx.barrier()

    # ---------------- the other BASELINE configs, as sub-objects of the default line ----------------
    scaled = None
    if not args.no_scaled:
        scaled = {}
        del x, y
        holder.clear()
        torch.cuda.empty_cache()
        for which, st_, wu_ in (("fwd7", 20, 3), ("fwd4096", 10, 3), ("fwd34_1m", 1, 1)):
            try:
                with torch.no_grad():
                    scaled[which] = scaled_leg(ctx, which, st_, wu_, ffma_peak)
            except Exception as e:
                scaled[which] = {"unavailable": f"{type(e).__name__}: {e}"[:300]}
    ctx.barrier()

    if rank == 0:
        peaks = {}
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
                peaks = json.load(f)
        except Exception:
            pass
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        hbm_src = "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback (B200_PROFILING.md)"
        Bc = min(Bg, 148 * 32)
        rows = Bc * T
        inproj_flops = FLOP_IH * rows
        inproj_bytes = rows * (I + 3 * H) * 4        # U read once + GI written once
        inproj_tflops = inproj_flops / (stage_ms["inproj"] * 1e-3) / 1e12
        nominal_peak = 148 * 128 * 2 * float(peaks.get("sm_max_mhz", 1965.0)) * 1e6 / 1e12
        path_tflops = FLOP_PER_SEQ * Bg * steps / (ms * 1e-3) / 1e12  # per GPU
        hbm_gbs = BYTES_PER_SEQ * Bg * steps / (ms * 1e-3) / 1e9      # per GPU, algorithmic
        kname = "inproj_kernel" if flags == 0 else "inproj_tc2_kernel"
        traffic, traffic_note = ncu_traffic_bytes(kname, inproj_bytes)
        stage_flops = {"gcn": 2 * (2 * S * S * F + 2 * S * F * F) * rows, "inproj": inproj_flops,
                       "recur": 2 * H * 3 * H * rows}
        roofline = {
            "bound": "fp32", "kernel": (f"{kname} (GRU input projection, FFMA2 GEMM)" if flags == 0 else
                                        f"{kname} (GRU input projection on tcgen05; fraction is of the FP32 FMA "
                                        "peak the FP32 path is bound by)"),
            "achieved": inproj_tflops, "peak": ffma_peak, "unit": "TFLOP/s", "frac": inproj_tflops / ffma_peak,
            "peak_source": "FFMA microbenchmark measured live on this GPU (wg_measure_ffma_tflops); "
                           "MEASURED_PEAKS.json has no FP32 figure",
            "peak_nominal": nominal_peak, "frac_of_nominal": inproj_tflops / nominal_peak,
            "traffic": traffic, "traffic_unit": "bytes per launch (ncu dram read+write)", "traffic_source": traffic_note,
            "algorithmic_bytes_per_launch": inproj_bytes, "algorithmic_flops_per_launch": inproj_flops,
            "kernel_ms": stage_ms,
            "kernel_frac_fp32": {k: stage_flops[k] / (stage_ms[k] * 1e-3) / 1e12 / ffma_peak for k in stage_flops},
            "path": {"achieved": path_tflops, "frac_fp32": path_tflops / ffma_peak,
                     "frac_fp32_of_nominal": path_tflops / nominal_peak,
                     "hbm_gbs": hbm_gbs, "hbm_peak": hbm_peak, "hbm_peak_source": hbm_src,
                     "frac_hbm": hbm_gbs / hbm_peak, "flop_per_seq": FLOP_PER_SEQ, "bytes_per_seq": BYTES_PER_SEQ},
        }
        cpu = None
        if not args.no_cpu_baseline and world == 1:  # reported on rank 0 at N=1 only
            adj_cpu = adj.cpu()
            v, threads, reps, secs, kind = cpu_reference_seq_per_s(sd, adj_cpu, n_seq=2048, min_seconds=12.0, max_reps=40)
            cpu = {"value": v, "unit": UNIT, "cores": threads, "kind": kind,
                   "sample": f"{reps} x 2048 sequences of the same workload in {secs:.1f} s, fp32, "
                             + ("the reference's own modules (oracle/_ref)" if kind == "reference" else "torch-CPU port")}
            if batch1 is not None:   # the reference called the way it calls its model: one window at a time
                _, fn_w, _ = reference_callable(sd, (F, F, F, I, H), "cpu")
                if fn_w is not None:
                    x1c = torch.rand((8, T, S, F))
                    fn_w(adj_cpu, x1c[:3])
                    t0 = time.perf_counter()
                    fn_w(adj_cpu, x1c)
                    fn_w(adj_cpu, x1c)
                    batch1["cpu_reference_ms_per_window"] = (time.perf_counter() - t0) / 16 * 1e3
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": warmup,
            "ms_per_step": ms / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32" if flags == 0 else "f32 (tensor-core contractions on error-compensated split operands, fp32 accumulate)",
            "data": "synthetic",
            "config": {"precision": args.precision,
                       "workload": "34-station GCN-GRU forward (wind_gnn_34.pth), T=168, batch 4096 per GPU "
                                   "(BASELINE.json configs[1])", "S": S, "T": T, "batch_per_gpu": Bg,
                       "global_batch": Bg * world, "parallelism": f"sequence-sharded x{world}, no collective",
                       "l2_policy": "inputs (1.22 GB per pass) larger than L2",
                       "station_sequence_predictions_per_s": value * S},
            "clocks": clocks.summary(), "e2e": e2e, "gpu_launches": launches_per_pass * steps,
            "roofline": roofline, "cpu_baseline": cpu, "gpu_eager": gpu_eager, "tensor_path": tensor_path,
            "train_step": train_step, "batch1": batch1, "scaled": scaled,
        }
        print(json.dumps(line), flush=True)
    if ctx.dist is not None:
        ctx.dist.barrier()
        ctx.dist.destroy_process_group()


if __name__ == "__main__":
    main()
