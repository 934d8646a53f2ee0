#!/usr/bin/env python
"""Measure the row-sparse update kernel and row-sparse embedding training on a B200.

    python scripts/bench_row_sparse.py kernel [--launches 200]
    python scripts/bench_row_sparse.py train  [--steps 12] [--rounds 2] [--gpus 2]

kernel  CUDA-event time of ps_launch_update_rows over many launches: a union of 8192 rows of
        D = 4096 out of a 65536-row table (3 GiB of fp32 state, far larger than the 126 MB L2),
        W = 4 fp8 slots, fan-out 4 bf16 destinations. Bytes per launch come from the model below;
        the rate is given as a fraction of the 6571 GB/s copy roofline in README.md.
train   examples/train_llama_ps.py at Llama-1b shapes (vocab 128256, seq 8192) on --gpus GPUs, dense
        embedding and --sparse-embedding alternating `rounds` times in this one call; reports the
        median step time after 2 warm-up steps and the pushed wire bytes per step.
Every result line carries the GPU name and power limit, read in the same call.
"""
from __future__ import annotations

import argparse
import json
import os
import re
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

COPY_ROOFLINE_GBS = 6571.0  # README.md: measured device-to-device copy rate on B200


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def kernel_bytes(W, R, U, D, outs, wire_bytes_per_elem=1 + 1 / 32):
    """W slots of R rows (ids + fp8 values) + 24 B/element of fp32 state (read + write master, m, v) for
    the U rows of the union + 2 B/element per bf16 destination"""
    return W * (R * 4 + R * D * wire_bytes_per_elem) + 24 * U * D + outs * U * D * 2


def bench_kernel(args):
    import torch

    import pslite_b200

    assert torch.cuda.is_available(), "the kernel benchmark needs a GPU"
    C = pslite_b200.native()
    dev = torch.device("cuda", 0)
    rows, D, U, W, n_outs = 65536, 4096, 8192, 4, 4
    n = rows * D
    g = torch.Generator(device=dev).manual_seed(0)
    master = torch.randn(n, device=dev, generator=g)
    m = torch.zeros(n, device=dev)
    v = torch.zeros(n, device=dev)
    outs = [torch.empty(n, dtype=torch.bfloat16, device=dev) for _ in range(n_outs)]
    scratch = torch.zeros(C.rows_scratch_bytes(rows, W), dtype=torch.uint8, device=dev)
    union = torch.randperm(rows, device=dev, generator=g)[:U]
    slots, counts = [], []
    for w in range(W):  # every slot holds all U rows: the union is U, each row summed over W slots
        R = U
        nb = C.rows_slot_bytes(R, D, C.GRAD_FP8BLOCK)
        buf = torch.zeros(nb, dtype=torch.uint8, device=dev)
        buf[:4 * R].view(torch.int32).copy_(union.sort().values.to(torch.int32))
        off = (R + 3) // 4 * 16
        vals = torch.randn(R * D, device=dev, generator=g) * 1e-3
        C.copy_codec(buf[off:], vals, C.CODEC_F32_TO_FP8BLOCK, 1.0)
        slots.append(buf)
        counts.append(R)

    def launch(step):
        C.fused_update_rows(slots, counts, C.GRAD_FP8BLOCK, D, master, m, v, outs, scratch, step=step)

    for s in range(1, 21):
        launch(s)
    torch.cuda.synchronize()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for s in range(args.launches):
        launch(21 + s)
    stop.record()
    torch.cuda.synchronize()
    ms = start.elapsed_time(stop) / args.launches
    nbytes = kernel_bytes(W, U, U, D, n_outs)
    gbs = nbytes / (ms * 1e-3) / 1e9
    bad = int(scratch[8:16].view(torch.int64).item())
    print(json.dumps({"bench": "update_rows_kernel", "gpu": gpu_info(), "rows": rows, "dim": D, "union": U,
                      "W": W, "format": "fp8", "outs": n_outs, "launches": args.launches,
                      "us_per_launch": round(ms * 1e3, 2), "model_bytes_per_launch": int(nbytes),
                      "GBps": round(gbs, 1), "fraction_of_copy_roofline": round(gbs / COPY_ROOFLINE_GBS, 3),
                      "bad_rows": bad}), flush=True)


def bench_train(args):
    from pslite_b200.utils.env import free_port

    script = os.path.join(ROOT, "examples", "train_llama_ps.py")
    results = {"dense": [], "sparse": []}
    for _ in range(args.rounds):
        for name in ("dense", "sparse"):
            cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
                   "--master-addr", "127.0.0.1", "--master-port", str(free_port()), script, "--model", "llama-1b",
                   "--steps", str(args.steps), "--grad-wire", "fp8"]
            if name == "sparse":
                cmd.append("--sparse-embedding")
            p = subprocess.run(cmd, capture_output=True, text=True, cwd=ROOT, timeout=1800)
            steps = [(float(t), int(b)) for t, b in re.findall(r"time ([\d.]+) ms push_bytes_wire (\d+)", p.stdout)]
            if p.returncode != 0 or len(steps) < 3:
                print((p.stdout + p.stderr)[-3000:], file=sys.stderr)
                raise SystemExit(f"{name} run failed (rc {p.returncode})")
            results[name].append(steps[2:])
    info = gpu_info()
    for name, runs in results.items():
        t = [s[0] for run in runs for s in run]
        b = [s[1] for run in runs for s in run]
        print(json.dumps({"bench": "llama1b_train", "gpus": args.gpus, "embedding": name, "gpu": info,
                          "steps_timed": len(t),
                          "median_step_ms": round(statistics.median(t), 1), "min_step_ms": round(min(t), 1),
                          "push_bytes_wire_per_step_rank0": int(statistics.median(b))}), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("what", choices=["kernel", "train"])
    ap.add_argument("--launches", type=int, default=200)
    ap.add_argument("--steps", type=int, default=12)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--gpus", type=int, default=2)
    args = ap.parse_args()
    bench_kernel(args) if args.what == "kernel" else bench_train(args)


if __name__ == "__main__":
    main()
