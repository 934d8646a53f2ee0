#!/usr/bin/env python
"""Llama PS training in ~60 lines: the tutorial of docs/tutorials.md §3 as a runnable script.

    torchrun --nproc-per-node 8 --master-addr 127.0.0.1 examples/train_llama_ps.py --model llama3-8b
    python examples/train_llama_ps.py --model tiny --steps 20        # one process: worker + server
    CUDA_VISIBLE_DEVICES= python examples/train_llama_ps.py --model tiny   # no GPU: shm van, host engine

Every rank is a worker and owns one shard of the optimizer state ("joint"); gradients leave from
autograd hooks (fp8 wire by default), the server engine runs fused AdamW on fp32 masters and writes
the new bf16 parameters back into every worker. Synthetic tokens.
"""
from __future__ import annotations

import argparse
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch  # noqa: E402

import pslite_b200  # noqa: E402
from pslite_b200.models.llama import Llama, LlamaConfig  # noqa: E402
from pslite_b200.parallel.launch import init_ps  # noqa: E402
from pslite_b200.parallel.ps_trainer import PSWorkerOptimizer  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--model", default="tiny", choices=["tiny", "llama-1b", "llama3-8b"])
    ap.add_argument("--seq-len", type=int, default=0)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--lr", type=float, default=3e-4)
    ap.add_argument("--grad-wire", default="fp8", choices=["fp8", "bf16"])
    ap.add_argument("--fused-pushpull", action="store_true")
    ap.add_argument("--sparse-embedding", action="store_true",
                    help="row-sparse input embedding: push only the rows a batch touched")
    args = ap.parse_args()

    use_cuda = torch.cuda.is_available()
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if int(os.environ.get("WORLD_SIZE", "1")) > 1:
        torch.distributed.init_process_group("cpu:gloo,cuda:nccl" if use_cuda else "gloo")
    dev = torch.device("cuda", local) if use_cuda else torch.device("cpu")
    if use_cuda:
        torch.cuda.set_device(dev)

    C = pslite_b200.native()
    ctx = init_ps("joint", van="nvl" if use_cuda else "shm")
    server = C.GpuServer(0, num_workers=ctx.num_workers, optimizer="adamw", lr=args.lr,
                         grad_scale=1.0 / ctx.num_workers)

    sparse = dict(sparse_embedding=args.sparse_embedding)
    if args.model == "tiny":
        cfg = LlamaConfig.tiny(**sparse)
    elif args.model == "llama-1b":
        cfg = LlamaConfig(dim=2048, n_layers=16, n_heads=32, n_kv_heads=8, ffn_dim=8192, ckpt_layers=0, **sparse)
    else:
        cfg = LlamaConfig.llama3_8b(ckpt_layers=0, **sparse)
    seq = args.seq_len or min(cfg.max_seq_len, 8192 if args.model != "tiny" else 64)
    with torch.device(dev):
        model = Llama(cfg).to(torch.bfloat16)
    model.init_weights(seed=0)

    kv = C.KVWorker(0, 0)
    opt = PSWorkerOptimizer(model.parameters(), kv, ctx.num_servers, ctx.num_workers, ctx.worker_rank,
                            grad_wire=args.grad_wire, fused_pushpull=args.fused_pushpull,
                            row_sparse=[model.embed.weight] if args.sparse_embedding else ()).attach()
    opt.init_parameters(barrier=lambda: C.barrier(0, C.WORKER_GROUP, "worker"))

    g = torch.Generator(device=dev).manual_seed(1 + ctx.worker_rank)
    tok = torch.randint(0, cfg.vocab_size, (1, seq + 1), device=dev, generator=g)
    import time

    times, wire = [], []
    for step in range(args.steps):
        t0, b0 = time.perf_counter(), opt.stats.push_bytes_wire
        loss = model(tok[:, :-1], tok[:, 1:])
        loss.backward()   # gradients are pushed from the hooks while backward still runs
        opt.step()        # every parameter chunk has been rewritten by its server
        if use_cuda:
            torch.cuda.synchronize()
        times.append(time.perf_counter() - t0)
        wire.append(opt.stats.push_bytes_wire - b0)
        if ctx.worker_rank == 0:
            print(f"step {step}: loss {loss.item():.4f} time {times[-1] * 1e3:.1f} ms "
                  f"push_bytes_wire {wire[-1]}", flush=True)
    if ctx.worker_rank == 0:
        print(f"server 0: {server.num_updates()} updates on the {'device' if server.on_device() else 'host'} engine")
    ctx.shutdown()


if __name__ == "__main__":
    main()
