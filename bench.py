#!/usr/bin/env python
"""Headline benchmark of pslite_b200 (driver contract: see the task statement).

    python bench.py --gpus N --steps K --warmup W [--impl ours|reference] [--metric pushpull|llama|resnet]
                    [--dump-outputs DIR]

Default metric — the reference's own headline benchmark (tests/test_benchmark.cc,
BASELINE.json "push+pull GB/s ... (test_benchmark)"): every worker ZPush-es and ZPull-s
`keys_per_server x num_servers` values of `len` bytes per step (= one round of the
reference's timing loop) and the job reports payload goodput with the reference's
formula (payload counted once per push+pull pair), in GB/s, summed over workers.
    every N      : N workers + N servers, one of each co-located on every GPU ("joint"; the same
                   topology at every N, so the payload per step grows with N and the driver's
                   scaling efficiency compares like with like). Worker r talks to all N servers:
                   1/N of its traffic stays in local HBM, the rest crosses NVLink.
    --topology split : N/2 worker GPUs + N/2 server GPUs (4w+4s at N=8, BASELINE.json config 2)
Values live in HBM and move as one-sided sm_100a copy kernels into peer memory; only
descriptors use TCP. `--metric llama` instead times Llama-3-8B synchronous PS training
(fp8 gradient push, fused server-side AdamW, bf16 pull) in tokens/s, `--metric resnet` ResNet-50
(BASELINE.json config 3: ZPush gradients / ZPull parameters, fused server-side SGD) in images/s.

`--impl reference` runs the UNMODIFIED reference build (baseline/_ref, ZMQ van — the
only reference transport buildable without ibverbs/UCX) through its own test_benchmark
binary with the same len / keys / mode and prints the same JSON line.
"""
from __future__ import annotations

import argparse
import json
import os
import re
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC_NAME = {
    "pushpull": "test_benchmark push+pull goodput",
    "llama": "Llama-3-8B PS training throughput",
    "resnet": "ResNet-50 PS training throughput",
}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "nccl-ddp"],
                    help="nccl-ddp (with --metric llama): SECONDARY baseline, not the reference — the same model "
                         "trained with NCCL all-reduce of the gradients + torch.optim.AdamW(fused=True) on every rank")
    ap.add_argument("--metric", default="pushpull", choices=["pushpull", "llama", "resnet"])
    ap.add_argument("--len", type=int, default=4096000, help="bytes per value (reference test.sh preset)")
    ap.add_argument("--keys-per-server", type=int, default=40)
    ap.add_argument("--topology", default=None, choices=[None, "joint", "split"])
    ap.add_argument("--van", default=None)
    ap.add_argument("--device", default="cuda", choices=["cuda", "cpu"],
                    help="cpu: self-check of this script's control flow on a GPU-less box (shm van, host "
                         "engine, host clock); its numbers are not benchmark results")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--e2e-native", action="store_true",
                    help="also time the end-to-end round through KVWorker.staged_push_pull (the H2D / push / "
                         "pull / D2H pipeline in one native call instead of a Python loop)")
    ap.add_argument("--copy-engine", type=int, default=int(os.environ.get("PS_COPY_ENGINE", "1")),
                    help="1: raw copies without a producer event are posted to the copy engine (on-demand "
                         "persistent kernel fed from a host-mapped ring) instead of one launch each")
    ap.add_argument("--sweep", default="", help="comma-separated extra message sizes (bytes) to report")
    # llama
    ap.add_argument("--seq-len", type=int, default=8192)
    ap.add_argument("--micro-batch", type=int, default=1)
    ap.add_argument("--grad-wire", default="fp8", choices=["fp8", "bf16"])
    ap.add_argument("--model", default="llama3-8b", choices=["llama3-8b", "llama-1b", "tiny"],
                    help="llama: which size; resnet: 'tiny' selects the smoke-test network, anything else ResNet-50")
    ap.add_argument("--image-batch", type=int, default=128, help="resnet: images per worker and step (224 x 224)")
    ap.add_argument("--ckpt-layers", type=int, default=-1)
    ap.add_argument("--attn-backend", default="auto", choices=["auto", "cudnn", "flash", "efficient", "math"])
    ap.add_argument("--lazy-wait", action="store_true",
                    help="llama: step() does not wait; every module waits for its own parameters before its "
                         "forward (hides the step tail)")
    ap.add_argument("--fused-pushpull", action="store_true",
                    help="llama: one KVWorker::ZPushPull per parameter chunk instead of push + pull; "
                         "pushpull: additionally time the fused operation (reported as fused_pushpull)")
    ap.add_argument("--nvls-reduce", action="store_true",
                    help="with --symmetric: bf16 gradients staged in symmetric memory and summed inside "
                         "the NVSwitch by the update kernel (multimem.ld_reduce)")
    ap.add_argument("--symmetric", action="store_true",
                    help="parameters in symmetric memory; NVLS multicast pull fan-out (N > 1)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what rank 0 received from the last one as DIR/<name>.npy "
                         "(float32): pushpull the pulled values, llama / resnet the loss and the updated "
                         "parameters. Past 60 MB in all, a fixed seeded sample of every array is written")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs records this project's timed path (--impl ours)")
    return args


DUMP_MAX_ELEMS = 15_000_000  # float32: 60 MB of .npy files at most


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """Writes out_dir/<name>.npy (float32) for every name -> list of tensors, each list flattened and joined.
    When all of them hold more than DUMP_MAX_ELEMS elements, every tensor keeps the same share of its
    elements (one at least, so a loss is never dropped), at positions drawn by a generator seeded with the
    tensor's size: the same arguments give the same positions in every run and every build."""
    import numpy as np
    import torch

    total = sum(t.numel() for ts in arrays.values() for t in ts)
    share = min(1.0, DUMP_MAX_ELEMS / max(total, 1))
    os.makedirs(out_dir, exist_ok=True)
    for name, ts in arrays.items():
        parts = []
        for t in ts:
            flat = t.detach().reshape(-1)
            m = max(1, int(flat.numel() * share))
            if m < flat.numel():
                g = torch.Generator().manual_seed(flat.numel())
                idx = torch.randint(0, flat.numel(), (m,), generator=g).sort().values
                flat = flat[idx.to(flat.device)]
            parts.append(flat.float().cpu())
        np.save(os.path.join(out_dir, f"{name}.npy"), torch.cat(parts).numpy())


# ----------------------------------------------------------------------------------------
# distributed plumbing
# ----------------------------------------------------------------------------------------
class Dist:
    """torch.distributed when WORLD_SIZE > 1 (gloo for host-side barriers / reductions so the
    measured GPUs run nothing but the benchmark), no-ops otherwise."""

    def __init__(self):
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        self.gloo = None
        if self.world > 1:
            import torch
            import torch.distributed as dist

            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            backend = "cpu:gloo,cuda:nccl" if torch.cuda.is_available() else "gloo"
            dist.init_process_group(backend=backend, rank=self.rank, world_size=self.world)
            self.gloo = dist.new_group(backend="gloo")

    def barrier(self):
        if self.world > 1:
            import torch.distributed as dist

            dist.barrier(group=self.gloo)

    def reduce(self, value: float, op: str) -> float:
        if self.world == 1:
            return value
        import torch
        import torch.distributed as dist

        t = torch.tensor([value], dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX if op == "max" else dist.ReduceOp.SUM, group=self.gloo)
        return float(t.item())

    def shutdown(self):
        if self.world > 1:
            import torch.distributed as dist

            dist.destroy_process_group()


class Gpu:
    """The few torch.cuda calls of this script behind one switch, so that `--device cpu` walks the
    same code (different MemDomain, different kernel implementations, host clock)."""

    def __init__(self, args, local_rank: int):
        import torch

        self.cuda = args.device == "cuda"
        self.dev = torch.device("cuda", local_rank) if self.cuda else torch.device("cpu")
        if self.cuda:
            torch.cuda.set_device(local_rank)

    def sync(self):
        if self.cuda:
            import torch

            torch.cuda.synchronize()

    def timer(self):
        """returns stop() -> elapsed milliseconds since this call (CUDA events on the GPU)"""
        import torch

        if not self.cuda:
            t0 = time.perf_counter()
            return lambda: (time.perf_counter() - t0) * 1e3
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()

        def stop():
            e1.record()
            e1.synchronize()
            return e0.elapsed_time(e1)
        return stop

    def stream(self):
        import torch

        return torch.cuda.Stream(device=self.dev) if self.cuda else None

    def on(self, stream):
        import contextlib

        import torch

        return torch.cuda.stream(stream) if self.cuda else contextlib.nullcontext()

    def buffer(self, C, nbytes: int, fill: int):
        """uint8 buffer the van can move one-sidedly: HBM, or shared memory on the host"""
        import torch

        if self.cuda:
            return torch.full((nbytes,), fill, dtype=torch.uint8, device=self.dev)
        return C.alloc_exportable(nbytes, "worker").fill_(fill)

    def pinned(self, t):
        return t.pin_memory() if self.cuda else t


# ----------------------------------------------------------------------------------------
# ours: push/pull
# ----------------------------------------------------------------------------------------
def run_pushpull(args, dist: Dist) -> dict:
    import torch

    from pslite_b200 import native
    from pslite_b200.parallel.launch import init_ps
    from pslite_b200.utils.timing import ClockSampler

    C = native()
    gpu = Gpu(args, dist.local_rank)
    topo = args.topology or "joint"
    ctx = init_ps(topo, van=args.van or ("nvl" if gpu.cuda else "shm"),
                  extra_env={"PS_COPY_ENGINE": int(args.copy_engine)})
    server = C.BenchServer(0) if ctx.is_server else None
    S, W = ctx.num_servers, ctx.num_workers
    total_keys = S * args.keys_per_server
    kv = keys = vals = None
    if ctx.is_worker:
        kv = C.KVWorker(0, 0)
        keys = [kv.server_key(k % S, k) for k in range(total_keys)]
        vals = [gpu.buffer(C, args.len, 1) for _ in range(total_keys)]
        for k in range(total_keys):  # rendezvous + store creation, untimed (as the reference does)
            kv.wait(kv.push(keys[k], vals[k], order_after_current_stream=False))
    dist.barrier()

    def one_round():
        # one call issues ZPush + ZPull for every key (test_benchmark's inner loop), then Wait all
        kv.wait_all(kv.push_pull_batch(keys, vals, order_after_current_stream=False))

    def verify(tag: str):
        """untimed data check: distinct patterns go up, the buffers are cleared, the pull must bring
        every byte back (the timed rounds move constant bytes and would not notice a lost copy)"""
        idx = sorted({0, 1, total_keys // 2, total_keys - 1})
        want = {}
        if ctx.is_worker:
            # every worker pushes the same bytes for a key (the benchmark's servers answer a pull from
            # the slot of whichever worker pushed that key first)
            for k in idx:
                pat = (torch.arange(args.len, dtype=torch.int32, device=vals[k].device) * (k + 3) + 7).to(torch.uint8)
                vals[k].copy_(pat)
                want[k] = pat
            gpu.sync()
            kv.wait_all(kv.push_pull_batch([keys[k] for k in idx], [vals[k] for k in idx],
                                           order_after_current_stream=False, pull=False))
            for k in idx:
                vals[k].zero_()
            gpu.sync()
        dist.barrier()  # all patterns are up before anybody pulls
        if ctx.is_worker:
            kv.wait_all(kv.push_pull_batch([keys[k] for k in idx], [vals[k] for k in idx],
                                           order_after_current_stream=False, push=False))
            gpu.sync()
            for k in idx:
                assert torch.equal(vals[k], want[k]), f"{tag}: key {k} came back different from what was pushed"
        dist.barrier()  # nobody restores the constant bytes while a peer still compares
        if ctx.is_worker:
            for k in idx:
                vals[k].fill_(1)
            gpu.sync()
            kv.wait_all(kv.push_pull_batch([keys[k] for k in idx], [vals[k] for k in idx],
                                           order_after_current_stream=False, pull=False))

    my_role = "worker" if ctx.is_worker else "server"

    def engine_items() -> int:
        # descriptors this GPU's copy engine has executed (one engine per device and process)
        return int(C.van_stats(my_role).get("engine_items", 0))

    engine_work = {"descriptors": 0}

    def timed(fn, steps: int):
        dist.barrier()
        gpu.sync()
        launches0 = C.kernel_launch_count()
        items0 = engine_items()
        stop = gpu.timer()
        if ctx.is_worker:
            for _ in range(steps):
                fn()
        gpu.sync()
        ms = stop()
        dist.barrier()  # servers keep serving until every worker is done
        launches = C.kernel_launch_count() - launches0
        engine_work["descriptors"] = int(dist.reduce(float(engine_items() - items0), "sum"))
        return dist.reduce(ms, "max"), dist.reduce(float(launches), "sum")

    # clocks are sampled from the warm-up on (same load as the timed steps): K steps of this
    # benchmark can be shorter than one nvidia-smi sampling period
    sampler = ClockSampler(dist.local_rank, period_ms=100).start() if dist.rank == 0 and gpu.cuda else None
    if ctx.is_worker:
        t_end = time.time() + 1.0
        n_warm = 0
        while n_warm < args.warmup or time.time() < t_end:
            one_round()
            n_warm += 1
    verify("before the timed rounds")
    ms, launches = timed(one_round, args.steps)
    copies_by_engine = engine_work["descriptors"]
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and dist.rank == 0:
        dump_outputs(args.dump_outputs, {"pulled_values": vals})  # before verify() overwrites them
    verify("after the timed rounds")
    payload = float(args.len) * total_keys * W  # per step, counted once per push+pull pair
    value = payload * args.steps / (ms * 1e-3) / 1e9

    e2e = None
    if not args.no_e2e:
        host_in = host_out = None
        if ctx.is_worker:
            host_in = [gpu.pinned(torch.full((args.len,), 2, dtype=torch.uint8)) for _ in range(total_keys)]
            host_out = [gpu.pinned(torch.empty(args.len, dtype=torch.uint8)) for _ in range(total_keys)]

        h2d_stream = gpu.stream() if ctx.is_worker else None
        d2h_stream = gpu.stream() if ctx.is_worker else None

        def e2e_round():
            # software pipeline over keys: H2D of key k+1 | push+pull of key k | D2H of key k-1
            # (PCIe is full duplex; the push waits on the event of its own H2D copy only)
            pulls = []
            with gpu.on(h2d_stream):
                for k in range(total_keys):
                    vals[k].copy_(host_in[k], non_blocking=True)      # H2D of this step's input
                    kv.push(keys[k], vals[k], order_after_current_stream=True)
                    pulls.append(kv.pull(keys[k], vals[k]))
            with gpu.on(d2h_stream):
                for k in range(total_keys):
                    kv.wait(pulls[k])                                 # value k is back in HBM
                    host_out[k].copy_(vals[k], non_blocking=True)     # D2H of the pulled result
            if d2h_stream is not None:
                d2h_stream.synchronize()

        if ctx.is_worker:
            e2e_round()
        e2e_steps = max(3, args.steps // 4)
        ms2, _ = timed(e2e_round, e2e_steps)
        e2e = {"value": payload * e2e_steps / (ms2 * 1e-3) / 1e9, "unit": "GB/s",
               "h2d_bytes_per_step": int(args.len) * total_keys * W,
               "d2h_bytes_per_step": int(args.len) * total_keys * W, "steps": e2e_steps}
        if args.e2e_native:
            def native_round():
                kv.staged_push_pull(keys, vals, host_in, host_out)
            if ctx.is_worker:
                native_round()
                assert all(int(h[0]) == 2 and int(h[-1]) == 2 for h in host_out), "staged round lost data"
            ms3, _ = timed(native_round, e2e_steps)
            e2e["native_call"] = {"value": payload * e2e_steps / (ms3 * 1e-3) / 1e9, "unit": "GB/s"}

    fused = None
    if args.fused_pushpull:
        # same bytes per key, but ONE KVWorker::ZPushPull instead of ZPush + ZPull (extension over the
        # reference API; reported next to the headline, never instead of it)
        def fused_round():
            kv.wait_all(kv.push_pull_batch(keys, vals, order_after_current_stream=False, fused=True))
        if ctx.is_worker:
            for _ in range(max(3, args.warmup)):
                fused_round()
        ms_f, _ = timed(fused_round, args.steps)
        fused = {"value": payload * args.steps / (ms_f * 1e-3) / 1e9, "unit": "GB/s", "ms_per_step": ms_f / args.steps}

    sweep = []
    for sz in [int(x) for x in args.sweep.split(",") if x]:
        nk = max(1, min(args.keys_per_server, (512 << 20) // max(sz, 1))) * S
        if ctx.is_worker:
            skeys = [kv.server_key(k % S, 100000 + k) for k in range(nk)]
            svals = [gpu.buffer(C, sz, 1) for _ in range(nk)]
            for k in range(nk):
                kv.wait(kv.push(skeys[k], svals[k], order_after_current_stream=False))

            def sround():
                ts = []
                for k in range(nk):
                    ts.append(kv.push(skeys[k], svals[k], order_after_current_stream=False))
                    ts.append(kv.pull(skeys[k], svals[k]))
                for t in ts:
                    kv.wait(t)
            for _ in range(3):
                sround()
        else:
            sround = None
        reps = max(3, min(50, int(2e9 // max(sz * nk, 1)) + 3))
        ms_s, _ = timed(sround, reps)
        sweep.append({"msg_bytes": sz, "keys": nk, "GBps": float(sz) * nk * W * reps / (ms_s * 1e-3) / 1e9,
                      "us_per_key": ms_s * 1e3 / reps / nk})
        if ctx.is_worker:
            del svals

    # what bounds this configuration, from this pod's measured peaks (profiles/r2/README.md): per GPU and key
    # pair, joint topology, (N-1)/N of the pushes and of the pull replies cross NVLink (672-703 GB/s in one
    # direction); at N = 1 both copies stay in HBM (read + write = 4 bytes of traffic per payload byte)
    if topo == "joint":
        n = max(1, dist.world)
        bound_per_gpu = 6571.0 / 4.0 if n == 1 else min(6571.0 / 4.0, 675.0 / (2.0 * (n - 1) / n))
        bound_what = "HBM copy peak / 4" if n == 1 else "NVLink egress: 675 GB/s / (2 (N-1)/N)"
    else:
        n = max(1, dist.world // 2)
        bound_per_gpu = 675.0  # every push leaves a worker GPU, every pull reply leaves a server GPU
        bound_what = "NVLink one direction (peer-copy kernel 672-703 GB/s) per worker"
    roofline = {"bound_GBps": round(bound_per_gpu * n, 1), "bound": bound_what,
                "fraction_of_bound": round(value / (bound_per_gpu * n), 3)}
    stats = {}
    for role in (["worker"] if ctx.is_worker else []) + (["server"] if ctx.is_server else []):
        stats[role] = {k: int(v) for k, v in C.van_stats(role).items()}
    ctx.shutdown()
    return {
        "sweep": sweep, "van_stats_rank0": stats, "roofline": roofline,
        "fused_pushpull": fused,
        "metric": METRIC_NAME["pushpull"], "value": value, "unit": "GB/s",
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "uint8 payload (bit-exact copy)", "data": "synthetic",
        "config": {"model": "test_benchmark PUSH_PULL", "msg_bytes": args.len,
                   "keys_per_server": args.keys_per_server, "num_workers": W, "num_servers": S,
                   "global_batch": total_keys * W, "seq_len": args.len,
                   "parallelism": f"{W}w+{S}s {'co-located' if topo == 'joint' else 'split'} on {dist.world} "
                                  f"{'GPU(s), nvl van' if gpu.cuda else 'CPU process(es), shm van (self-check, not a result)'}",
                   "l2": f"working set {args.len * total_keys / 1e6:.0f} MB per worker > 126 MB L2"},
        "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches),
        # with the copy engine a launch is one (re)start of the persistent kernel; the copies themselves are
        # descriptors it executes — this many inside the timed region, summed over the GPUs
        "gpu_copy_engine_descriptors": copies_by_engine,
    }


# ----------------------------------------------------------------------------------------
# ours: Llama-3-8B PS training
# ----------------------------------------------------------------------------------------
def run_llama(args, dist: Dist) -> dict:
    import torch

    from pslite_b200 import native
    from pslite_b200.models.llama import Llama, LlamaConfig
    from pslite_b200.parallel.launch import init_ps
    from pslite_b200.parallel.ps_trainer import PSWorkerOptimizer
    from pslite_b200.utils.timing import ClockSampler

    C = native()
    gpu = Gpu(args, dist.local_rank)
    dev = gpu.dev
    topo = args.topology or "joint"
    ctx = init_ps(topo, van=args.van or ("nvl" if gpu.cuda else "shm"))
    W, S = ctx.num_workers, ctx.num_servers
    server = None
    if ctx.is_server:
        server = C.GpuServer(0, num_workers=W, optimizer="adamw", lr=3e-4, beta1=0.9, beta2=0.95,
                             eps=1e-8, weight_decay=0.1, grad_scale=1.0 / W, fuse_pull=True)
    if args.model == "llama3-8b":
        cfg = LlamaConfig.llama3_8b(max_seq_len=args.seq_len)
    elif args.model == "llama-1b":
        cfg = LlamaConfig(dim=2048, n_layers=16, n_heads=32, n_kv_heads=8, ffn_dim=8192,
                          max_seq_len=args.seq_len)
    else:
        cfg = LlamaConfig.tiny(max_seq_len=args.seq_len)
    # measured on one B200 (worker + its server shard on the same GPU, 8.03 B parameters,
    # seq 8192): no activation recomputation fits (53 GB of torch allocations + 104 GB of
    # server state / landing slots) and is the fastest setting
    cfg.ckpt_layers = args.ckpt_layers if args.ckpt_layers >= 0 else 0
    cfg.attn_backend = args.attn_backend
    B, T = args.micro_batch, args.seq_len
    model = opt = kv = None
    if ctx.is_worker:
        with torch.device(dev):
            model = Llama(cfg).to(torch.bfloat16)
        model.init_weights(seed=0)
        model.train()
    use_symm = args.symmetric and dist.world > 1 and gpu.cuda
    mc = 0
    if use_symm:
        import torch.distributed as tdist

        from pslite_b200.parallel.ps_trainer import setup_symmetric_params, symmetric_layout

        with torch.device("meta"):
            shapes = list(Llama(cfg).parameters())
        _, total = symmetric_layout(shapes)
        plist = list(model.parameters()) if model is not None else None
        flat, hdl, mc, peers, nbytes = setup_symmetric_params(plist, total, tdist.group.WORLD, dev,
                                                              list(range(W)))
        if server is not None:
            server.set_symmetric(mc, peers, nbytes)
    gbuf = None
    if use_symm and args.nvls_reduce and mc:
        from pslite_b200.parallel.ps_trainer import setup_symmetric_grads

        gbuf, ghdl, gmc, gbytes = setup_symmetric_grads(total, tdist.group.WORLD, dev,
                                                              "worker" if ctx.is_worker else "server")
        if server is not None:
            server.set_symmetric_grads(gmc, gbytes)
        dist.barrier()
    if ctx.is_worker:
        kv = C.KVWorker(0, 0)
        opt = PSWorkerOptimizer(model.parameters(), kv, S, W, ctx.worker_rank,
                                grad_wire=args.grad_wire, symmetric=use_symm,
                                grad_buffer=gbuf, fused_pushpull=args.fused_pushpull and gbuf is None).attach()
        opt.init_parameters(barrier=lambda: C.barrier(0, C.WORKER_GROUP, "worker"))
        if args.lazy_wait:
            opt.enable_lazy_wait(model)
    dist.barrier()
    g = torch.Generator().manual_seed(1234 + dist.rank)
    host_tok = gpu.pinned(torch.randint(0, cfg.vocab_size, (B, T + 1), generator=g))

    def step(e2e: bool):
        if e2e:
            tok = host_tok.to(dev, non_blocking=True)
        else:
            tok = step.dev_tok
        loss = model(tok[:, :-1], tok[:, 1:])
        loss.backward()
        opt.step()
        step.loss = loss
        return loss.item() if e2e else loss

    step.dev_tok = host_tok.to(dev) if ctx.is_worker else None

    def timed(fn, steps):
        dist.barrier()
        gpu.sync()
        l0 = C.kernel_launch_count()
        stop = gpu.timer()
        if ctx.is_worker:
            for _ in range(steps):
                fn()
            opt.wait_all()  # lazy waits: the last step's parameters must have arrived inside the timed region
        gpu.sync()
        ms = stop()
        dist.barrier()
        return dist.reduce(ms, "max"), dist.reduce(float(C.kernel_launch_count() - l0), "sum")

    if ctx.is_worker:
        for _ in range(args.warmup):
            step(False)
    sampler = ClockSampler(dist.local_rank).start() if dist.rank == 0 and gpu.cuda else None
    ms, launches = timed(lambda: step(False), args.steps)
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and dist.rank == 0:
        dump_outputs(args.dump_outputs, {"loss": [step.loss], "parameters": list(model.parameters())})
    tokens = B * T * W
    value = tokens * args.steps / (ms * 1e-3)
    e2e = None
    if not args.no_e2e:
        k = max(2, args.steps // 2)
        ms2, _ = timed(lambda: step(True), k)
        e2e = {"value": tokens * k / (ms2 * 1e-3), "unit": "tokens/s",
               "h2d_bytes_per_step": int(host_tok.numel() * host_tok.element_size()) * W,
               "d2h_bytes_per_step": 4 * W, "steps": k}
    mfu = None
    if ctx.is_worker:
        peak = 1386e12
        mfu = cfg.flops_per_token(T) * B * T / (ms / args.steps * 1e-3) / peak
    peak_mem = round(torch.cuda.max_memory_allocated() / 2**30, 1) if gpu.cuda else None
    stats = {"server_updates": server.num_updates() if server else 0,
             "server_fused_fanouts": server.num_fused_fanouts() if server else 0,
             "server_multicast_fanouts": server.num_multicast_fanouts() if server else 0,
             "server_switch_reductions": server.num_switch_reductions() if server else 0,
             "multicast_available": bool(mc)}
    ctx.shutdown()
    return {
        "metric": METRIC_NAME["llama"], "value": value, "unit": "tokens/s",
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic tokens, random-init weights",
        "config": {"model": args.model, "params": cfg.num_params(), "global_batch": B * W,
                   "seq_len": T,
                   "parallelism": f"ps-dp{W} ({W}w+{S}s {topo}), grad wire "
                                  f"{'bf16 in-switch reduce' if gbuf is not None else args.grad_wire}, server AdamW",
                   "ckpt_layers": cfg.ckpt_layers, "l2": "per-step working set >> 126 MB L2"},
        "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "mfu_vs_sustained_bf16": mfu,
        "peak_torch_mem_gb": peak_mem,
        "server": stats,
    }


# ----------------------------------------------------------------------------------------
# ours: ResNet-50 PS training (BASELINE.json config 3)
# ----------------------------------------------------------------------------------------
def run_resnet(args, dist: Dist) -> dict:
    """ResNet-50, bf16, channels-last, synchronous data parallelism through the parameter server: every
    worker pushes its gradients (KVWorker ZPush, bf16 or block-scaled fp8 on the wire), the servers run the
    fused sum + SGD update on their key ranges and the workers pull the new parameters (ZPull). Convolutions
    are cuDNN's; what this repo contributes to the step is the gradient / parameter traffic and the update.
    BatchNorm statistics stay worker-local."""
    import torch

    from pslite_b200 import native
    from pslite_b200.models.resnet import resnet50, resnet_tiny
    from pslite_b200.parallel.launch import init_ps
    from pslite_b200.parallel.ps_trainer import PSWorkerOptimizer
    from pslite_b200.utils.timing import ClockSampler

    C = native()
    gpu = Gpu(args, dist.local_rank)
    dev = gpu.dev
    topo = args.topology or "joint"
    ctx = init_ps(topo, van=args.van or ("nvl" if gpu.cuda else "shm"))
    W, S = ctx.num_workers, ctx.num_servers
    server = None
    if ctx.is_server:
        server = C.GpuServer(0, num_workers=W, optimizer="sgd", lr=0.1, weight_decay=1e-4, grad_scale=1.0 / W,
                             fuse_pull=True)
    tiny = args.model == "tiny"
    B = args.image_batch if not tiny else min(args.image_batch, 4)
    side = 224 if not tiny else 32
    classes = 1000 if not tiny else 10
    model = opt = None
    if ctx.is_worker:
        torch.manual_seed(0)  # the same initial weights in every run
        with torch.device(dev):
            model = (resnet_tiny(classes) if tiny else resnet50(classes)).to(torch.bfloat16)
        # weights and activations channels-last (cuDNN's NHWC kernels); the PS moves a weight as the flat buffer
        # of its storage, whatever the order of the dimensions in it
        model = model.to(memory_format=torch.channels_last)
        model.train()
        kv = C.KVWorker(0, 0)
        opt = PSWorkerOptimizer(model.parameters(), kv, S, W, ctx.worker_rank, grad_wire=args.grad_wire,
                                fused_pushpull=args.fused_pushpull).attach()
        opt.init_parameters(barrier=lambda: C.barrier(0, C.WORKER_GROUP, "worker"))
    dist.barrier()
    g = torch.Generator().manual_seed(4321 + dist.rank)
    host_img = gpu.pinned(torch.randn(B, 3, side, side, generator=g).to(torch.bfloat16))
    host_lbl = gpu.pinned(torch.randint(0, classes, (B,), generator=g))
    loss_fn = torch.nn.CrossEntropyLoss()

    def step(e2e: bool):
        if e2e:
            img = host_img.to(dev, non_blocking=True).contiguous(memory_format=torch.channels_last)
            lbl = host_lbl.to(dev, non_blocking=True)
        else:
            img, lbl = step.dev
        loss = loss_fn(model(img).float(), lbl)
        loss.backward()
        opt.step()
        step.loss = loss
        return loss.item() if e2e else loss

    if ctx.is_worker:
        step.dev = (host_img.to(dev).contiguous(memory_format=torch.channels_last), host_lbl.to(dev))

    def timed(fn, steps):
        dist.barrier()
        gpu.sync()
        l0 = C.kernel_launch_count()
        stop = gpu.timer()
        if ctx.is_worker:
            for _ in range(steps):
                fn()
            opt.wait_all()
        gpu.sync()
        ms = stop()
        dist.barrier()
        return dist.reduce(ms, "max"), dist.reduce(float(C.kernel_launch_count() - l0), "sum")

    if ctx.is_worker:
        for _ in range(args.warmup):
            step(False)
    sampler = ClockSampler(dist.local_rank).start() if dist.rank == 0 and gpu.cuda else None
    ms, launches = timed(lambda: step(False), args.steps)
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and dist.rank == 0:
        dump_outputs(args.dump_outputs, {"loss": [step.loss], "parameters": list(model.parameters())})
    images = B * W
    value = images * args.steps / (ms * 1e-3)
    e2e = None
    if not args.no_e2e:
        k = max(2, args.steps // 2)
        ms2, _ = timed(lambda: step(True), k)
        e2e = {"value": images * k / (ms2 * 1e-3), "unit": "images/s",
               "h2d_bytes_per_step": int(host_img.numel() * host_img.element_size()
                                         + host_lbl.numel() * host_lbl.element_size()) * W,
               "d2h_bytes_per_step": 4 * W, "steps": k}
    params = sum(p.numel() for p in model.parameters()) if model is not None else None
    stats = {"server_updates": server.num_updates() if server else 0,
             "server_fused_fanouts": server.num_fused_fanouts() if server else 0}
    ctx.shutdown()
    return {
        "metric": METRIC_NAME["resnet"], "value": value, "unit": "images/s",
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic images, random-init weights",
        "config": {"model": "resnet-tiny" if tiny else "resnet50", "params": params, "global_batch": B * W,
                   "seq_len": side,
                   "parallelism": f"ps-dp{W} ({W}w+{S}s {topo}), grad wire {args.grad_wire}, server SGD",
                   "l2": "activations of a step >> 126 MB L2"},
        "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "server": stats,
    }


# ----------------------------------------------------------------------------------------
# secondary baseline: NCCL data parallelism (NOT the reference — it has no trainer)
# ----------------------------------------------------------------------------------------
def run_llama_ddp(args, dist: Dist) -> dict:
    """Same model, same batch, same step structure as run_llama, but the gradients are summed with
    NCCL all-reduce (bucketed, overlapped by DistributedDataParallel) and every rank runs
    torch.optim.AdamW(fused=True) on its full bf16 replica. Gives tokens/s an anchor."""
    import torch
    import torch.distributed as tdist

    from pslite_b200.models.llama import Llama, LlamaConfig
    from pslite_b200.utils.timing import ClockSampler

    gpu = Gpu(args, dist.local_rank)
    dev = gpu.dev
    if args.model == "llama3-8b":
        cfg = LlamaConfig.llama3_8b(max_seq_len=args.seq_len)
    elif args.model == "llama-1b":
        cfg = LlamaConfig(dim=2048, n_layers=16, n_heads=32, n_kv_heads=8, ffn_dim=8192, max_seq_len=args.seq_len)
    else:
        cfg = LlamaConfig.tiny(max_seq_len=args.seq_len)
    cfg.ckpt_layers = args.ckpt_layers if args.ckpt_layers >= 0 else 0
    cfg.attn_backend = args.attn_backend
    B, T, W = args.micro_batch, args.seq_len, dist.world
    with torch.device(dev):
        model = Llama(cfg).to(torch.bfloat16)
    model.init_weights(seed=0)
    model.train()
    net = model
    if W > 1:
        from torch.nn.parallel import DistributedDataParallel as DDP

        net = DDP(model, device_ids=[dist.local_rank] if gpu.cuda else None, gradient_as_bucket_view=True,
                  bucket_cap_mb=256)
    opt = torch.optim.AdamW(model.parameters(), lr=3e-4, betas=(0.9, 0.95), eps=1e-8, weight_decay=0.1,
                            fused=gpu.cuda)
    g = torch.Generator().manual_seed(1234 + dist.rank)
    host_tok = gpu.pinned(torch.randint(0, cfg.vocab_size, (B, T + 1), generator=g))
    dev_tok = host_tok.to(dev)

    def step(e2e: bool):
        tok = host_tok.to(dev, non_blocking=True) if e2e else dev_tok
        loss = net(tok[:, :-1], tok[:, 1:])
        loss.backward()
        opt.step()
        opt.zero_grad(set_to_none=True)
        return loss.item() if e2e else loss

    def timed(fn, steps):
        dist.barrier()
        gpu.sync()
        stop = gpu.timer()
        for _ in range(steps):
            fn()
        gpu.sync()
        ms = stop()
        dist.barrier()
        return dist.reduce(ms, "max")

    for _ in range(args.warmup):
        step(False)
    sampler = ClockSampler(dist.local_rank).start() if dist.rank == 0 and gpu.cuda else None
    ms = timed(lambda: step(False), args.steps)
    clocks = sampler.stop() if sampler else None
    tokens = B * T * W
    k = max(2, args.steps // 2)
    ms2 = timed(lambda: step(True), k)
    return {
        "impl": "nccl-ddp", "note": "secondary baseline (NCCL all-reduce + fused AdamW), NOT the reference",
        "metric": METRIC_NAME["llama"], "value": tokens * args.steps / (ms * 1e-3), "unit": "tokens/s",
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16", "data": "synthetic tokens, random-init weights",
        "config": {"model": args.model, "params": cfg.num_params(), "global_batch": B * W, "seq_len": T,
                   "parallelism": f"dp{W} NCCL all-reduce, bf16 AdamW states on every rank",
                   "ckpt_layers": cfg.ckpt_layers},
        "clocks": clocks, "gpu_launches": 0,
        "e2e": {"value": tokens * k / (ms2 * 1e-3), "unit": "tokens/s",
                "h2d_bytes_per_step": int(host_tok.numel() * host_tok.element_size()) * W, "d2h_bytes_per_step": 4 * W},
        "mfu_vs_sustained_bf16": cfg.flops_per_token(T) * B * T / (ms / args.steps * 1e-3) / 1386e12,
        "peak_torch_mem_gb": round(torch.cuda.max_memory_allocated() / 2**30, 1) if gpu.cuda else None,
    }


# ----------------------------------------------------------------------------------------
# reference arm
# ----------------------------------------------------------------------------------------
def reference_goodput(worker_output: str) -> float | None:
    """Gbps of the last window the reference test_benchmark printed (the one after warm-up)."""
    found = re.findall(r"Application goodput: ([0-9.eE+-]+) Gbps", worker_output)
    return float(found[-1]) if found else None


def run_reference(args, dist: Dist) -> dict:
    if args.metric != "pushpull":
        return {"impl": "reference", "unavailable":
                "the reference is a communication library with no trainer or model code; only its test_benchmark can be run"}
    sys.path.insert(0, os.path.join(ROOT, "baseline"))
    import build_reference

    res = build_reference.build()
    if not res["ok"]:
        return {"impl": "reference", "unavailable": res["why"]}
    out = None
    if dist.rank == 0:
        # same shape as our arm: N workers + N servers (N/2 + N/2 with --topology split)
        W = S = dist.world if (args.topology or "joint") == "joint" else max(1, dist.world // 2)
        port = 12000 + (os.getpid() % 20000)
        env = dict(os.environ)
        env.update({"DMLC_NUM_WORKER": str(W), "DMLC_NUM_SERVER": str(S),
                    "DMLC_PS_ROOT_URI": "127.0.0.1", "DMLC_PS_ROOT_PORT": str(port),
                    "DMLC_NODE_HOST": "127.0.0.1", "DMLC_GROUP_SIZE": "1", "DMLC_LOCAL": "1",
                    "NUM_KEY_PER_SERVER": str(args.keys_per_server),
                    "LOG_DURATION": str(args.steps),
                    "TOTAL_DURATION": str(args.steps * (1 + max(1, -(-args.warmup // args.steps))))})
        for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK", "MASTER_ADDR", "MASTER_PORT"):
            env.pop(k, None)
        cmd = [res["bin"], str(args.len), "10", "1"]
        procs, logs = [], []
        t0 = time.time()
        for role, n in (("scheduler", 1), ("server", S), ("worker", W)):
            for _ in range(n):
                e = dict(env)
                e["DMLC_ROLE"] = role
                p = subprocess.Popen(cmd, env=e, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
                procs.append((role, p))
        gbps = []
        ok = True
        for role, p in procs:
            try:
                o, _ = p.communicate(timeout=1800)
            except subprocess.TimeoutExpired:
                p.kill()
                o, _ = p.communicate()
                ok = False
            if role == "worker":
                found = reference_goodput(o)
                if found is not None:
                    gbps.append(found)
                else:
                    ok = False
        wall = time.time() - t0
        if ok and len(gbps) == W:
            value = sum(gbps) / 8.0  # Gbps -> GB/s, summed over workers
            payload = float(args.len) * args.keys_per_server * S * W
            out = {"impl": "reference", "metric": METRIC_NAME["pushpull"], "value": value,
                   "unit": "GB/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                   "ms_per_step": payload / (value * 1e9) * 1e3, "higher_is_better": True,
                   "scaling": "weak", "vs_baseline": None, "dtype": "uint8 payload", "data": "synthetic",
                   "config": {"model": "test_benchmark PUSH_PULL", "msg_bytes": args.len,
                              "keys_per_server": args.keys_per_server, "num_workers": W,
                              "num_servers": S, "global_batch": args.keys_per_server * S * W,
                              "seq_len": args.len,
                              "parallelism": f"{W}w+{S}s processes, reference ZMQ van over ipc:// with CPU buffers "
                                             "(its RDMA/UCX vans need ibverbs/UCX, absent in this image; ZMQ cannot carry device pointers)"},
                   "timing": "host clock inside the reference binary (its own goodput print), last LOG_DURATION window",
                   # the reference's buffers live in host memory: its goodput IS host-to-host end to end
                   "e2e": {"value": value, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                           "note": "values start and end in host memory; no device involved"},
                   "wall_s": wall, "gpu_launches": 0}
        else:
            out = {"impl": "reference", "unavailable": "reference test_benchmark did not report goodput"}
    dist.barrier()
    return out


def main():
    args = parse_args()
    if args.impl != "reference":
        # a wedged run should say where it is stuck instead of dying silently under the caller's
        # timeout: after PS_BENCH_WATCHDOG_S seconds dump every Python thread's stack and exit
        import faulthandler

        faulthandler.dump_traceback_later(int(os.environ.get("PS_BENCH_WATCHDOG_S", "1500")), exit=True)
    dist = Dist()
    if args.gpus != dist.world and dist.world > 1:
        args.gpus = dist.world
    if args.impl == "reference":
        out = run_reference(args, dist)
    elif args.impl == "nccl-ddp":
        args.metric = "llama"
        out = run_llama_ddp(args, dist)
    elif args.metric == "llama":
        out = run_llama(args, dist)
    elif args.metric == "resnet":
        out = run_resnet(args, dist)
    else:
        out = run_pushpull(args, dist)
    if dist.rank == 0 and out is not None:
        out.setdefault("impl", "ours")
        out.setdefault("n_gpus", args.gpus)
        out.setdefault("steps", args.steps)
        out.setdefault("warmup", args.warmup)
        print(json.dumps(out), flush=True)
    if args.impl != "reference":
        import faulthandler

        faulthandler.cancel_dump_traceback_later()
    dist.shutdown()


if __name__ == "__main__":
    main()
