"""Row-sparse embedding training through the PS, checked against single-process torch optimizers.

usage: torchrun --nproc-per-node=2 train_rows.py <van> <grad_wire> <steps> [llama|slots]
Joint topology: every rank is a worker and a server (2 workers + 2 servers for 2 ranks).

llama  tiny Llama with `sparse_embedding=True`; the embedding travels as row-sparse pushes
       (`row_sparse=[embed.weight]`). Rank 0 replays the job in one process with
       torch.optim.SparseAdam (embedding) + torch.optim.AdamW (everything else, weight decay 0)
       on the same seeded batches and compares parameters. Token ids stay below TOUCHED, so the
       rows above it are never pushed (empty pushes) and must keep their initial bits.
slots  one embedding table, fp8 rows, a different number of touched rows every step: every
       (worker, key) pair makes exactly one landing-slot rendezvous (SendOpts::slot_bytes).
"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

import pslite_b200  # noqa: E402
from pslite_b200.models.llama import Llama, LlamaConfig  # noqa: E402
from pslite_b200.parallel.launch import init_ps  # noqa: E402
from pslite_b200.parallel.ps_trainer import PSWorkerOptimizer  # noqa: E402
from rows_ref import make_slot  # noqa: E402

LR, B1, B2, EPS = 3e-3, 0.9, 0.95, 1e-8
TOUCHED = 200  # token ids < TOUCHED; vocab 512


def batch(rank, step, dev, cfg):
    g = torch.Generator(device=dev).manual_seed(1000 * rank + step)
    tok = torch.randint(0, TOUCHED, (2, 33), device=dev, generator=g)
    return tok[:, :-1], tok[:, 1:]


def make_model(dev):
    cfg = LlamaConfig.tiny(sparse_embedding=True)
    with torch.device(dev):
        model = Llama(cfg).to(torch.bfloat16)
    model.init_weights(seed=3)
    return model, cfg


def reference(W, steps, dev, lazy=True):
    """the same job in one process: bf16 model = bf16(fp32 master), gradients averaged over the W
    workers in fp32, SparseAdam for the embedding (lazy; with lazy=False dense AdamW on the
    densified gradient, for contrast), AdamW for the rest"""
    model, cfg = make_model(dev)
    params = list(model.parameters())
    master = [p.detach().float().clone().requires_grad_(True) for p in params]
    emb = [i for i, p in enumerate(params) if p is model.embed.weight][0]
    sparse_opt = (torch.optim.SparseAdam([master[emb]], lr=LR, betas=(B1, B2), eps=EPS) if lazy else
                  torch.optim.AdamW([master[emb]], lr=LR, betas=(B1, B2), eps=EPS, weight_decay=0.0, foreach=False))
    dense_opt = torch.optim.AdamW([m for i, m in enumerate(master) if i != emb], lr=LR, betas=(B1, B2), eps=EPS,
                                  weight_decay=0.0, foreach=False)
    for s in range(steps):
        acc = [None] * len(params)
        for r in range(W):
            model.zero_grad(set_to_none=True)
            x, y = batch(r, s, dev, cfg)
            model(x, y).backward()
            for i, p in enumerate(params):
                g = p.grad.float()
                acc[i] = g if acc[i] is None else acc[i] + g
        for i, m in enumerate(master):
            g = acc[i].coalesce() if acc[i].is_sparse else acc[i]
            m.grad = (g if lazy or not g.is_sparse else g.to_dense()) * (1.0 / W)
        sparse_opt.step()
        dense_opt.step()
        with torch.no_grad():
            for p, m in zip(params, master):
                p.copy_(m.to(torch.bfloat16))
    return [p.detach().clone() for p in params]


def main():
    van, wire, steps = sys.argv[1], sys.argv[2], int(sys.argv[3])
    mode = sys.argv[4] if len(sys.argv) > 4 else "llama"
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", rank))
    use_cuda = van == "nvl"
    dist.init_process_group("gloo")
    C = pslite_b200.native()
    if use_cuda:
        torch.cuda.set_device(local % torch.cuda.device_count())
    dev = torch.device("cuda", torch.cuda.current_device()) if use_cuda else torch.device("cpu")
    ctx = init_ps("joint", van=van)
    W = ctx.num_workers
    server = C.GpuServer(0, num_workers=W, optimizer="adamw", lr=LR, beta1=B1, beta2=B2, eps=EPS, weight_decay=0.0,
                         grad_scale=1.0 / W, fuse_pull=True)
    dist.barrier()
    kv = C.KVWorker(0, 0)
    ok = True
    msg = ""
    if mode == "slots":
        # raw row pushes from a buffer the van can write one-sidedly (device memory, or exportable shared
        # memory on a CPU run), R changing every step; the landing slot is requested at the buffer's size
        rows, dim, keys = 1024, 64, 4
        per = rows // keys
        fmt = C.GRAD_FP8BLOCK if wire == "fp8" else C.GRAD_BF16
        cap = C.rows_slot_bytes(per, dim, fmt)
        keyids = [kv.server_key(j % ctx.num_servers, j) for j in range(keys)]
        bufs = [torch.zeros(cap, dtype=torch.uint8, device=dev) if use_cuda else C.alloc_exportable(cap, "worker")
                for _ in keyids]
        table = torch.zeros(rows * dim, dtype=torch.bfloat16, device=dev)
        if ctx.worker_rank == 0:
            ts = [kv.push(k, table[j * per * dim:(j + 1) * per * dim], cmd=C.CMD_INIT_BF16,
                          option=C.INIT_ROW_SPARSE | (dim << 8)) for j, k in enumerate(keyids)]
            for t in ts:
                kv.wait(t)
        C.barrier(0, C.WORKER_GROUP, "worker")
        g = torch.Generator().manual_seed(7 + rank)
        for s in range(steps):
            ts = []
            for j, k in enumerate(keyids):
                r = (s * 37 + rank * 11 + j * 5) % per  # a different number of rows every step (0 included)
                ids = torch.randperm(per, generator=g)[:r].sort().values
                vals = torch.randn(r, dim, generator=g)
                raw, _ = make_slot(C, ids, vals, fmt)
                n = max(16, raw.numel())
                bufs[j][:raw.numel()].copy_(raw.to(dev))
                ts.append(kv.push(k, bufs[j][:n], cmd=C.CMD_GRAD_ROWS, option=(r << 2) | fmt, slot_bytes=cap))
                ts.append(kv.pull(k, table[j * per * dim:(j + 1) * per * dim]))
            for t in ts:
                kv.wait(t)
        rv = C.van_stats("worker").get("push_slot_rendezvous", -1)
        ok = rv == keys and bool(torch.isfinite(table.float()).all())
        msg = f"push_slot_rendezvous={rv} keys={keys}"
    else:
        model, cfg = make_model(dev)
        init = [p.detach().clone() for p in model.parameters()]
        opt = PSWorkerOptimizer(model.parameters(), kv, ctx.num_servers, W, ctx.worker_rank, grad_wire=wire,
                                chunk_elems=1 << 14, row_sparse=[model.embed.weight]).attach()
        opt.init_parameters(barrier=lambda: C.barrier(0, C.WORKER_GROUP, "worker"))
        wire_bytes = []
        for s in range(steps):
            before = opt.stats.push_bytes_wire
            x, y = batch(ctx.worker_rank, s, dev, cfg)
            model(x, y).backward()
            opt.step()
            wire_bytes.append(opt.stats.push_bytes_wire - before)
        opt.wait_all()
        if use_cuda:
            torch.cuda.synchronize()
        emb = model.embed.weight.detach()
        # rows no batch touched: never stepped, never rewritten
        ok = torch.equal(emb[TOUCHED:], init[0][TOUCHED:])
        msg += f"untouched_rows_bit_identical={ok} "
        ref = reference(W, steps, dev) if wire == "bf16" else None
        if ref is not None:
            # fp32 state on both sides with different rounding: once a bf16 parameter lands on the neighbouring
            # bf16 value, later gradients differ a little and Adam's normalised step amplifies that, so single
            # elements may end a few learning rates apart. Bound those, and require the embedding to be far
            # closer to the lazy (SparseAdam) result than to dense AdamW on the same gradients.
            dense = reference(W, steps, dev, lazy=False)
            worst = max((p.float() - r.float()).abs().max().item() for p, r in zip(model.parameters(), ref))
            e = model.embed.weight.float()
            d_lazy = (e - ref[0].float()).norm().item()
            d_dense = (e - dense[0].float()).norm().item()
            ok = ok and worst <= 4 * LR and d_lazy <= 0.25 * d_dense
            msg += f"vs_torch_max_abs={worst:.2e} embed_dist_lazy={d_lazy:.3e} embed_dist_dense_adamw={d_dense:.3e} "
        # the embedding's row pushes stay far below a dense push of the table
        dense_emb = model.embed.weight.numel() * 2
        msg += f"push_bytes_wire/step={wire_bytes[-1]} dense_embedding_bf16={dense_emb} "
        # every replica equals bf16 of the master of the server that owns the chunk (this rank checks the
        # chunks of its own server; the checksums below tie the workers' replicas together)
        replica_ok = True
        for p, per in zip(model.parameters(), opt.chunks):
            flat = p.detach().reshape(-1)
            for c in per:
                if c.server == ctx.server_rank:
                    want = server.read_master(c.key).to(torch.bfloat16).to(dev)
                    replica_ok = replica_ok and torch.equal(flat[c.start:c.stop], want)
        ok = ok and replica_ok and server.num_bad_rows() == 0
        msg += f"replica_equals_master={replica_ok} bad_rows={server.num_bad_rows()}"
    if mode == "llama":
        chk = torch.tensor([sum(float(p.double().sum()) for p in model.parameters())], dtype=torch.float64)
        sums = [torch.zeros(1, dtype=torch.float64) for _ in range(world)]
        dist.all_gather(sums, chk)
        same = all(float(x) == float(sums[0]) for x in sums)
        ok = ok and same
        msg += f" checksums_equal={same}"
    print(f"rank {rank}: {'ok' if ok else 'MISMATCH'} {msg}", flush=True)
    flag = torch.tensor([1.0 if ok else 0.0])
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    ctx.shutdown()
    dist.destroy_process_group()
    if rank == 0:
        print("PASS" if flag.item() > 0 else "FAIL", flush=True)
    sys.exit(0 if flag.item() > 0 else 1)


if __name__ == "__main__":
    main()
