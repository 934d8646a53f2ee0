"""The server engine with row-sparse shards, driven by raw pushes from one worker in the same process.

usage: torchrun --nproc-per-node=1 rows_server.py <mode> <van>
  async      async_updates: every kCmdGradRows push is its own optimizer step (W = 1, no outputs)
  ckpt       save / load a checkpoint holding a row shard and a dense shard; a row shard keeps its
             row width across the checkpoint; a file in the format written before row shards existed
             (dense keys only) still loads
  err_dense  kCmdGradRows to a dense shard: the server refuses it with a message
  err_dim    a row shard whose row width is not a multiple of 8: refused at init
Prints PASS when every check holds.
"""
import os
import struct
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, HERE)

import torch  # noqa: E402

import pslite_b200  # noqa: E402
from pslite_b200.parallel.launch import init_ps  # noqa: E402
from rows_ref import GRAD_BF16, GRAD_F32, make_slot, reference_round  # noqa: E402

ROWS, DIM = 64, 16
LR = 1e-2


def main():
    mode, van = sys.argv[1], sys.argv[2]
    C = pslite_b200.native()
    use_cuda = van == "nvl"
    dev = torch.device("cuda", 0) if use_cuda else torch.device("cpu")
    ctx = init_ps("joint", van=van)
    server = C.GpuServer(0, num_workers=1, optimizer="adamw", lr=LR, beta1=0.9, beta2=0.95, eps=1e-8,
                         weight_decay=0.0, grad_scale=1.0, fuse_pull=True, async_updates=mode == "async")
    kv = C.KVWorker(0, 0)
    row_key, dense_key = kv.server_key(0, 0), kv.server_key(0, 1)
    gen = torch.Generator().manual_seed(5)
    init = torch.randn(ROWS * DIM, generator=gen)
    replica = torch.zeros(ROWS * DIM, dtype=torch.bfloat16, device=dev)

    def wait(ts):
        kv.wait(ts)

    def push_init(key, dim):
        opt = (C.INIT_ROW_SPARSE | (dim << 8)) if dim else 0
        wait(kv.push(key, init.to(torch.bfloat16).to(dev), cmd=C.CMD_INIT_BF16, option=opt))

    def push_rows(key, ids, fmt=GRAD_F32):
        vals = torch.randn(len(ids), DIM, generator=gen) * 0.1
        raw, read = make_slot(C, ids, vals, fmt, pad=16)
        ts = [kv.push(key, raw.to(dev), cmd=C.CMD_GRAD_ROWS, option=(len(ids) << 2) | fmt)]
        if mode != "async":  # a synchronous round runs once its worker has also asked for the result
            ts.append(kv.pull(key, replica))
        for t in ts:
            wait(t)
        return read

    ok = True
    if mode == "err_dense":
        push_init(dense_key, 0)
        push_rows(dense_key, torch.tensor([1, 2]))
        ok = False  # not reached: the server refuses the push
    elif mode == "err_dim":
        push_init(row_key, 12)
        ok = False
    elif mode == "async":
        push_init(row_key, DIM)
        ref = {"master": init.to(torch.bfloat16).double().view(ROWS, DIM).clone(),
               "m": torch.zeros(ROWS, DIM, dtype=torch.float64), "v": torch.zeros(ROWS, DIM, dtype=torch.float64)}
        opt = dict(optimizer="adamw", lr=LR, beta1=0.9, beta2=0.95, eps=1e-8, weight_decay=0.0, grad_scale=1.0)
        for step, ids in enumerate([[3, 7, 9], [], [7, 60, 61, 62], [0]], start=1):
            before = server.read_master(row_key).view(ROWS, DIM)
            ids = torch.tensor(ids, dtype=torch.int64)
            read = push_rows(row_key, ids)
            reference_round(ref, [(ids, read)], opt, step, DIM)
            got = server.read_master(row_key).view(ROWS, DIM)
            untouched = torch.ones(ROWS, dtype=torch.bool)
            untouched[ids] = False
            ok = ok and torch.equal(got[untouched], before[untouched])
            ok = ok and torch.allclose(got.double(), ref["master"], rtol=1e-5, atol=1e-6)
        print(f"async: updates={server.num_updates()} ok={ok}", flush=True)
        ok = ok and server.num_updates() == 4 and server.num_bad_rows() == 0
    elif mode == "ckpt":
        push_init(row_key, DIM)
        push_init(dense_key, 0)
        push_rows(row_key, torch.tensor([1, 5, 9]), GRAD_BF16)
        # 3 ids, one out of range and one repeated: 2 bad, the valid rows are applied
        push_rows(row_key, torch.tensor([2, ROWS + 1, 2]), GRAD_BF16)
        bad = server.num_bad_rows()
        ok = bad == 2
        n_all = 2 * ROWS * DIM
        scratch = C.rows_scratch_bytes(ROWS, 1)
        ok = ok and server.state_bytes() == n_all * 12 + scratch
        saved = server.read_master(row_key)
        tmp = tempfile.TemporaryDirectory()
        path = os.path.join(tmp.name, "rows.ckpt")
        ok = ok and server.save(path)
        push_rows(row_key, torch.tensor([1, 2, 3]), GRAD_BF16)
        ok = ok and not torch.equal(server.read_master(row_key), saved)
        ok = ok and server.load(path)
        ok = ok and torch.equal(server.read_master(row_key), saved)
        # still a row shard after the load: row pushes are accepted and only touch their rows
        push_rows(row_key, torch.tensor([4]), GRAD_BF16)
        after = server.read_master(row_key).view(ROWS, DIM)
        keep = torch.ones(ROWS, dtype=torch.bool)
        keep[4] = False
        ok = ok and torch.equal(after[keep], saved.view(ROWS, DIM)[keep])
        with open(path, "rb") as f:
            raw = f.read()
        flags = [struct.unpack_from("<QQii", raw, 16 + i * (24 + 12 * ROWS * DIM)) for i in range(2)]
        row_flag = [e[3] for e in flags if e[0] == row_key][0]
        ok = ok and row_flag == (1 | 4 | (DIM << 8))
        # a file in the format written before row shards existed: dense keys, flag bits 0 and 1 only
        old = os.path.join(os.path.dirname(path), "dense.ckpt")
        n = 40
        vals = [torch.randn(n, generator=gen) for _ in range(3)]
        with open(old, "wb") as f:
            f.write(b"PSB2CKPT" + struct.pack("<Q", 1))
            f.write(struct.pack("<QQii", dense_key + 100, n, 7, 1 | 2))
            for t in vals:
                f.write(t.numpy().tobytes())
        ok = ok and server.load(old) and torch.equal(server.read_master(dense_key + 100), vals[0])
        print(f"ckpt: bad_rows={bad} state_bytes={server.state_bytes()} row_flag={row_flag:#x} ok={ok}", flush=True)
    ctx.shutdown()
    print("PASS" if ok else "FAIL", flush=True)
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
