"""Row-sparse shards (embedding tables): the fused rows update and the server engine around it.

`fused_update_rows` is checked against an independent float64 reference (tests/helpers/rows_ref.py)
with lazy semantics: only rows some slot pushed are stepped, every other row of master, m, v and of
every destination stays bit for bit. Guard bytes around every buffer catch stray writes. Each case
runs on the CPU twin (`cpu`) and on the sm_100a kernels (`cuda`, marked gpu); on the GPU the kernel
is also compared with the twin and with itself (two launches on the same inputs).
"""
import os
import sys

import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "helpers"))

from rows_ref import GRAD_BF16, GRAD_F32, GRAD_FP8BLOCK, make_slot, reference_round  # noqa: E402

GUARD = 256
SENTINEL = 0xA5
FMTS = {"f32": GRAD_F32, "bf16": GRAD_BF16, "fp8": GRAD_FP8BLOCK}
DEVICES = [pytest.param("cpu", id="cpu"), pytest.param("cuda", id="cuda", marks=pytest.mark.gpu)]


def _require(device):
    if device == "cuda" and not torch.cuda.is_available():
        pytest.skip("no CUDA device")


def _f32(x):
    return float(torch.tensor(x, dtype=torch.float32))


class Guarded:
    """`bytes` starts GUARD bytes into a buffer filled with `fill`, and GUARD sentinel bytes follow it"""

    def __init__(self, nbytes, device, fill=SENTINEL):
        self.buf = torch.full((GUARD + nbytes + GUARD,), SENTINEL, dtype=torch.uint8, device=device)
        self.bytes = self.buf[GUARD:GUARD + nbytes]
        self.bytes.fill_(fill)

    def view(self, dtype):
        return self.bytes.view(dtype)

    def guards_intact(self):
        return bool((self.buf[:GUARD] == SENTINEL).all()) and bool((self.buf[-GUARD:] == SENTINEL).all())


def _row_sets(pattern, rows, W, gen, r_max):
    """W lists of unique row ids (int64), shaped by `pattern`"""
    def pick(k):
        return torch.randperm(rows, generator=gen)[:k].sort().values
    k = min(rows, r_max)
    if pattern == "identical":
        s = pick(k)
        return [s.clone() for _ in range(W)]
    if pattern == "disjoint":
        perm = torch.randperm(rows, generator=gen)
        per = max(1, min(k, rows // W))
        return [perm[w * per:(w + 1) * per].sort().values if (w + 1) * per <= rows else perm[:0]
                for w in range(W)]
    if pattern == "empty":  # every other slot pushes nothing
        return [pick(k) if w % 2 else torch.zeros(0, dtype=torch.int64) for w in range(W)]
    if pattern == "all_empty":
        return [torch.zeros(0, dtype=torch.int64) for _ in range(W)]
    if pattern == "full":  # every slot pushes every row: the union is the whole table
        return [torch.arange(rows) for _ in range(W)]
    # overlapping: random subsets of about a third of the rows each
    return [torch.randperm(rows, generator=gen)[:max(1, min(k, rows // 3))] for _ in range(W)]


def run_rows_case(C, device, rows, dim, W, fmt, optimizer="adamw", rounds=4, pattern="overlapping",
                  n_outs=1, out_f32=False, max_ctas=0, r_max=1 << 30, bad_ids=False, seed=0, twin_check=False):
    """runs `rounds` rounds of fused_update_rows and checks every invariant; returns the final state"""
    gen = torch.Generator().manual_seed(seed)
    n = rows * dim
    adam = optimizer == "adamw"
    lr, b1, b2, eps = _f32(1e-2), _f32(0.9), _f32(0.95), _f32(1e-8)
    wd = _f32(0.1) if not adam else _f32(0.01)
    gs = _f32(1.0 / W)
    opt = dict(optimizer=optimizer, lr=lr, beta1=b1, beta2=b2, eps=eps, weight_decay=wd, grad_scale=gs)
    if not adam:
        opt["beta1"] = _f32(0.9)

    st = {k: Guarded(n * 4, device) for k in ("master", "m", "v")}
    master, m, v = (st[k].view(torch.float32) for k in ("master", "m", "v"))
    master.copy_(torch.randn(n, generator=gen).to(device))
    m.zero_()
    v.zero_()
    ref = {k: t.double().reshape(rows, dim).clone() for k, t in (("master", master), ("m", m), ("v", v))}
    osz = 4 if out_f32 else 2
    outs_g = [Guarded(n * osz, device) for _ in range(n_outs)]
    outs = [o.view(torch.float32 if out_f32 else torch.bfloat16) for o in outs_g]
    scratch_g = Guarded(C.rows_scratch_bytes(rows, W), device, fill=0)
    scratch = scratch_g.bytes
    expect_outs = [o.clone() for o in outs]  # all sentinel
    bad_total = 0
    fmt_id = FMTS[fmt]
    col_mag = torch.logspace(-3, 1, dim)

    for step in range(1, rounds + 1):
        sets = _row_sets(pattern, rows, W, gen, r_max)
        if bad_ids:  # one out-of-range id and one repeat in slot 0
            s0 = sets[0]
            extra = [rows + 3]
            if len(s0):
                extra.append(int(s0[0]))
            sets[0] = torch.cat([s0, torch.tensor(extra, dtype=torch.int64)])
        # the contributions to one element share a sign, so fp32 and fp64 sums cannot differ in sign
        sign = (torch.randint(0, 2, (rows, dim), generator=gen) * 2 - 1).float()
        slot_bufs, slot_ref = [], []
        for ids in sets:
            safe = ids.clamp(max=rows - 1)
            vals = sign[safe] * col_mag * torch.rand(len(ids), dim, generator=gen) * 0.05
            raw, read = make_slot(C, ids.to(device), vals.to(device), fmt_id)
            g = Guarded(raw.numel(), device)
            g.bytes.copy_(raw)
            slot_bufs.append(g)
            slot_ref.append((ids, read.to(device)))
        before = {k: t.clone() for k, t in (("master", master), ("m", m), ("v", v))}
        slots_before = [b.buf.clone() for b in slot_bufs]

        def launch(mst, mm, vv, oo, scr):
            C.fused_update_rows([b.bytes for b in slot_bufs], [len(s) for s in sets], fmt_id, dim, mst, mm, vv,
                                oo, scr, optimizer=optimizer, lr=lr, beta1=opt["beta1"], beta2=b2, eps=eps,
                                weight_decay=wd, step=step, grad_scale=gs, max_ctas=max_ctas)
            if device == "cuda":
                torch.cuda.synchronize()

        if device == "cuda":
            # a second launch on copies of the same inputs must agree bit for bit
            cp = [t.clone() for t in (master, m, v)]
            co = [o.clone() for o in outs]
            cs = scratch.clone()
            launch(cp[0], cp[1], cp[2], co, cs)
        if twin_check:
            tw = [t.cpu().clone() for t in (master, m, v)]
            tw_scr = scratch.cpu().clone()
            C.fused_update_rows([b.bytes.cpu() for b in slot_bufs], [len(s) for s in sets], fmt_id, dim, tw[0],
                                tw[1], tw[2], [], tw_scr, optimizer=optimizer, lr=lr, beta1=opt["beta1"],
                                beta2=b2, eps=eps, weight_decay=wd, step=step, grad_scale=gs)
        launch(master, m, v, outs, scratch)
        union, bad = reference_round(ref, slot_ref, opt, step, dim)
        bad_total += bad

        if device == "cuda":
            for a, b in zip(cp, (master, m, v)):
                assert torch.equal(a, b), f"round {step}: two launches on the same inputs differ"
            for a, b in zip(co, outs):
                assert torch.equal(a, b), f"round {step}: two launches wrote different outputs"
        # exact invariants: guards, slots, untouched rows, destinations, scratch
        for k, b in st.items():
            assert b.guards_intact(), f"round {step}: a write landed next to {k}"
        for i, b in enumerate(outs_g):
            assert b.guards_intact(), f"round {step}: a write landed next to output {i}"
        assert scratch_g.guards_intact(), f"round {step}: a write landed next to the scratch"
        for i, b in enumerate(slot_bufs):
            assert torch.equal(b.buf, slots_before[i]), f"round {step}: gradient slot {i} changed"
        touched = torch.zeros(rows, dtype=torch.bool)
        if union:
            touched[torch.tensor(union)] = True
        untouched = (~touched).to(device)
        for k, t in (("master", master), ("m", m), ("v", v)):
            assert torch.equal(t.view(rows, dim)[untouched], before[k].view(rows, dim)[untouched]), \
                f"round {step}: an untouched row of {k} changed"
        if not adam:
            assert torch.equal(v, before["v"]), f"round {step}: SGD wrote v"
        tdev = touched.to(device)
        for i, o in enumerate(outs):
            e = expect_outs[i].view(rows, dim)
            e[tdev] = master.view(rows, dim)[tdev].to(e.dtype)
            assert torch.equal(o, expect_outs[i]), f"round {step}: output {i} is not the updated rows (only)"
        hdr = scratch[:16].cpu()
        assert int(hdr[:8].view(torch.int32)[0]) == 0, "the union count was not reset for the next round"
        assert int(hdr[8:16].view(torch.int64)[0]) == bad_total, f"round {step}: bad-id count"
        # touched[rows] and slot_of[W][rows] must be clean for the next round (list[] past count is dead)
        words = scratch[16:].view(torch.int32)
        assert int(words[:rows].count_nonzero()) == 0 and int(words[2 * rows:].count_nonzero()) == 0, \
            f"round {step}: the scratch was not left clean"
        if twin_check:
            for a, b, name in zip(tw, (master, m, v), ("master", "m", "v")):
                # same summation order and decode; the kernel's MUFU sqrt / reciprocal differ from the
                # twin's IEEE ones by a few ulp of one step's update
                torch.testing.assert_close(b.cpu(), a, rtol=2e-6, atol=1e-7, msg=lambda s: f"twin {name}: {s}")

        # against float64: the tolerances of the dense update tests, times the round count
        for k, t, atol in (("master", master, 1e-6), ("m", m, 1e-7), ("v", v, 1e-9)):
            if k == "v" and not adam:
                continue
            torch.testing.assert_close(t.double().view(rows, dim), ref[k], rtol=1e-5 * step, atol=atol * step,
                                       msg=lambda s: f"round {step} {k}: {s}")
    return master, m, v


# ---------------------------------------------------------------------------------------------
# kernel + CPU twin
# ---------------------------------------------------------------------------------------------
def _small_cases():
    cases = []
    for fmt in ("f32", "bf16", "fp8"):
        for W, pattern in ((1, "overlapping"), (2, "disjoint"), (3, "identical"), (4, "empty"),
                           (8, "overlapping"), (5, "all_empty")):
            cases.append(dict(fmt=fmt, W=W, pattern=pattern, optimizer="adamw", rounds=4))
        cases.append(dict(fmt=fmt, W=3, pattern="overlapping", optimizer="sgd", rounds=3))
    cases.append(dict(fmt="bf16", W=2, pattern="overlapping", optimizer="adamw", rounds=2, dim=8))
    cases.append(dict(fmt="f32", W=6, pattern="overlapping", optimizer="sgd", rounds=3, dim=8))
    return [pytest.param(c, id="{fmt}-W{W}-{pattern}-{optimizer}-D{d}".format(d=c.get("dim", 64), **c))
            for c in cases]


@pytest.mark.parametrize("device", DEVICES)
@pytest.mark.parametrize("case", _small_cases())
def test_update_rows_matches_fp64(native, device, case):
    _require(device)
    case = dict(case)
    dim = case.pop("dim", 64)
    run_rows_case(native, device, rows=96, dim=dim, n_outs=2, twin_check=device == "cuda", **case)


@pytest.mark.parametrize("device", DEVICES)
@pytest.mark.parametrize("fmt", ["f32", "bf16", "fp8"])
def test_update_rows_counts_bad_ids(native, device, fmt):
    """an id >= rows and an id repeated within a slot are skipped and counted, and nothing is written
    for them (the guards and the untouched-row checks inside run_rows_case)"""
    _require(device)
    run_rows_case(native, device, rows=64, dim=32, W=3, fmt=fmt, rounds=2, bad_ids=True, n_outs=1)


@pytest.mark.parametrize("device", DEVICES)
@pytest.mark.parametrize("n_outs,out_f32,max_ctas", [(0, False, 0), (9, False, 0), (1, True, 0), (2, False, 1)])
def test_update_rows_fanout_and_grid(native, device, n_outs, out_f32, max_ctas):
    _require(device)
    run_rows_case(native, device, rows=200, dim=64, W=4, fmt="bf16", rounds=2, n_outs=n_outs, out_f32=out_f32,
                  max_ctas=max_ctas)


def test_update_rows_validates_arguments(native):
    C = native
    rows, dim = 16, 32
    master, m, v = (torch.zeros(rows * dim) for _ in range(3))
    scratch = torch.zeros(C.rows_scratch_bytes(rows, 2), dtype=torch.uint8)
    slot = torch.zeros(C.rows_slot_bytes(4, dim, GRAD_BF16), dtype=torch.uint8)

    def call(**kw):
        args = dict(grads=[slot], num_rows=[4], grad_format=GRAD_BF16, dim=dim, master=master, m=m, v=v, outs=[],
                    scratch=scratch)
        args.update(kw)
        C.fused_update_rows(**args)

    call()
    with pytest.raises(RuntimeError, match="row counts"):
        call(num_rows=[4, 4])
    with pytest.raises(RuntimeError, match="1 to 8 gradient slots"):
        call(grads=[slot] * 9, num_rows=[0] * 9)
    with pytest.raises(RuntimeError, match="multiple of 8"):
        call(dim=12, master=torch.zeros(12 * 4))
    with pytest.raises(RuntimeError, match="multiple of 32"):
        call(dim=8, grad_format=GRAD_FP8BLOCK, master=torch.zeros(8 * 4))
    with pytest.raises(RuntimeError, match="whole number of rows"):
        call(master=torch.zeros(rows * dim + 8))
    with pytest.raises(RuntimeError, match="rows need"):
        call(num_rows=[5])
    with pytest.raises(RuntimeError, match="scratch holds"):
        call(scratch=scratch[:16])
    with pytest.raises(RuntimeError, match="v must be float32"):
        call(v=torch.zeros(8))
    with pytest.raises(RuntimeError, match="must be contiguous"):
        call(m=torch.zeros(rows * dim * 2)[::2])
    with pytest.raises(RuntimeError, match="bfloat16 or all float32"):
        call(outs=[torch.zeros(rows * dim, dtype=torch.float16)])
    with pytest.raises(RuntimeError, match="elements, master"):
        call(outs=[torch.zeros(rows * dim - 1, dtype=torch.bfloat16)])
    with pytest.raises(RuntimeError, match="step count starts at 1"):
        call(step=0)


@pytest.mark.gpu
@pytest.mark.parametrize("rows,dim,W,fmt,pattern,r_max,n_outs,max_ctas", [
    pytest.param(8192, 4096, 2, "fp8", "full", 1 << 30, 1, 0, id="8192x4096-full-union-fp8"),
    pytest.param(1 << 21, 16, 4, "bf16", "overlapping", 4096, 1, 0, id="2M-rows-x16-sparse-bf16"),
    pytest.param(1024, 8192, 3, "f32", "overlapping", 300, 9, 0, id="1024x8192-f32-fanout9"),
    pytest.param(4096, 8, 8, "bf16", "overlapping", 1 << 30, 1, 1, id="4096x8-W8-one-cta"),
    pytest.param(2048, 64, 8, "fp8", "identical", 512, 1, 0, id="2048x64-W8-identical-fp8"),
])
def test_update_rows_real_shapes_gpu(native, rows, dim, W, fmt, pattern, r_max, n_outs, max_ctas):
    _require("cuda")
    run_rows_case(native, "cuda", rows=rows, dim=dim, W=W, fmt=fmt, rounds=2, pattern=pattern, r_max=r_max,
                  n_outs=n_outs, max_ctas=max_ctas, twin_check=True)


@pytest.mark.gpu
def test_update_rows_refuses_misaligned_pointers(native):
    _require("cuda")
    C = native
    rows, dim = 64, 32
    dev = "cuda"
    master, m, v = (torch.zeros(rows * dim, device=dev) for _ in range(3))
    scratch = torch.zeros(C.rows_scratch_bytes(rows, 1), dtype=torch.uint8, device=dev)
    nbytes = C.rows_slot_bytes(4, dim, GRAD_BF16)
    slot = torch.zeros(nbytes + 16, dtype=torch.uint8, device=dev)
    out = torch.zeros(rows * dim + 8, dtype=torch.bfloat16, device=dev)

    def call(grads, outs, mm=m):
        C.fused_update_rows(grads, [4], GRAD_BF16, dim, master, mm, v, outs, scratch)
        torch.cuda.synchronize()

    call([slot[:nbytes]], [out[:rows * dim]])
    with pytest.raises(RuntimeError, match="misaligned"):
        call([slot[4:4 + nbytes]], [])
    with pytest.raises(RuntimeError, match="misaligned"):
        call([slot[:nbytes]], [out[1:1 + rows * dim]])
    with pytest.raises(RuntimeError, match="misaligned"):
        big = torch.zeros(rows * dim + 1, device=dev)
        call([slot[:nbytes]], [], mm=big[1:])


# ---------------------------------------------------------------------------------------------
# the server engine and the trainer, end to end
# ---------------------------------------------------------------------------------------------
def _torchrun(helper, nproc, args, cuda=False, timeout=280):
    """runs a helper under torchrun in its own session and kills whatever of it is left afterwards"""
    import signal
    import subprocess

    from pslite_b200.utils.env import free_port

    env = dict(os.environ)
    env.update({"PSLITE_NO_AUTOBUILD": "1", "OMP_NUM_THREADS": "1"})
    if not cuda:
        env["CUDA_VISIBLE_DEVICES"] = ""
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={nproc}",
           "--master-addr", "127.0.0.1", "--master-port", str(free_port()), os.path.join(HERE, "helpers", helper)]
    p = subprocess.Popen(cmd + [str(a) for a in args], env=env, cwd=os.path.dirname(HERE), stdout=subprocess.PIPE,
                         stderr=subprocess.STDOUT, text=True, start_new_session=True)
    try:
        out, _ = p.communicate(timeout=timeout)
    finally:
        try:
            os.killpg(p.pid, signal.SIGKILL)
        except ProcessLookupError:
            pass
        p.wait()
    return p.returncode, out


@pytest.mark.timeout(300)
@pytest.mark.parametrize("van", ["shm", "zmq"])
def test_sparse_embedding_training_matches_sparse_adam(native, van):
    """tiny Llama, sparse_embedding=True, 2 workers + 2 servers on the host engine: the parameters match
    SparseAdam (embedding) + AdamW (rest) run in one process, not dense AdamW; untouched rows keep their
    bits; every replica equals bf16 of its server's master. zmq is the TCP van: its pulls are answered
    two-sided with the whole chunk."""
    rc, out = _torchrun("train_rows.py", 2, [van, "bf16", 6])
    assert rc == 0 and "PASS" in out, out[-3000:]


@pytest.mark.timeout(300)
def test_sparse_embedding_training_fp8_rows(native):
    rc, out = _torchrun("train_rows.py", 2, ["shm", "fp8", 5])
    assert rc == 0 and "PASS" in out, out[-3000:]


@pytest.mark.timeout(300)
def test_row_push_reuses_its_landing_slot(native):
    """ten steps with a different number of rows every step: one slot rendezvous per (worker, key)"""
    rc, out = _torchrun("train_rows.py", 2, ["shm", "fp8", 10, "slots"])
    assert rc == 0 and "PASS" in out and "push_slot_rendezvous=4 keys=4" in out, out[-3000:]


@pytest.mark.timeout(200)
@pytest.mark.parametrize("mode", ["async", "ckpt"])
def test_row_shard_server_behaviour(native, mode):
    rc, out = _torchrun("rows_server.py", 1, [mode, "shm"])
    assert rc == 0 and "PASS" in out, out[-3000:]


@pytest.mark.timeout(200)
@pytest.mark.parametrize("mode,message", [
    ("err_dense", "is a dense shard: it takes kCmdGrad pushes, not kCmdGradRows"),
    ("err_dim", "the row width 12 is not a multiple of 8"),
])
def test_row_shard_server_refuses_bad_requests(native, mode, message):
    rc, out = _torchrun("rows_server.py", 1, [mode, "shm"])
    assert rc != 0 and message in out, out[-3000:]


@pytest.mark.gpu
@pytest.mark.timeout(300)
@pytest.mark.parametrize("mode", ["async", "ckpt"])
def test_row_shard_server_behaviour_gpu(native, mode):
    _require("cuda")
    rc, out = _torchrun("rows_server.py", 1, [mode, "nvl"], cuda=True)
    assert rc == 0 and "PASS" in out, out[-3000:]


@pytest.mark.gpu
@pytest.mark.timeout(300)
@pytest.mark.parametrize("wire", ["bf16", "fp8"])
def test_sparse_embedding_training_gpu(native, wire):
    """worker and server co-located on one GPU (nvl van): row pushes land one-sidedly in HBM, the rows
    kernel steps the union and writes the touched rows into the worker's parameter"""
    _require("cuda")
    rc, out = _torchrun("train_rows.py", 1, ["nvl", wire, 6], cuda=True)
    assert rc == 0 and "PASS" in out and "replica_equals_master=True" in out, out[-3000:]


@pytest.mark.gpu
@pytest.mark.timeout(300)
def test_row_push_reuses_its_landing_slot_gpu(native):
    _require("cuda")
    rc, out = _torchrun("train_rows.py", 1, ["nvl", "fp8", 10, "slots"], cuda=True)
    assert rc == 0 and "PASS" in out, out[-3000:]


@pytest.mark.gpu
@pytest.mark.timeout(300)
def test_sparse_embedding_training_two_gpus(native):
    _require("cuda")
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    rc, out = _torchrun("train_rows.py", 2, ["nvl", "bf16", 6], cuda=True)
    assert rc == 0 and "PASS" in out, out[-3000:]


def test_dense_gradient_on_row_sparse_parameter_is_refused(native):
    from pslite_b200.parallel.ps_trainer import PSWorkerOptimizer

    class NoNetwork:  # the hook must refuse the gradient before anything is sent
        def server_key(self, server, j):
            return j

    emb = torch.nn.Embedding(16, 8)  # sparse=False: dense gradients
    opt = PSWorkerOptimizer([emb.weight], NoNetwork(), 1, 1, 0, chunk_elems=1024, row_sparse=[emb.weight]).attach()
    assert [(c.start, c.stop, c.dim) for c in opt.chunks[0]] == [(0, 128, 8)]
    with pytest.raises(ValueError, match="row_sparse but its gradient is dense"):
        emb(torch.tensor([1, 3])).sum().backward()


def test_row_sparse_chunks_are_whole_rows(native):
    from pslite_b200.parallel.ps_trainer import PSWorkerOptimizer

    class NoNetwork:
        def server_key(self, server, j):
            return 1000 * server + j

    emb = torch.nn.Embedding(100, 48, sparse=True)
    lin = torch.nn.Linear(48, 4)
    params = [emb.weight] + list(lin.parameters())
    opt = PSWorkerOptimizer(params, NoNetwork(), 2, 1, 0, chunk_elems=1024, row_sparse=[emb.weight])
    rows_per_key = 1024 // 48
    assert [(c.start, c.stop) for c in opt.chunks[0]] == [
        (a * 48, min(100, a + rows_per_key) * 48) for a in range(0, 100, rows_per_key)]
    assert all(c.dim == 48 for c in opt.chunks[0]) and all(c.dim == 0 for per in opt.chunks[1:] for c in per)
