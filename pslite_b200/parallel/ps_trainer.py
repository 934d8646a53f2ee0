"""Synchronous data-parallel training through the parameter server.

Worker side of the BytePS-style loop the reference is built for (docs/overview.md:60-69:
"workers push gradients, pull weights") written for B200:

* every parameter tensor is cut into chunks (`chunk_elems`, default 32 Mi elements) and
  each chunk is a key; chunk j lives on server j % S (the test_benchmark key encoding);
* gradients are pushed from `post_accumulate_grad` hooks *during backward*: the push is a
  one-sided write into the server's HBM slot issued by an sm_100a kernel on the van's
  stream, fused with the wire transform (block-scaled fp8 by default, or bf16), gated on
  an event recorded on the autograd stream — backward never waits for communication;
* the pull of the same key is issued right behind the push; the server answers it from
  its fused update kernel, which stores the new bf16 parameters straight into
  `param.data` of every worker over NVLink. `step()` only waits for those descriptors;
* gradient tensors are handed to the transport and dropped (`p.grad = None`), so there is
  no flat gradient buffer to zero and backward's peak memory shrinks as it proceeds.

The optimizer state (fp32 master, Adam moments) lives only on the servers, sharded by key.

Embedding tables whose gradients are sparse (`nn.Embedding(sparse=True)`) can be passed as
`row_sparse`: they are chunked on row boundaries, each worker pushes only the rows its batch
touched (ids + values, `CMD_GRAD_ROWS`), and the server steps and rewrites only the union of
those rows ("lazy" AdamW / SGD: untouched rows get no momentum step and no weight decay).

With NVSwitch multicast (`symmetric=True`, `grad_buffer=...`) a whole round is ONE kernel per
shard that never touches NCCL: `multimem.ld_reduce` (the switch sums the W workers' gradient
buffers in fp32) -> AdamW on the fp32 state -> `multimem.st` (the switch replicates the new
bf16 parameters into every worker's `param.data`): reduce-scatter + optimizer + all-gather
fused, tile by tile, over NVLink.
"""
from __future__ import annotations

from dataclasses import dataclass

import torch

from .. import native


@dataclass
class _Chunk:
    key: int
    param_index: int
    start: int
    stop: int
    server: int
    dim: int = 0  # row-sparse parameter: row width (the chunk is whole rows); 0 = dense


@dataclass
class PSTrainerStats:
    pushes: int = 0
    pulls: int = 0
    push_bytes_wire: int = 0
    pull_bytes: int = 0
    keys: int = 0


def _round_up(n: int, m: int) -> int:
    return (n + m - 1) // m * m


def symmetric_layout(params) -> tuple[list[int], int]:
    """Element offsets of every parameter inside the job-wide symmetric bf16 buffer
    (each parameter starts on a 128-byte boundary) and the total element count."""
    offs, cur = [], 0
    for p in params:
        offs.append(cur)
        cur += _round_up(p.numel(), 64)
    return offs, max(cur, 64)


def _native_symmetric() -> bool:
    """PS_SYMM_BACKEND=torch falls back to torch.distributed._symmetric_memory (round-1 behaviour)"""
    import os

    return os.environ.get("PS_SYMM_BACKEND", "native") != "torch"



def setup_symmetric_params(params, total_elems: int, group, device, worker_ranks: list[int],
                           role: str | None = None):
    """Move `params` (may be None on server-only ranks) into a symmetric-memory buffer that
    every rank of `group` allocates identically, rendezvous, and return
    (flat, multicast_ptr, peer_ptrs_of_workers, nbytes). `role` names the van of this process to
    allocate through ("worker" / "server"; default: worker if it has parameters). With NVSwitch multicast support the
    server's update kernel can then publish new parameters to ALL workers with one
    multimem.st stream (NVLS) instead of one unicast stream per worker."""
    if _native_symmetric():
        # the runtime's own allocator (Van::AllocSymmetric: cuMemCreate + POSIX handles over unix
        # sockets + cuMulticast*) — no dependency on torch's private symmetric-memory module
        local, mc, _, _, _, wblocks, _ = native().alloc_symmetric(
            "params", total_elems * 2, role or ("worker" if params is not None else "server"))
        flat = local.view(torch.bfloat16)[:total_elems]
        hdl = local  # keeps the tensor alive next to its views
        if params is not None:
            offs, _ = symmetric_layout(params)
            with torch.no_grad():
                for p, off in zip(params, offs):
                    view = flat[off:off + p.numel()].view(p.shape)
                    view.copy_(p.data)
                    p.data = view
        return flat, hdl, int(mc), [int(wblocks[r]) for r in worker_ranks], total_elems * 2
    import torch.distributed._symmetric_memory as symm_mem

    flat = symm_mem.empty(total_elems, dtype=torch.bfloat16, device=device)
    hdl = symm_mem.rendezvous(flat, group)
    if params is not None:
        offs, _ = symmetric_layout(params)
        with torch.no_grad():
            for p, off in zip(params, offs):
                view = flat[off:off + p.numel()].view(p.shape)
                view.copy_(p.data)
                p.data = view
    mc = int(hdl.multicast_ptr) if getattr(hdl, "multicast_ptr", 0) else 0
    peers = [int(hdl.buffer_ptrs[r]) for r in worker_ranks]
    return flat, hdl, mc, peers, total_elems * 2


def setup_symmetric_grads(total_elems: int, group, device, role: str = "worker"):
    """Second job-wide symmetric bf16 buffer, for gradients (same layout as the parameters).
    Every rank of `group` allocates it zero-filled — server-only ranks never write theirs, so
    they add nothing to the in-switch sum. Returns (flat, handle, multicast_ptr, nbytes)."""
    if _native_symmetric():
        local, mc, _, _, _, _, _ = native().alloc_symmetric("grads", total_elems * 2, role)
        flat = local.view(torch.bfloat16)[:total_elems]  # zero-filled by the allocator
        return flat, local, int(mc), total_elems * 2
    import torch.distributed._symmetric_memory as symm_mem

    flat = symm_mem.empty(total_elems, dtype=torch.bfloat16, device=device)
    flat.zero_()
    hdl = symm_mem.rendezvous(flat, group)
    torch.cuda.synchronize(device)
    mc = int(hdl.multicast_ptr) if getattr(hdl, "multicast_ptr", 0) else 0
    return flat, hdl, mc, total_elems * 2


def _flat(t: torch.Tensor) -> torch.Tensor:
    """The parameter (or gradient) as the 1-D buffer that travels: a view of its storage in STORAGE order.
    Contiguous tensors are the usual case; channels-last convolution weights are dense but permuted, and
    their storage order is as good a wire order as any — as long as gradient and parameter agree on it."""
    if t.is_contiguous():
        return t.view(-1)
    dense = (t.dim() == 4 and t.is_contiguous(memory_format=torch.channels_last)) or \
            (t.dim() == 5 and t.is_contiguous(memory_format=torch.channels_last_3d))
    assert dense, "PS parameters must be dense (contiguous or channels-last)"
    return t.as_strided((t.numel(),), (1,), t.storage_offset())


class PSWorkerOptimizer:
    """Drop-in "optimizer" for a worker: hooks gradients, exposes step()/zero_grad()."""

    def __init__(self, params, kv, num_servers: int, num_workers: int, worker_rank: int,
                 grad_wire: str = "fp8", chunk_elems: int = 32 << 20, app_barrier=None,
                 symmetric: bool = False, grad_buffer: torch.Tensor | None = None,
                 fused_pushpull: bool = False, no_decay_1d: bool = True, row_sparse=()):
        C = native()
        self._C = C
        self.kv = kv
        self.S = num_servers
        self.W = num_workers
        self.rank = worker_rank
        self.params = [p for p in params if p.requires_grad]
        assert chunk_elems % 1024 == 0
        self.chunk_elems = chunk_elems
        self.grad_wire = grad_wire
        self.stats = PSTrainerStats()
        self._pending: list[int] = []
        self._pending_by_param: dict[int, list[int]] = {}
        self._lazy = False
        self._hooks = []
        self._barrier = app_barrier
        self.accumulate = False  # True on non-final micro-batches: keep grads local
        # byte offset of every parameter in the symmetric buffer (see setup_symmetric_params)
        self.symm_off = [o * 2 for o in symmetric_layout(self.params)[0]] if symmetric else None
        # NVLS aggregation: gradients are staged (bf16) in this symmetric buffer and the server
        # reads the sum over all workers with multimem.ld_reduce (see setup_symmetric_grads)
        # one request + one reply per chunk (KVWorker::ZPushPull) instead of push, ack, pull, reply
        self.fused_pushpull = fused_pushpull
        # the usual rule: norm gains / biases (1-D tensors) are not weight-decayed; the server
        # learns it per shard from the option bits of the initial push
        self.no_decay_1d = no_decay_1d
        assert not (fused_pushpull and grad_buffer is not None), "push-pull stages no symmetric gradients"
        self.grad_buffer = grad_buffer
        # 2-D parameters whose gradients arrive as sparse COO tensors (nn.Embedding(sparse=True))
        self.row_sparse = {id(p) for p in row_sparse}
        assert not (self.row_sparse and grad_buffer is not None), "row-sparse gradients are not reduced in the switch"
        self._staging: dict[int, torch.Tensor] = {}  # key -> worst-case row push of that chunk
        if grad_buffer is not None:
            assert symmetric, "in-switch reduction uses the symmetric parameter layout"
            assert grad_buffer.dtype == torch.bfloat16 and grad_buffer.is_contiguous()
        # chunk table
        self.chunks: list[list[_Chunk]] = []
        j = 0
        for i, p in enumerate(self.params):
            _flat(p.data)  # (asserts that the parameter is dense)
            per = []
            n = p.numel()
            dim = 0
            step = chunk_elems
            if id(p) in self.row_sparse:
                assert p.dim() == 2, "row_sparse parameters are 2-D tables"
                dim = p.shape[1]
                step = max(1, chunk_elems // dim) * dim  # whole rows per key
            for a in range(0, n, step):
                b = min(n, a + step)
                server = j % self.S
                per.append(_Chunk(kv.server_key(server, j), i, a, b, server, dim))
                j += 1
            self.chunks.append(per)
        assert len(self.row_sparse) == sum(1 for per in self.chunks if per and per[0].dim), \
            "every row_sparse parameter must be one of the trained parameters"
        self.stats.keys = j

    # -- wire format -------------------------------------------------------------
    def _codec(self, t: torch.Tensor) -> int:
        C = self._C
        if self.grad_buffer is not None:  # the switch adds bf16 values
            return C.CODEC_F32_TO_BF16 if t.dtype == torch.float32 else C.CODEC_RAW
        if self.grad_wire == "fp8":
            return C.CODEC_F32_TO_FP8BLOCK if t.dtype == torch.float32 else C.CODEC_BF16_TO_FP8BLOCK
        if t.dtype == torch.float32:
            return C.CODEC_F32_TO_BF16
        return C.CODEC_RAW  # bf16 gradients travel as they are

    # -- one-time parameter initialisation ----------------------------------------
    def init_parameters(self, barrier=None):
        """Worker 0 seeds the servers with the initial values; everyone then pulls them."""
        C = self._C
        if self.rank == 0:
            ts = []
            for p, per in zip(self.params, self.chunks):
                flat = _flat(p.data)
                cmd = C.CMD_INIT_F32 if p.dtype == torch.float32 else C.CMD_INIT_BF16
                opt_bits = C.INIT_NO_WEIGHT_DECAY if (self.no_decay_1d and p.dim() <= 1) else 0
                for c in per:
                    bits = opt_bits | (C.INIT_ROW_SPARSE | (c.dim << 8) if c.dim else 0)
                    ts.append(self.kv.push(c.key, flat[c.start:c.stop], cmd=cmd, option=bits))
            for t in ts:
                self.kv.wait(t)
        (barrier or self._barrier or (lambda: None))()
        ts = []
        for p, per in zip(self.params, self.chunks):
            assert p.dtype == torch.bfloat16, "servers emit bf16 parameters"
            flat = _flat(p.data)
            for c in per:
                ts.append(self.kv.pull(c.key, flat[c.start:c.stop], symm_offset=self._symm(c)))
        for t in ts:
            self.kv.wait(t)

    def _symm(self, c: _Chunk) -> int:
        return -1 if self.symm_off is None else self.symm_off[c.param_index] + c.start * 2

    # -- gradient hooks ---------------------------------------------------------------
    def attach(self):
        for i, p in enumerate(self.params):
            self._hooks.append(p.register_post_accumulate_grad_hook(self._make_hook(i)))
        return self

    def detach(self):
        for h in self._hooks:
            h.remove()
        self._hooks.clear()

    def _make_hook(self, i: int):
        def hook(p: torch.Tensor):
            if self.accumulate:
                return
            g = p.grad
            p.grad = None  # the transport keeps the tensor alive until the push completes
            self._push_pull(i, g)
        return hook

    def enable_lazy_wait(self, model: torch.nn.Module):
        """Hide the tail of a step: `step()` stops waiting and every module instead waits, right
        before its forward, for the chunks of *its own* parameters. The pulls of late layers then
        overlap the next forward of the early ones (gradients are pushed last-layer-first, so the
        first layers' parameters — needed first — are also the last to come back). Call
        `wait_all()` before reading parameters outside a forward pass (evaluation, checksums)."""
        index = {id(p): i for i, p in enumerate(self.params)}
        for module in model.modules():
            mine = [index[id(p)] for p in module.parameters(recurse=False) if id(p) in index]
            if mine:
                self._hooks.append(module.register_forward_pre_hook(
                    lambda _m, _inp, mine=tuple(mine): self._wait_params(mine)))
        self._lazy = True
        return self

    def _wait_params(self, indices):
        for i in indices:
            pend = self._pending_by_param.pop(i, None)
            if pend:
                for ts in pend:
                    self.kv.wait(ts)

    def wait_all(self):
        """Block until nothing is in flight (also what a non-lazy step() does)."""
        self._wait_params(list(self._pending_by_param.keys()))
        pend, self._pending = self._pending, []
        for ts in pend:
            self.kv.wait(ts)

    def _push_pull(self, i: int, g: torch.Tensor):
        if self._lazy:
            mark = len(self._pending)
            self._push_pull_now(i, g)
            self._pending_by_param.setdefault(i, []).extend(self._pending[mark:])
            del self._pending[mark:]
            return
        self._push_pull_now(i, g)

    def _row_format(self, dim: int) -> int:
        C = self._C
        return C.GRAD_FP8BLOCK if self.grad_wire == "fp8" and dim % 32 == 0 else C.GRAD_BF16

    def _push_rows(self, i: int, g: torch.Tensor):
        """push the touched rows of every chunk of a row-sparse parameter, then pull the chunk"""
        C = self._C
        p = self.params[i].data
        if not g.is_sparse:
            raise ValueError(f"parameter {i} is row_sparse but its gradient is dense: build it with "
                             "nn.Embedding(sparse=True) or leave it out of row_sparse")
        g = g.float().coalesce()  # (repeated tokens of a batch are summed in fp32, not in the gradient's bf16)
        ids = g.indices()[0]
        vals = g.values()
        per = self.chunks[i]
        dim = per[0].dim
        fmt = self._row_format(dim)
        bounds = torch.tensor([c.start // dim for c in per] + [per[-1].stop // dim], device=ids.device)
        cuts = torch.searchsorted(ids, bounds).tolist()  # (the row counts travel in the request)
        pflat = _flat(p)
        for k, c in enumerate(per):
            lo, hi = cuts[k], cuts[k + 1]
            r = hi - lo
            rows = (c.stop - c.start) // dim
            stage = self._staging.get(c.key)
            if stage is None:
                stage = torch.zeros(C.rows_slot_bytes(rows, dim, fmt), dtype=torch.uint8, device=p.device)
                self._staging[c.key] = stage
            nbytes = C.rows_slot_bytes(r, dim, fmt)
            if r:
                ids_w = (r + 3) // 4 * 4
                stage[:4 * r].view(torch.int32).copy_(ids[lo:hi] - c.start // dim)
                stage[4 * r:4 * ids_w].zero_()
                body = stage[4 * ids_w:nbytes]
                v = vals[lo:hi].reshape(-1)
                if fmt == C.GRAD_FP8BLOCK:
                    C.copy_codec(body, v.contiguous(), C.CODEC_F32_TO_FP8BLOCK, 1.0)
                else:
                    body.view(torch.bfloat16).copy_(v)
                payload = stage[:nbytes]
            else:
                payload = stage[:16].zero_()  # a worker whose batch touched no row of this chunk still takes part
            self._pending.append(self.kv.push(c.key, payload, cmd=C.CMD_GRAD_ROWS, codec=C.CODEC_RAW,
                                              option=(r << 2) | fmt, slot_bytes=stage.numel()))
            self._pending.append(self.kv.pull(c.key, pflat[c.start:c.stop], symm_offset=self._symm(c)))
            self.stats.pushes += 1
            self.stats.pulls += 1
            self.stats.push_bytes_wire += payload.numel()
            self.stats.pull_bytes += (c.stop - c.start) * 2

    def _push_pull_now(self, i: int, g: torch.Tensor):
        if self.chunks[i] and self.chunks[i][0].dim:
            self._push_rows(i, g)
            return
        p = self.params[i].data
        if p.is_contiguous():
            if not g.is_contiguous():
                g = g.contiguous()
        elif g.stride() != p.stride():
            g = torch.empty_like(p, dtype=g.dtype).copy_(g)  # the parameter's (dense, permuted) layout
        gflat = _flat(g)
        pflat = _flat(p)
        codec = self._codec(g)
        for c in self.chunks[i]:
            gs = gflat[c.start:c.stop]
            if self.fused_pushpull:
                self._pending.append(self.kv.push_pull(c.key, gs, pflat[c.start:c.stop], cmd=self._C.CMD_GRAD,
                                                       codec=codec, scale=1.0, pull_symm_offset=self._symm(c)))
                self.stats.pushes += 1
                self.stats.pulls += 1
                self.stats.push_bytes_wire += self._C.wire_bytes(codec, gs.numel() * gs.element_size())
                self.stats.pull_bytes += (c.stop - c.start) * 2
                continue
            if self.grad_buffer is not None:
                self._pending.append(self.kv.push(c.key, gs, cmd=self._C.CMD_GRAD, codec=codec, scale=1.0,
                                                  symm_offset=self._symm(c),
                                                  symm_base=self.grad_buffer.data_ptr()))
            else:
                self._pending.append(self.kv.push(c.key, gs, cmd=self._C.CMD_GRAD, codec=codec, scale=1.0))
            self._pending.append(self.kv.pull(c.key, pflat[c.start:c.stop], symm_offset=self._symm(c)))
            self.stats.pushes += 1
            self.stats.pulls += 1
            self.stats.push_bytes_wire += self._C.wire_bytes(codec, gs.numel() * gs.element_size())
            self.stats.pull_bytes += (c.stop - c.start) * 2

    # -- optimizer-like surface ---------------------------------------------------------
    def step(self):
        """Block until every parameter chunk of this round has been rewritten by its server
        (with enable_lazy_wait(): return at once, the modules wait for their own parameters)."""
        if self._lazy:
            return
        pend, self._pending = self._pending, []
        for ts in pend:
            self.kv.wait(ts)

    def set_lr(self, lr: float):
        """Learning-rate schedules: tell every server its new rate (they may live in other processes).
        Every worker may call it with the same value; only worker 0 sends. Takes effect with the next
        update a server runs, so call it between `step()` and the next backward."""
        if self.rank != 0:
            return
        value = torch.tensor([lr], dtype=torch.float32)
        seen = set()
        ts = []
        for per in self.chunks:
            for c in per:
                if c.server not in seen:
                    seen.add(c.server)
                    ts.append(self.kv.push(c.key, value, cmd=self._C.CMD_SET_LR))
        for t in ts:
            self.kv.wait(t)

    def zero_grad(self, set_to_none: bool = True):
        for p in self.params:
            p.grad = None
