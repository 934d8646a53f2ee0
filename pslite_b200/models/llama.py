"""Llama-3 decoder (the worker-side model of the PS training benchmark).

The reference library contains no model code (SURVEY §0); BASELINE.json names
"Llama-3-8B bf16 PS training" as a target config, so the architecture is defined
here: RMSNorm -> GQA attention with RoPE -> SwiGLU MLP, untied embedding / LM head,
vocab 128256, 32 layers, d_model 4096, 32 heads / 8 KV heads, d_ff 14336, theta 5e5.
GEMMs go through cuBLAS (plain library GEMMs), attention through PyTorch SDPA; the
parameter-server data path (push / fused update / pull) is this repo's own kernels.
Activation checkpointing is per layer and partial (`ckpt_layers`) so a single 180 GB
B200 can host the worker *and* its server shard at sequence length 8192.
"""
from __future__ import annotations

import math
from dataclasses import dataclass

import torch
import torch.nn as nn
import torch.nn.functional as F
from torch.utils.checkpoint import checkpoint


@dataclass
class LlamaConfig:
    vocab_size: int = 128256
    dim: int = 4096
    n_layers: int = 32
    n_heads: int = 32
    n_kv_heads: int = 8
    ffn_dim: int = 14336
    rope_theta: float = 500000.0
    norm_eps: float = 1e-5
    max_seq_len: int = 8192
    ckpt_layers: int = 32          # how many (leading) layers recompute in backward
    loss_chunk: int = 2048         # tokens per LM-head / cross-entropy chunk
    attn_backend: str = "auto"     # auto | cudnn | flash | efficient | math (PyTorch SDPA backends)
    fused_ops: bool = True         # own RoPE-split / SwiGLU kernels on CUDA (pslite_b200.ops.fused)
    sparse_embedding: bool = False # input embedding with sparse (row) gradients: nn.Embedding(sparse=True)

    @staticmethod
    def llama3_8b(**kw) -> "LlamaConfig":
        return LlamaConfig(**kw)

    @staticmethod
    def tiny(**kw) -> "LlamaConfig":
        base = dict(vocab_size=512, dim=128, n_layers=2, n_heads=4, n_kv_heads=2, ffn_dim=256,
                    max_seq_len=128, ckpt_layers=0, loss_chunk=64)
        base.update(kw)
        return LlamaConfig(**base)

    def num_params(self) -> int:
        hd = self.dim // self.n_heads
        attn = self.dim * self.dim * 2 + 2 * self.dim * hd * self.n_kv_heads
        mlp = 3 * self.dim * self.ffn_dim
        return self.n_layers * (attn + mlp + 2 * self.dim) + 2 * self.vocab_size * self.dim + self.dim

    def flops_per_token(self, seq_len: int) -> float:
        """fwd+bwd matmul FLOPs per token (6 x params in GEMMs + attention), no recompute."""
        hd = self.dim // self.n_heads
        dense = self.n_layers * (self.dim * self.dim * 2 + 2 * self.dim * hd * self.n_kv_heads +
                                 3 * self.dim * self.ffn_dim) + self.vocab_size * self.dim
        attn = self.n_layers * 2 * seq_len * self.dim / 2  # causal: half of QK^T and PV
        return 6.0 * dense + 6.0 * attn


def precompute_rope(head_dim: int, seq_len: int, theta: float, device, dtype=torch.float32):
    inv = 1.0 / (theta ** (torch.arange(0, head_dim, 2, device=device, dtype=torch.float32) / head_dim))
    t = torch.arange(seq_len, device=device, dtype=torch.float32)
    ang = torch.outer(t, inv)
    return torch.cos(ang).to(dtype), torch.sin(ang).to(dtype)


def apply_rope(x: torch.Tensor, cos: torch.Tensor, sin: torch.Tensor) -> torch.Tensor:
    """x: [B, S, H, D] (half-split rotation); cos/sin: [S, D/2]"""
    d2 = x.shape[-1] // 2
    x1, x2 = x[..., :d2], x[..., d2:]
    c = cos[None, :, None, :]
    s = sin[None, :, None, :]
    return torch.cat((x1 * c - x2 * s, x2 * c + x1 * s), dim=-1).to(x.dtype)


class RMSNorm(nn.Module):
    def __init__(self, dim: int, eps: float):
        super().__init__()
        self.eps = eps
        self.weight = nn.Parameter(torch.ones(dim))

    def forward(self, x):
        return F.rms_norm(x, (x.shape[-1],), self.weight, self.eps)


def _sdpa_context(backend: str):
    """Restrict PyTorch SDPA to one backend (cuDNN's fused attention is the tcgen05 path on
    Blackwell; the bundled flash kernels are the sm_80-era mma.sync ones)."""
    import contextlib

    if backend == "auto":
        return contextlib.nullcontext()
    from torch.nn.attention import SDPBackend, sdpa_kernel

    table = {"cudnn": SDPBackend.CUDNN_ATTENTION, "flash": SDPBackend.FLASH_ATTENTION,
             "efficient": SDPBackend.EFFICIENT_ATTENTION, "math": SDPBackend.MATH}
    return sdpa_kernel([table[backend]])


class Attention(nn.Module):
    def __init__(self, cfg: LlamaConfig):
        super().__init__()
        self.backend = cfg.attn_backend
        self.fused = cfg.fused_ops
        self.n_heads, self.n_kv = cfg.n_heads, cfg.n_kv_heads
        self.hd = cfg.dim // cfg.n_heads
        self.wqkv = nn.Linear(cfg.dim, (cfg.n_heads + 2 * cfg.n_kv_heads) * self.hd, bias=False)
        self.wo = nn.Linear(cfg.dim, cfg.dim, bias=False)

    def forward(self, x, cos, sin):
        B, S, _ = x.shape
        qkv = self.wqkv(x)
        if self.fused and qkv.is_cuda:
            from ..ops.fused import rope_split

            q, k, v = rope_split(qkv, cos, sin, self.n_heads, self.n_kv, self.hd)
            q, k, v = q.transpose(1, 2), k.transpose(1, 2), v.transpose(1, 2)
        else:
            q, k, v = qkv.split([self.n_heads * self.hd, self.n_kv * self.hd, self.n_kv * self.hd], dim=-1)
            q = apply_rope(q.view(B, S, self.n_heads, self.hd), cos, sin).transpose(1, 2)
            k = apply_rope(k.view(B, S, self.n_kv, self.hd), cos, sin).transpose(1, 2)
            v = v.view(B, S, self.n_kv, self.hd).transpose(1, 2)
        with _sdpa_context(self.backend):
            o = F.scaled_dot_product_attention(q, k, v, is_causal=True,
                                               enable_gqa=self.n_kv != self.n_heads)
        return self.wo(o.transpose(1, 2).reshape(B, S, -1))


class MLP(nn.Module):
    def __init__(self, cfg: LlamaConfig):
        super().__init__()
        self.w13 = nn.Linear(cfg.dim, 2 * cfg.ffn_dim, bias=False)  # gate and up fused
        self.w2 = nn.Linear(cfg.ffn_dim, cfg.dim, bias=False)
        self.fused = cfg.fused_ops

    def forward(self, x):
        gu = self.w13(x)
        if self.fused and gu.is_cuda:
            from ..ops.fused import swiglu

            return self.w2(swiglu(gu))
        g, u = gu.chunk(2, dim=-1)
        return self.w2(F.silu(g) * u)


class Block(nn.Module):
    def __init__(self, cfg: LlamaConfig):
        super().__init__()
        self.attn_norm = RMSNorm(cfg.dim, cfg.norm_eps)
        self.attn = Attention(cfg)
        self.mlp_norm = RMSNorm(cfg.dim, cfg.norm_eps)
        self.mlp = MLP(cfg)

    def forward(self, x, cos, sin):
        x = x + self.attn(self.attn_norm(x), cos, sin)
        return x + self.mlp(self.mlp_norm(x))


class Llama(nn.Module):
    def __init__(self, cfg: LlamaConfig):
        super().__init__()
        self.cfg = cfg
        self.embed = nn.Embedding(cfg.vocab_size, cfg.dim, sparse=cfg.sparse_embedding)
        self.layers = nn.ModuleList(Block(cfg) for _ in range(cfg.n_layers))
        self.norm = RMSNorm(cfg.dim, cfg.norm_eps)
        self.lm_head = nn.Linear(cfg.dim, cfg.vocab_size, bias=False)
        self._rope = None

    @torch.no_grad()
    def init_weights(self, std: float = 0.02, seed: int = 0):
        g = torch.Generator(device=self.embed.weight.device)
        g.manual_seed(seed)
        for name, p in self.named_parameters():
            if p.dim() == 1:
                p.fill_(1.0)
            else:
                scale = std / math.sqrt(2 * self.cfg.n_layers) if name.endswith(("wo.weight", "w2.weight")) else std
                p.normal_(0.0, scale, generator=g)

    def _rope_tables(self, S: int, device):
        if self._rope is None or self._rope[0].shape[0] < S or self._rope[0].device != device:
            hd = self.cfg.dim // self.cfg.n_heads
            self._rope = precompute_rope(hd, max(S, self.cfg.max_seq_len), self.cfg.rope_theta, device)
        return self._rope[0][:S], self._rope[1][:S]

    def hidden(self, tokens: torch.Tensor) -> torch.Tensor:
        B, S = tokens.shape
        cos, sin = self._rope_tables(S, tokens.device)
        x = self.embed(tokens)
        for i, layer in enumerate(self.layers):
            if self.training and i < self.cfg.ckpt_layers:
                x = checkpoint(layer, x, cos, sin, use_reentrant=False)
            else:
                x = layer(x, cos, sin)
        return self.norm(x)

    def forward(self, tokens: torch.Tensor, targets: torch.Tensor | None = None):
        h = self.hidden(tokens)
        if targets is None:
            return self.lm_head(h)
        # chunked LM head + cross entropy: never materialise [tokens, vocab] logits at once
        h2 = h.reshape(-1, h.shape[-1])
        t2 = targets.reshape(-1)
        n = h2.shape[0]
        total = h2.new_zeros((), dtype=torch.float32)
        step = self.cfg.loss_chunk
        for a in range(0, n, step):
            total = total + checkpoint(self._chunk_loss, h2[a:a + step], t2[a:a + step],
                                       use_reentrant=False)
        return total / n

    def _chunk_loss(self, h, t):
        return F.cross_entropy(self.lm_head(h).float(), t, reduction="sum")
