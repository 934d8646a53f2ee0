"""Row-sparse gradient slots and an independent fp64 reference of the row-sparse update.

A slot is what a worker pushes with kCmdGradRows (see ps_update_rows_args):
    [u32 ids, R entries, zero-padded to a multiple of 4][values]
    values: f32 R*D | bf16 R*D | fp8 block [R*D e4m3][R*D/32 e8m0]
`make_slot` builds one (the fp8 values through the project's codec) and also returns the values the
server reads from it, decoded here by torch's own float8_e4m3fn, not by the project's decoder.
`reference_round` applies one round in float64 with the documented lazy semantics.
"""
import torch

GRAD_F32, GRAD_BF16, GRAD_FP8BLOCK = 0, 1, 2
CODEC_F32_TO_FP8BLOCK = 3


def slot_bytes(r, d, fmt):
    ids = (r + 3) // 4 * 16
    e = r * d
    return ids + {GRAD_F32: 4 * e, GRAD_BF16: 2 * e, GRAD_FP8BLOCK: e + e // 32}[fmt]


def decode_fp8_block(payload, scales, n):
    """e4m3 bytes * 2^(scale byte - 127), byte clamped to [1, 254] as every decoder does"""
    q = payload[:n].view(torch.float8_e4m3fn).to(torch.float64)
    e = scales.to(torch.int64).clamp(1, 254) - 127
    return q * torch.pow(2.0, e.to(torch.float64)).repeat_interleave(32)[:n]


def make_slot(C, ids, vals, fmt, pad=0):
    """ids: int64 [R] (written as u32), vals: float32 [R, D] -> (uint8 slot, float64 [R, D] as read)"""
    dev = vals.device
    r, d = vals.shape
    out = torch.zeros(slot_bytes(r, d, fmt) + pad, dtype=torch.uint8, device=dev)
    idw = (r + 3) // 4 * 4
    if r:
        out[:4 * r].view(torch.int32).copy_(ids.to(torch.int64).to(torch.int32))
    body = out[4 * idw:4 * idw + slot_bytes(r, d, fmt) - 4 * idw]
    if fmt == GRAD_F32:
        body.view(torch.float32).copy_(vals.reshape(-1))
        read = vals.to(torch.float64)
    elif fmt == GRAD_BF16:
        b = vals.to(torch.bfloat16)
        body.view(torch.bfloat16).copy_(b.reshape(-1))
        read = b.to(torch.float64)
    else:
        n = r * d
        if n:
            C.copy_codec(body, vals.contiguous().reshape(-1), CODEC_F32_TO_FP8BLOCK, 1.0)
        read = decode_fp8_block(body[:n], body[n:n + n // 32], n).reshape(r, d)
    return out, read


def reference_round(state, slots, opt, step, dim):
    """state: dict of float64 master/m/v [rows, D]; slots: list of (ids int64, values float64 [R, D]).
    Returns the union (sorted row ids) and the number of ids the server must skip."""
    rows = state["master"].shape[0]
    g = {}
    bad = 0
    for ids, vals in slots:
        seen = set()
        for i, rid in enumerate(ids.tolist()):
            if rid >= rows or rid in seen:
                bad += 1
                continue
            seen.add(rid)
            g[rid] = vals[i] if rid not in g else g[rid] + vals[i]
    union = sorted(g)
    if not union:
        return union, bad
    idx = torch.tensor(union, dtype=torch.int64, device=state["master"].device)
    G = torch.stack([g[r] for r in union]).to(state["master"].device) * opt["grad_scale"]
    p, m = state["master"][idx], state["m"][idx]
    lr, b1, b2, eps, wd = opt["lr"], opt["beta1"], opt["beta2"], opt["eps"], opt["weight_decay"]
    if opt["optimizer"] == "adamw":
        v = state["v"][idx]
        m = b1 * m + (1 - b1) * G
        v = b2 * v + (1 - b2) * G * G
        bc1, bc2 = 1 - b1 ** step, 1 - b2 ** step
        p = p - lr * ((m / bc1) / (torch.sqrt(v / bc2) + eps) + wd * p)
        state["v"][idx] = v
    else:
        G = G + wd * p
        m = b1 * m + G
        p = p - lr * m
    state["master"][idx] = p
    state["m"][idx] = m
    return union, bad
