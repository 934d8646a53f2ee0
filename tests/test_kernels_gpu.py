"""Numerics of the sm_100a kernels against plain PyTorch fp32 references (B200 only)."""
import pytest
import torch

pytestmark = pytest.mark.gpu


def _require_cuda():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


def ref_fp8_block(x: torch.Tensor):
    """fp32 reference of the block-scaled e4m3 wire format: per-32 power-of-two scale."""
    n = x.numel()
    pad = (32 - n % 32) % 32
    xp = torch.cat([x.float(), x.new_zeros(pad, dtype=torch.float32)]).view(-1, 32)
    amax = xp.abs().amax(dim=1)
    e = torch.ceil(torch.log2(amax.clamp_min(1e-38) / 448.0)).clamp(-126, 127)  # 2^-126: smallest decodable scale
    e = torch.where(amax > 0, e, torch.full_like(e, -127.0))
    scale = torch.exp2(e)
    q = (xp / scale[:, None]).to(torch.float8_e4m3fn).float() * scale[:, None]
    return q.view(-1)[:n]


@pytest.mark.parametrize("n", [1, 31, 4096, 100003, 1 << 20])
def test_raw_copy(native, n):
    _require_cuda()
    src = torch.randint(0, 255, (n,), dtype=torch.uint8, device="cuda")
    dst = torch.zeros_like(src)
    native.copy_codec(dst, src, native.CODEC_RAW, 1.0)
    torch.cuda.synchronize()
    assert torch.equal(dst, src)


def test_multi_segment_copy(native):
    """one launch, many unrelated buffers (launch coalescing), incl. unaligned and tiny ones"""
    _require_cuda()
    sizes = [1, 15, 16, 4097, 65536, 1 << 20, 3 * (1 << 20) + 5] * 7  # 49 segments: two launches
    srcs = [torch.randint(0, 255, (n,), dtype=torch.uint8, device="cuda") for n in sizes]
    srcs[3] = torch.randint(0, 255, (4098,), dtype=torch.uint8, device="cuda")[1:]  # misaligned source
    dsts = [torch.zeros(s.numel(), dtype=torch.uint8, device="cuda") for s in srcs]
    native.copy_multi(dsts, srcs)
    torch.cuda.synchronize()
    for d, s in zip(dsts, srcs):
        assert torch.equal(d, s)


@pytest.mark.parametrize("codec_name,n", [("raw", 1), ("raw", 4096000), ("raw", 100003), ("bf16", 100003),
                                          ("fp8", 1 << 20), ("fp8", 40)])
def test_copy_with_in_kernel_completion_signal(native, codec_name, n):
    """the copy kernels finish with st.release.sys on a flag word (the descriptor gate of the nvl van):
    a host thread that only POLLS the flag — no event, no synchronize — must then find every byte"""
    _require_cuda()
    x = torch.randn(n, device="cuda")
    if codec_name == "raw":
        src = x.view(torch.uint8)
        codec, out_bytes = native.CODEC_RAW, src.numel()
    elif codec_name == "bf16":
        src = x.view(torch.uint8)
        codec, out_bytes = native.CODEC_F32_TO_BF16, 2 * n
    else:
        src = x.view(torch.uint8)
        codec, out_bytes = native.CODEC_F32_TO_FP8BLOCK, native.wire_bytes(native.CODEC_F32_TO_FP8BLOCK, 4 * n)
    ref = torch.zeros(out_bytes, dtype=torch.uint8, device="cuda")
    native.copy_codec(ref, src, codec, 0.5)
    torch.cuda.synchronize()
    flag = torch.zeros(1, dtype=torch.int64).pin_memory()
    counter = torch.zeros(64, dtype=torch.int32, device="cuda")
    side = torch.cuda.Stream()
    for value in (1, 2, 7):  # the arrival counter resets itself: the same word serves every launch
        dst = torch.zeros(out_bytes, dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()
        native.copy_signal(dst, src, codec, 0.5, 0, flag, value, counter)
        import time

        t0 = time.time()
        while int(flag[0]) != value:
            assert time.time() - t0 < 20, "the kernel never signalled"
        with torch.cuda.stream(side):  # an unrelated stream: ordering comes from the flag alone
            got = dst.to("cpu", non_blocking=False)
        assert torch.equal(got, ref.cpu()), f"bytes missing after the signal (value {value})"
    torch.cuda.synchronize()
    assert int(counter[0]) == 0


@pytest.mark.parametrize("n", [8, 1000, 100003])
def test_f32_to_bf16_scaled(native, n):
    _require_cuda()
    x = torch.randn(n, device="cuda")
    out = torch.empty(n, dtype=torch.bfloat16, device="cuda")
    native.copy_codec(out.view(torch.uint8), x.view(torch.uint8), native.CODEC_F32_TO_BF16, 0.25)
    torch.cuda.synchronize()
    ref = (x * 0.25).to(torch.bfloat16)
    assert torch.equal(out, ref)


@pytest.mark.parametrize("src_dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("n", [32, 4096, 100003])
def test_fp8_block_quant_roundtrip(native, src_dtype, n):
    _require_cuda()
    x = (torch.randn(n, device="cuda") * torch.logspace(-3, 2, n, device="cuda")).to(src_dtype)
    codec = native.CODEC_F32_TO_FP8BLOCK if src_dtype == torch.float32 else native.CODEC_BF16_TO_FP8BLOCK
    wire = torch.zeros(native.wire_bytes(codec, x.numel() * x.element_size()), dtype=torch.uint8, device="cuda")
    native.copy_codec(wire, x.view(torch.uint8), codec, 1.0)
    dec = torch.empty(n, dtype=torch.float32, device="cuda")
    native.decode(dec, wire, n, native.GRAD_FP8BLOCK)
    torch.cuda.synchronize()
    ref = ref_fp8_block(x.float())
    # identical scale choice and RN rounding -> bit-identical to the fp32 reference
    assert torch.allclose(dec, ref, rtol=0, atol=0), (dec - ref).abs().max()


@pytest.mark.parametrize("fmt", ["bf16", "fp8", "f32"])
@pytest.mark.parametrize("W,fan", [(1, 1), (2, 3), (4, 5)])
def test_fused_adamw_update(native, fmt, W, fan):
    _require_cuda()
    n = 50003
    torch.manual_seed(0)
    p = torch.randn(n, device="cuda")
    m = torch.randn(n, device="cuda") * 0.1
    v = torch.rand(n, device="cuda") * 0.01
    grads_f32 = [torch.randn(n, device="cuda") * 0.05 for _ in range(W)]
    if fmt == "bf16":
        wires = [g.to(torch.bfloat16) for g in grads_f32]
        dec = [w.float() for w in wires]
        gfmt = native.GRAD_BF16
    elif fmt == "f32":
        wires = grads_f32
        dec = grads_f32
        gfmt = native.GRAD_F32
    else:
        wires, dec = [], []
        for g in grads_f32:
            w = torch.zeros(native.wire_bytes(native.CODEC_F32_TO_FP8BLOCK, n * 4), dtype=torch.uint8, device="cuda")
            native.copy_codec(w, g.view(torch.uint8), native.CODEC_F32_TO_FP8BLOCK, 1.0)
            wires.append(w)
            dec.append(ref_fp8_block(g))
        gfmt = native.GRAD_FP8BLOCK
    lr, b1, b2, eps, wd, step, gs = 1e-2, 0.9, 0.95, 1e-8, 0.1, 3, 1.0 / W
    # fp32 PyTorch reference
    g = sum(dec) * gs
    m_ref = b1 * m + (1 - b1) * g
    v_ref = b2 * v + (1 - b2) * g * g
    mhat = m_ref / (1 - b1 ** step)
    vhat = v_ref / (1 - b2 ** step)
    p_ref = p - lr * (mhat / (vhat.sqrt() + eps) + wd * p)
    pk, mk, vk = p.clone(), m.clone(), v.clone()
    outs = [torch.empty(n, dtype=torch.bfloat16, device="cuda") for _ in range(fan)]
    native.fused_update(wires, gfmt, pk, mk, vk, outs, "adamw", lr, b1, b2, eps, wd, step, gs, 0)
    torch.cuda.synchronize()
    assert torch.allclose(mk, m_ref, rtol=1e-5, atol=1e-7)
    assert torch.allclose(vk, v_ref, rtol=1e-5, atol=1e-9)
    assert torch.allclose(pk, p_ref, rtol=1e-5, atol=1e-6)
    for o in outs:
        assert torch.equal(o, pk.to(torch.bfloat16))


@pytest.mark.parametrize("n", [1, 5, 7, 9, 33, 257])
@pytest.mark.parametrize("fmt", ["bf16", "fp8", "f32"])
def test_update_of_tiny_and_ragged_shards(native, n, fmt):
    """same cases as tests/test_kernels_host.py: shards shorter than one group / one fp8 block"""
    _require_cuda()
    torch.manual_seed(n)
    p = torch.randn(n, device="cuda")
    m, v = torch.zeros(n, device="cuda"), torch.zeros(n, device="cuda")
    g32 = torch.randn(n, device="cuda") * 0.1
    if fmt == "bf16":
        wire, dec, gfmt = g32.to(torch.bfloat16), g32.to(torch.bfloat16).float(), native.GRAD_BF16
    elif fmt == "f32":
        wire, dec, gfmt = g32, g32, native.GRAD_F32
    else:
        wire = torch.zeros(native.wire_bytes(native.CODEC_F32_TO_FP8BLOCK, n * 4), dtype=torch.uint8, device="cuda")
        native.copy_codec(wire, g32.view(torch.uint8), native.CODEC_F32_TO_FP8BLOCK, 1.0)
        dec, gfmt = ref_fp8_block(g32), native.GRAD_FP8BLOCK
    out = torch.empty(n, dtype=torch.bfloat16, device="cuda")
    pk = p.clone()
    native.fused_update([wire], gfmt, pk, m, v, [out], "sgd", 0.5, 0.0, 0.0, 0.0, 0.0, 1, 1.0, 0)
    torch.cuda.synchronize()
    assert torch.allclose(pk, p - 0.5 * dec, rtol=1e-6, atol=1e-7)
    assert torch.equal(out, pk.to(torch.bfloat16))


def test_fused_sgd_update(native):
    _require_cuda()
    n = 4099
    p = torch.randn(n, device="cuda")
    m = torch.zeros(n, device="cuda")
    v = torch.zeros(n, device="cuda")
    g = torch.randn(n, device="cuda").to(torch.bfloat16)
    out = torch.empty(n, dtype=torch.bfloat16, device="cuda")
    pk = p.clone()
    native.fused_update([g], native.GRAD_BF16, pk, m, v, [out], "sgd", 0.1, 0.9, 0.0, 0.0, 0.0, 1, 1.0, 0)
    torch.cuda.synchronize()
    ref = p - 0.1 * g.float()
    assert torch.allclose(pk, ref, rtol=1e-6, atol=1e-6)


def test_fused_rope_split_matches_reference(native):
    _require_cuda()
    from pslite_b200.models.llama import precompute_rope
    from pslite_b200.ops.fused import rope_split, rope_split_reference

    B, S, H, KV, D = 2, 48, 8, 2, 64
    cos, sin = precompute_rope(D, 64, 500000.0, "cuda")
    qkv = torch.randn(B, S, (H + 2 * KV) * D, device="cuda", dtype=torch.bfloat16, requires_grad=True)
    qkv_ref = qkv.detach().clone().requires_grad_(True)
    q, k, v = rope_split(qkv, cos, sin, H, KV, D)
    qr, kr, vr = rope_split_reference(qkv_ref, cos, sin, H, KV, D)
    assert torch.allclose(q.float(), qr.float(), atol=2e-2, rtol=2e-2)
    assert torch.allclose(k.float(), kr.float(), atol=2e-2, rtol=2e-2)
    assert torch.equal(v, vr)
    gq, gk, gv = torch.randn_like(q), torch.randn_like(k), torch.randn_like(v)
    (q * gq).sum().add((k * gk).sum()).add((v * gv).sum()).backward()
    (qr * gq).sum().add((kr * gk).sum()).add((vr * gv).sum()).backward()
    assert torch.allclose(qkv.grad.float(), qkv_ref.grad.float(), atol=3e-2, rtol=3e-2)


def test_fused_swiglu_matches_reference(native):
    _require_cuda()
    from pslite_b200.ops.fused import swiglu, swiglu_reference

    gu = (torch.randn(3, 40, 2 * 256, device="cuda") * 2).to(torch.bfloat16).requires_grad_(True)
    gu_ref = gu.detach().clone().float().requires_grad_(True)
    out = swiglu(gu)
    g, u = gu_ref.chunk(2, dim=-1)
    ref = torch.nn.functional.silu(g) * u
    assert torch.allclose(out.float(), ref, atol=2e-2, rtol=2e-2)
    assert torch.allclose(out.float(), swiglu_reference(gu.detach()).float(), atol=2e-2, rtol=2e-2)
    d = torch.randn_like(out)
    out.backward(d)
    ref.backward(d.float())
    assert torch.allclose(gu.grad.float(), gu_ref.grad, atol=3e-2, rtol=3e-2)


def test_copy_engine_selfcheck_and_message_rate():
    """apps/engine_bench on one GPU: descriptors posted to the copy engine (persistent kernel, TMA workers)
    against one launch per copy; every configuration verifies the bytes it moved. The engine must move a
    small message in a fraction of what a launch costs, and 16 MB copies at HBM-class bandwidth."""
    import json
    import os
    import subprocess

    _require_cuda()
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = os.path.join(root, "build", "engine_bench")
    if not os.path.exists(exe):
        pytest.skip("build/engine_bench not built (make)")
    r = subprocess.run([exe], capture_output=True, text=True, timeout=240, cwd=root)
    assert r.returncode == 0, (r.stdout + r.stderr)[-3000:]
    rows = [json.loads(l) for l in r.stdout.splitlines() if l.startswith("{")]
    summary = rows[-1]
    assert summary["data_failures"] == 0 and summary["engine_items"] > 0 and summary["engine_launches"] >= 1
    eng = {d["bytes"]: d for d in rows if d.get("path") == "engine" and "bytes" in d}
    lau = {d["bytes"]: d for d in rows if d.get("path") == "launch" and "bytes" in d}
    assert eng[1024]["us_per_msg"] < 0.6 * lau[1024]["us_per_msg"], (eng[1024], lau[1024])
    assert eng[16 << 20]["GBps"] > 1000, eng[16 << 20]
    print({b: (eng[b]["us_per_msg"], eng[b]["GBps"]) for b in sorted(eng)})
