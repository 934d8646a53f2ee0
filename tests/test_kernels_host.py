"""Numerics of the CPU twins of the data-plane kernels (src/kernels/host_kernels.cc) against plain
PyTorch fp32 references — the same cases as tests/test_kernels_gpu.py, runnable without a GPU —
plus (GPU only) a bit-exactness check of the sm_100a kernels against these twins."""
import pytest
import torch

from test_kernels_gpu import ref_fp8_block


@pytest.mark.parametrize("n", [1, 31, 4096, 100003])
def test_host_raw_copy(native, n):
    src = torch.randint(0, 255, (n,), dtype=torch.uint8)
    dst = torch.zeros_like(src)
    native.copy_codec(dst, src, native.CODEC_RAW, 1.0)
    assert torch.equal(dst, src)


def test_host_multi_segment_copy(native):
    """copy_multi on CPU tensors (the GPU version is one launch for all segments)"""
    srcs = [torch.randint(0, 255, (n,), dtype=torch.uint8) for n in (1, 15, 16, 4097, 1 << 20, 3 * (1 << 20) + 5)]
    dsts = [torch.zeros_like(s) for s in srcs]
    native.copy_multi(dsts, srcs)
    assert all(torch.equal(d, s) for d, s in zip(dsts, srcs))


@pytest.mark.parametrize("n", [8, 1000, 100003, 600001])
def test_host_f32_to_bf16_scaled(native, n):
    x = torch.randn(n)
    out = torch.empty(n, dtype=torch.bfloat16)
    native.copy_codec(out.view(torch.uint8), x.view(torch.uint8), native.CODEC_F32_TO_BF16, 0.25)
    assert torch.equal(out, (x * 0.25).to(torch.bfloat16))
    y = torch.empty(n, dtype=torch.bfloat16)
    native.copy_codec(y.view(torch.uint8), out.view(torch.uint8), native.CODEC_BF16_SCALE, 0.5)
    assert torch.equal(y, (out.float() * 0.5).to(torch.bfloat16))


@pytest.mark.parametrize("src_dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("n", [32, 4096, 100003])
def test_host_fp8_block_quant_roundtrip(native, src_dtype, n):
    x = (torch.randn(n) * torch.logspace(-3, 2, n)).to(src_dtype)
    codec = native.CODEC_F32_TO_FP8BLOCK if src_dtype == torch.float32 else native.CODEC_BF16_TO_FP8BLOCK
    wire = torch.zeros(native.wire_bytes(codec, x.numel() * x.element_size()), dtype=torch.uint8)
    native.copy_codec(wire, x.view(torch.uint8), codec, 1.0)
    dec = torch.empty(n, dtype=torch.float32)
    native.decode(dec, wire, n, native.GRAD_FP8BLOCK)
    ref = ref_fp8_block(x.float())
    assert torch.equal(dec, ref), (dec - ref).abs().max()


def test_host_e4m3_encoding_is_exhaustively_right(native):
    """every e4m3 code point survives encode(decode(code)); ties and saturation follow RN-satfinite"""
    codes = torch.arange(256, dtype=torch.uint8)
    vals = codes.view(torch.float8_e4m3fn).float()
    finite = torch.isfinite(vals)
    x = vals[finite].repeat_interleave(1)
    n = x.numel()
    pad = (32 - n % 32) % 32
    # one block per value so that the shared scale is decided by that value alone
    blocks = torch.zeros(n, 32)
    blocks[:, 0] = x
    wire = torch.zeros(native.wire_bytes(native.CODEC_F32_TO_FP8BLOCK, blocks.numel() * 4), dtype=torch.uint8)
    native.copy_codec(wire, blocks.view(-1).view(torch.uint8), native.CODEC_F32_TO_FP8BLOCK, 1.0)
    dec = torch.empty(blocks.numel())
    native.decode(dec, wire, blocks.numel(), native.GRAD_FP8BLOCK)
    assert torch.equal(dec.view(n, 32)[:, 0], x)  # exactly representable after block scaling
    assert pad >= 0


@pytest.mark.parametrize("fmt", ["bf16", "fp8", "f32"])
@pytest.mark.parametrize("W,fan", [(1, 1), (2, 3), (4, 5)])
def test_host_fused_adamw_update(native, fmt, W, fan):
    n = 50003
    torch.manual_seed(0)
    p = torch.randn(n)
    m = torch.randn(n) * 0.1
    v = torch.rand(n) * 0.01
    grads_f32 = [torch.randn(n) * 0.05 for _ in range(W)]
    if fmt == "bf16":
        wires = [g.to(torch.bfloat16) for g in grads_f32]
        dec = [w.float() for w in wires]
        gfmt = native.GRAD_BF16
    elif fmt == "f32":
        wires, dec, gfmt = grads_f32, grads_f32, native.GRAD_F32
    else:
        wires, dec = [], []
        for g in grads_f32:
            w = torch.zeros(native.wire_bytes(native.CODEC_F32_TO_FP8BLOCK, n * 4), dtype=torch.uint8)
            native.copy_codec(w, g.view(torch.uint8), native.CODEC_F32_TO_FP8BLOCK, 1.0)
            wires.append(w)
            dec.append(ref_fp8_block(g))
        gfmt = native.GRAD_FP8BLOCK
    lr, b1, b2, eps, wd, step, gs = 1e-2, 0.9, 0.95, 1e-8, 0.1, 3, 1.0 / W
    g = sum(dec) * gs
    m_ref = b1 * m + (1 - b1) * g
    v_ref = b2 * v + (1 - b2) * g * g
    p_ref = p - lr * ((m_ref / (1 - b1 ** step)) / ((v_ref / (1 - b2 ** step)).sqrt() + eps) + wd * p)
    pk, mk, vk = p.clone(), m.clone(), v.clone()
    outs = [torch.empty(n, dtype=torch.bfloat16) for _ in range(fan)]
    native.fused_update(wires, gfmt, pk, mk, vk, outs, "adamw", lr, b1, b2, eps, wd, step, gs, 0)
    assert torch.allclose(mk, m_ref, rtol=1e-5, atol=1e-7)
    assert torch.allclose(vk, v_ref, rtol=1e-5, atol=1e-9)
    assert torch.allclose(pk, p_ref, rtol=1e-5, atol=1e-6)
    for o in outs:
        assert torch.equal(o, pk.to(torch.bfloat16))


@pytest.mark.parametrize("n", [1, 5, 7, 9, 33, 257])
@pytest.mark.parametrize("fmt", ["bf16", "fp8", "f32"])
def test_host_update_of_tiny_and_ragged_shards(native, n, fmt):
    """shards shorter than one 8-element group / one 32-element fp8 block, and ragged tails"""
    torch.manual_seed(n)
    p, m, v = torch.randn(n), torch.zeros(n), torch.zeros(n)
    g32 = torch.randn(n) * 0.1
    if fmt == "bf16":
        wire, dec, gfmt = g32.to(torch.bfloat16), g32.to(torch.bfloat16).float(), native.GRAD_BF16
    elif fmt == "f32":
        wire, dec, gfmt = g32, g32, native.GRAD_F32
    else:
        wire = torch.zeros(native.wire_bytes(native.CODEC_F32_TO_FP8BLOCK, n * 4), dtype=torch.uint8)
        native.copy_codec(wire, g32.view(torch.uint8), native.CODEC_F32_TO_FP8BLOCK, 1.0)
        dec, gfmt = ref_fp8_block(g32), native.GRAD_FP8BLOCK
    out = torch.empty(n, dtype=torch.bfloat16)
    pk = p.clone()
    native.fused_update([wire], gfmt, pk, m, v, [out], "sgd", 0.5, 0.0, 0.0, 0.0, 0.0, 1, 1.0, 0)
    assert torch.allclose(pk, p - 0.5 * dec, rtol=1e-6, atol=1e-7)
    assert torch.equal(out, pk.to(torch.bfloat16))


def test_host_fused_sgd_update(native):
    n = 4099
    p = torch.randn(n)
    m, v = torch.zeros(n), torch.zeros(n)
    g = torch.randn(n).to(torch.bfloat16)
    out = torch.empty(n, dtype=torch.bfloat16)
    pk = p.clone()
    native.fused_update([g], native.GRAD_BF16, pk, m, v, [out], "sgd", 0.1, 0.9, 0.0, 0.0, 0.0, 1, 1.0, 0)
    assert torch.allclose(pk, p - 0.1 * g.float(), rtol=1e-6, atol=1e-6)
    assert torch.equal(out, pk.to(torch.bfloat16))


@pytest.mark.gpu
@pytest.mark.parametrize("codec_name", ["CODEC_F32_TO_BF16", "CODEC_BF16_SCALE", "CODEC_F32_TO_FP8BLOCK",
                                        "CODEC_BF16_TO_FP8BLOCK"])
def test_gpu_wire_bytes_equal_host_wire_bytes(native, codec_name):
    """the sm_100a push kernels and their CPU twins produce the same bytes for the same input, also
    from and to views that are not 16-byte aligned (the bf16 codecs then run their scalar tail
    kernel; the fp8 codec refuses a misaligned source before launching anything)"""
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    codec = getattr(native, codec_name)
    n = 100003
    x = torch.randn(n) * torch.logspace(-3, 2, n)
    if codec_name.startswith("CODEC_BF16"):
        x = x.to(torch.bfloat16)
    nbytes = native.wire_bytes(codec, x.numel() * x.element_size())
    host = torch.zeros(nbytes, dtype=torch.uint8)
    native.copy_codec(host, x.view(torch.uint8), codec, 0.5)
    dev = torch.zeros(nbytes, dtype=torch.uint8, device="cuda")
    native.copy_codec(dev, x.cuda().view(torch.uint8), codec, 0.5)
    torch.cuda.synchronize()
    assert torch.equal(dev.cpu(), host)

    # the same input one element into a larger buffer: 4 (f32) or 2 (bf16) bytes off 16-byte alignment
    src_shifted = torch.zeros(n + 1, dtype=x.dtype, device="cuda")
    src_shifted[1:] = x.cuda()
    src_shifted = src_shifted[1:]
    if codec_name.endswith("FP8BLOCK"):
        with pytest.raises(RuntimeError, match="misaligned"):
            native.copy_codec(dev, src_shifted.view(torch.uint8), codec, 0.5)
        return
    for src, dst_off in ((src_shifted, 0), (x.cuda(), 2), (src_shifted, 2)):
        out = torch.full((nbytes + dst_off,), 0xA5, dtype=torch.uint8, device="cuda")
        native.copy_codec(out[dst_off:], src.view(torch.uint8), codec, 0.5)
        torch.cuda.synchronize()
        assert torch.equal(out[dst_off:].cpu(), host), f"source shifted: {src is src_shifted}, destination +{dst_off}"
        assert bool((out[:dst_off] == 0xA5).all())
