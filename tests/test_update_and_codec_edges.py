"""The fused update kernel (K_update) and the fp8 block codec at the shapes production runs and at
their edges, against plain fp64 references.

K_update is checked against fp64 `torch.optim.AdamW` / `torch.optim.SGD`, fed with gradients that an
independent Python decoder reads from the very bytes the kernel reads. The shapes walk the TMA
flavour's pipeline (stage reuse, mbarrier parity flips, uneven tiles per CTA, the scalar tail) and the
LDG flavour's grid passes; guard regions around every buffer catch stray writes. The fp8 codec is
checked against an exact encoder built on `torch.frexp`, at tiny, denormal, boundary and huge block
maxima. Every case runs on the CPU twin (`cpu`) and on the sm_100a kernels (`cuda`, marked gpu).
"""
import os
import re
import subprocess
import sys

import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)

T = 2048              # elements per k_update_tma tile
COPY_CHUNK = 32 * 1024  # bytes per k_copy_tma stage
GUARD = 4 * T         # guard bytes before and after every buffer: a tile of fp32 state, 16-byte aligned
SENTINEL = 0xA5
CPU_MAX_N = 1 << 20
B200_SMS = 148        # the twin has no grid: on the CPU the shapes are those of a B200

DEVICES = [pytest.param("cpu", id="cpu"), pytest.param("cuda", id="cuda", marks=pytest.mark.gpu)]


def _require(device):
    if device == "cuda" and not torch.cuda.is_available():
        pytest.skip("no CUDA device")


def _sm_count(device):
    if device == "cpu":
        return B200_SMS
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


def _f32(x):
    """the float32 value the kernel receives for a Python float"""
    return float(torch.tensor(x, dtype=torch.float32))


# ---------------------------------------------------------------------------------------------
# guarded buffers
# ---------------------------------------------------------------------------------------------
class Guarded:
    """`view` starts GUARD bytes into a sentinel-filled byte buffer and is followed by GUARD more"""

    def __init__(self, nbytes, device):
        self.nbytes = nbytes
        self.buf = torch.full((GUARD + nbytes + GUARD,), SENTINEL, dtype=torch.uint8, device=device)
        self.bytes = self.buf[GUARD:GUARD + nbytes]

    def view(self, dtype):
        return self.bytes.view(dtype)

    def guards_intact(self):
        head, tail = self.buf[:GUARD], self.buf[GUARD + self.nbytes:]
        return bool((head == SENTINEL).all()) and bool((tail == SENTINEL).all())


# ---------------------------------------------------------------------------------------------
# K_update cases
# ---------------------------------------------------------------------------------------------
FMT_BYTES = {"bf16": 2, "f32": 4}


class Case:
    def __init__(self, name, n, fmt, W, fan, opt, flavour, out_f32=False, max_ctas=0, steps=None):
        self.name, self.n_of, self.fmt, self.W, self.fan, self.opt = name, n, fmt, W, fan, opt
        self.flavour, self.out_f32, self.max_ctas = flavour, out_f32, max_ctas
        self.steps = steps or (4 if opt == "adamw" else 3)

    def __repr__(self):
        return self.name


# n as a function of the SM count S; `flavour` is what the default build must run for the case
UPDATE_CASES = [
    # 4T - 1: fewer than 4 full tiles, the TMA flavour declines; LDG with a 7-element tail
    Case("4T-1/bf16/W1/fan1/adamw", lambda S: 4 * T - 1, "bf16", 1, 1, "adamw", "ldg"),
    Case("4T-1/fp8/W3/fan9/sgd", lambda S: 4 * T - 1, "fp8", 3, 9, "sgd", "ldg"),
    # 4T: the smallest TMA launch, no tail
    Case("4T/bf16/W8/fan1/adamw", lambda S: 4 * T, "bf16", 8, 1, "adamw", "tma"),
    Case("4T/f32/W6/fan1/sgd", lambda S: 4 * T, "f32", 6, 1, "sgd", "tma"),  # 3 stages = 216 KB
    Case("4T/fp8/W5/fan0/adamw", lambda S: 4 * T, "fp8", 5, 0, "adamw", "ldg"),
    # S*T: exactly one tile per CTA
    Case("ST/f32/W7/fan1/adamw", lambda S: S * T, "f32", 7, 1, "adamw", "ldg"),  # 240 KB: LDG
    Case("ST/fp8/W1/fan1/sgd", lambda S: S * T, "fp8", 1, 1, "sgd", "ldg"),
    Case("ST/bf16/W3/fan9/sgd", lambda S: S * T, "bf16", 3, 9, "sgd", "tma"),
    # 3*S*T + 2047: every stage used once; CTA 0 runs a 2047-element scalar tail
    Case("3ST+2047/bf16/W5/fan1/adamw", lambda S: 3 * S * T + 2047, "bf16", 5, 1, "adamw", "tma"),
    Case("3ST+2047/fp8/W8/fan1/adamw", lambda S: 3 * S * T + 2047, "fp8", 8, 1, "adamw", "ldg"),
    Case("3ST+2047/f32/W3/fan1/sgd/out_f32", lambda S: 3 * S * T + 2047, "f32", 3, 1, "sgd", "ldg",
         out_f32=True),
    # 7*S*T + 13: the mbarrier parity flips twice; the LDG grid (4 CTAs/SM) makes two passes
    Case("7ST+13/f32/W8/fan1/adamw", lambda S: 7 * S * T + 13, "f32", 8, 1, "adamw", "ldg"),
    Case("7ST+13/bf16/W1/fan0/sgd", lambda S: 7 * S * T + 13, "bf16", 1, 0, "sgd", "tma"),
    Case("7ST+13/fp8/W3/fan1/sgd", lambda S: 7 * S * T + 13, "fp8", 3, 1, "sgd", "ldg"),
    # one CTA streams 40 tiles through the 3-stage ring
    Case("40T+5/bf16/W3/fan1/adamw/1cta", lambda S: 40 * T + 5, "bf16", 3, 1, "adamw", "tma", max_ctas=1),
    Case("40T+5/fp8/W1/fan1/adamw/1cta", lambda S: 40 * T + 5, "fp8", 1, 1, "adamw", "ldg", max_ctas=1),
    # 10 tiles over 3 CTAs: 4 / 3 / 3
    Case("10T+1000/f32/W5/fan9/adamw/3cta", lambda S: 10 * T + 1000, "f32", 5, 9, "adamw", "tma", max_ctas=3),
    Case("10T+1000/fp8/W5/fan1/sgd/3cta", lambda S: 10 * T + 1000, "fp8", 5, 1, "sgd", "ldg", max_ctas=3),
    # the chunk size training and bench.py push by default
    Case("32Mi/bf16/W2/fan3/adamw", lambda S: 32 << 20, "bf16", 2, 3, "adamw", "tma", steps=1),
]
BIG_CASE = UPDATE_CASES[-1].name


def _update_params():
    params = []
    for c in UPDATE_CASES:
        if c.n_of(B200_SMS) <= CPU_MAX_N:
            params.append(pytest.param("cpu", c, id=f"cpu-{c.name}"))
        params.append(pytest.param("cuda", c, id=f"cuda-{c.name}", marks=pytest.mark.gpu))
    return params


def _forced_update_flavour():
    v = os.environ.get("PS_UPDATE_TMA")
    if v is None:
        return None
    try:
        return int(v) != 0
    except ValueError:
        return False


def expected_flavour(c, n):
    """which K_update flavour must run `c` in this process (PS_UPDATE_TMA forces one for every format)"""
    forced = _forced_update_flavour()
    if forced is None:
        return c.flavour
    if not forced:
        return "ldg"
    grad_tile = {"bf16": 2 * T, "fp8": T, "f32": 4 * T}[c.fmt]
    fits = 3 * (3 * 4 * T + c.W * grad_tile) <= 220 * 1024
    return "tma" if (fits and n // T >= 4 and not c.out_f32) else "ldg"


def _slot_bytes(fmt, n):
    npad = (n + 31) // 32 * 32
    return {"bf16": 2 * n, "f32": 4 * n, "fp8": npad + npad // 32}[fmt]


def decode_slot(slot_bytes, fmt, n):
    """fp64 value of a gradient slot, read from its bytes without the project's decoders"""
    if fmt == "bf16":
        return slot_bytes[:2 * n].view(torch.bfloat16).double()
    if fmt == "f32":
        return slot_bytes[:4 * n].view(torch.float32).double()
    npad = (n + 31) // 32 * 32
    q = slot_bytes[:npad].view(torch.float8_e4m3fn).float().double()
    e = slot_bytes[npad:npad + npad // 32].double() - 127.0
    return (q.view(-1, 32) * torch.exp2(e)[:, None]).view(-1)[:n]


def _fill_slot(native, slot, fmt, g32):
    if fmt == "bf16":
        slot.view(torch.bfloat16).copy_(g32.to(torch.bfloat16))
    elif fmt == "f32":
        slot.view(torch.float32).copy_(g32)
    else:  # the encoder of the same device: the push kernel on the GPU, its twin on the CPU
        native.copy_codec(slot, g32.contiguous().view(torch.uint8), native.CODEC_F32_TO_FP8BLOCK, 1.0)


def _kernel_flavours(prof):
    names = {e.name for e in prof.events()}
    ran = set()
    for name in names:
        if "k_update_tma" in name:
            ran.add("tma")
        elif re.search(r"\bk_update<", name):
            ran.add("ldg")
    return ran


def run_update_case(native, c, device, check_flavour=None):
    """run `c` for c.steps steps against fp64 torch.optim; returns the set of K_update flavours seen"""
    S = _sm_count(device)
    n = c.n_of(S)
    W, adam = c.W, c.opt == "adamw"
    gen = torch.Generator(device=device).manual_seed(n * 31 + W * 7 + c.fan)
    gfmt = {"bf16": native.GRAD_BF16, "f32": native.GRAD_F32, "fp8": native.GRAD_FP8BLOCK}[c.fmt]
    lr, b1, b2, eps, wd = (1e-2, 0.9, 0.95, 1e-8, 0.1) if adam else (0.1, 0.9, 0.0, 0.0, 0.01)
    gs = _f32(1.0 / W)

    bufs = {k: Guarded(4 * n, device) for k in ("master", "m", "v")}
    master, m, v = (bufs[k].view(torch.float32) for k in ("master", "m", "v"))
    master.copy_(torch.randn(n, generator=gen, device=device))
    m.zero_()  # both oracles start their moments at zero
    if adam:
        v.zero_()
    else:  # SGD must not touch v at all
        v.copy_(torch.randn(n, generator=gen, device=device))
    v_before = v.clone()
    out_dtype = torch.float32 if c.out_f32 else torch.bfloat16
    out_bufs = [Guarded(n * (4 if c.out_f32 else 2), device) for _ in range(c.fan)]
    outs = [b.view(out_dtype) for b in out_bufs]
    slot_bufs = [Guarded(_slot_bytes(c.fmt, n), device) for _ in range(W)]

    p64 = torch.nn.Parameter(master.double().clone())
    if adam:
        oracle = torch.optim.AdamW([p64], lr=_f32(lr), betas=(_f32(b1), _f32(b2)), eps=_f32(eps),
                                   weight_decay=_f32(wd), foreach=False)
    else:
        oracle = torch.optim.SGD([p64], lr=_f32(lr), momentum=_f32(b1), dampening=0,
                                 weight_decay=_f32(wd), foreach=False)
    seen = set()
    for step in range(1, c.steps + 1):
        # fresh gradients; the W slots of one element share a sign, so the fp32 sum in the kernel
        # cannot cancel to a different sign than the fp64 sum (AdamW's m/sqrt(v) would flip with it)
        sign = torch.randint(0, 2, (n,), generator=gen, device=device).float() * 2 - 1
        mag = torch.logspace(-3, 1, n, device=device)  # so that fp8 blocks get many different scales
        for b in slot_bufs:
            g32 = sign * mag * torch.rand(n, generator=gen, device=device) * 0.05
            _fill_slot(native, b.bytes, c.fmt, g32)
        slots_before = [b.buf.clone() for b in slot_bufs]
        g64 = sum(decode_slot(b.bytes, c.fmt, n) for b in slot_bufs) * gs

        def launch():
            native.fused_update([b.bytes if c.fmt == "fp8" else b.view(torch.bfloat16 if c.fmt == "bf16" else
                                                                             torch.float32) for b in slot_bufs],
                                gfmt, master, m, v, outs, optimizer=c.opt, lr=lr, beta1=b1, beta2=b2, eps=eps,
                                weight_decay=wd, step=step, grad_scale=gs, max_ctas=c.max_ctas)
            if device == "cuda":
                torch.cuda.synchronize()

        if device == "cuda" and step == 1 and check_flavour:
            from torch.profiler import ProfilerActivity, profile

            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                launch()
            seen = _kernel_flavours(prof)
            want = expected_flavour(c, n)
            assert seen == {want}, f"{c.name} (n={n}): expected the {want} flavour, the profiler saw {seen}"
        else:
            launch()
        p64.grad = g64
        oracle.step()

        # exact invariants
        for k, b in bufs.items():
            assert b.guards_intact(), f"step {step}: a write landed next to {k}"
        for i, b in enumerate(out_bufs):
            assert b.guards_intact(), f"step {step}: a write landed next to output {i}"
        for i, b in enumerate(slot_bufs):
            assert torch.equal(b.buf, slots_before[i]), f"step {step}: gradient slot {i} changed"
        for i, o in enumerate(outs):
            want = master if c.out_f32 else master.to(torch.bfloat16)
            assert torch.equal(o, want), f"step {step}: output {i} is not the updated master"
        if not adam:
            assert torch.equal(v, v_before), f"step {step}: SGD wrote v"

        # The single-step tolerances of the older tests (rtol 1e-5, atol 1e-6 on p), times the step
        # count: the kernel carries fp32 state (and uses MUFU sqrt / reciprocal) and the oracle fp64,
        # so their difference can grow by one step's rounding each step, never by more.
        st = oracle.state[p64]
        torch.testing.assert_close(master.double(), p64.detach(), rtol=1e-5 * step, atol=1e-6 * step,
                                   msg=lambda s: f"step {step} p: {s}")
        m_ref = st["exp_avg"] if adam else st["momentum_buffer"]
        torch.testing.assert_close(m.double(), m_ref, rtol=1e-5 * step, atol=1e-7 * step,
                                   msg=lambda s: f"step {step} m: {s}")
        if adam:
            torch.testing.assert_close(v.double(), st["exp_avg_sq"], rtol=1e-5 * step, atol=1e-9 * step,
                                       msg=lambda s: f"step {step} v: {s}")
    return seen


@pytest.mark.parametrize("device,case", _update_params())
def test_fused_update_matches_fp64_optimizer(native, device, case):
    _require(device)
    run_update_case(native, case, device, check_flavour=True)


# ---------------------------------------------------------------------------------------------
# raw copy, TMA flavour
# ---------------------------------------------------------------------------------------------
def copy_cases(S):
    """(bytes, max_ctas): under, at and just over one stage (the 15 bytes after the last 16-byte word
    go to the byte kernel), three chunks per CTA, and one CTA wrapping its 4-stage ring with a short
    last chunk"""
    C = COPY_CHUNK
    return [(C - 1, 0), (C, 0), (C + 15, 0), (3 * S * C + 7, 0), (9 * C + 4096 + 3, 1)]


def run_copy_tma_cases(native):
    from torch.profiler import ProfilerActivity, profile

    S = _sm_count("cuda")
    forced = os.environ.get("PS_COPY_TMA")
    tma_on = forced is not None and forced.strip() not in ("", "0")
    gen = torch.Generator(device="cuda").manual_seed(5)
    for nbytes, max_ctas in copy_cases(S):
        src = torch.randint(0, 256, (nbytes,), dtype=torch.uint8, device="cuda", generator=gen)
        dst = Guarded(nbytes, "cuda")
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            native.copy_codec(dst.bytes, src, native.CODEC_RAW, 1.0, max_ctas)
            torch.cuda.synchronize()
        ran_tma = any("k_copy_tma" in e.name for e in prof.events())
        assert ran_tma == (tma_on and nbytes >= COPY_CHUNK), (nbytes, ran_tma)
        assert torch.equal(dst.bytes, src), f"{nbytes} B, max_ctas={max_ctas}: bytes differ"
        assert dst.guards_intact(), f"{nbytes} B, max_ctas={max_ctas}: a write landed outside the destination"


# ---------------------------------------------------------------------------------------------
# forced flavours: PS_UPDATE_TMA / PS_COPY_TMA are read once per process, so they run in children
# ---------------------------------------------------------------------------------------------
def _child_main(which):
    import pslite_b200

    native = pslite_b200.native()
    if which == "copy":
        run_copy_tma_cases(native)
    else:
        seen = set()
        for c in UPDATE_CASES:
            if c.name != BIG_CASE:
                print(c.name, flush=True)
                seen |= run_update_case(native, c, "cuda", check_flavour=True)
        print("flavours", sorted(seen), flush=True)
    print("child ok", flush=True)


@pytest.mark.gpu
@pytest.mark.parametrize("env", [{"PS_UPDATE_TMA": "0"}, {"PS_UPDATE_TMA": "1"}, {"PS_COPY_TMA": "1"}],
                         ids=["update_ldg", "update_tma", "copy_tma"])
def test_forced_flavours_in_child_process(env):
    """the same cases with PS_UPDATE_TMA=0 (bf16/f32 on LDG, beyond one grid pass), PS_UPDATE_TMA=1
    (fp8 slots on the TMA flavour) and PS_COPY_TMA=1 (k_copy_tma)"""
    _require("cuda")
    which = "copy" if "PS_COPY_TMA" in env else "update"
    child_env = {k: v for k, v in os.environ.items() if k not in ("PS_UPDATE_TMA", "PS_COPY_TMA")}
    child_env.update(env)
    code = (f"import sys; sys.path[:0] = [{HERE!r}, {ROOT!r}]; "
            f"import test_update_and_codec_edges as t; t._child_main({which!r})")
    r = subprocess.run([sys.executable, "-c", code], env=child_env, capture_output=True, text=True,
                       timeout=1200, cwd=ROOT)
    assert r.returncode == 0 and "child ok" in r.stdout, (r.stdout[-3000:] + r.stderr[-6000:])
    if env.get("PS_UPDATE_TMA") == "1":
        assert "'tma'" in r.stdout.splitlines()[-2]


# ---------------------------------------------------------------------------------------------
# alignment, argument checks, several devices
# ---------------------------------------------------------------------------------------------
def _small_update_args(device, n=4 * T, fmt="bf16"):
    master = torch.randn(n, device=device)
    m, v = torch.zeros(n, device=device), torch.zeros(n, device=device)
    g = (torch.randn(n, device=device) * 0.01).to(torch.bfloat16)
    out = torch.empty(n, dtype=torch.bfloat16, device=device)
    return [g], master, m, v, [out]


@pytest.mark.gpu
@pytest.mark.parametrize("which", ["master", "m", "v", "grad", "out"])
def test_misaligned_update_pointer_is_refused_before_launch(native, which):
    """both flavours move 16-byte vectors: ps_launch_update refuses any other alignment"""
    _require("cuda")
    n = 4 * T
    grads, master, m, v, outs = _small_update_args("cuda", n)
    shifted = {  # a view starting 4 (fp32) / 8 (bf16) bytes into a 16-byte aligned allocation
        "master": torch.randn(n + 1, device="cuda")[1:],
        "m": torch.zeros(n + 1, device="cuda")[1:],
        "v": torch.zeros(n + 1, device="cuda")[1:],
        "grad": torch.zeros(n + 4, dtype=torch.bfloat16, device="cuda")[4:],
        "out": torch.zeros(n + 4, dtype=torch.bfloat16, device="cuda")[4:],
    }[which]
    if which == "master":
        master = shifted
    elif which == "m":
        m = shifted
    elif which == "v":
        v = shifted
    elif which == "grad":
        grads = [shifted]
    else:
        outs = [shifted]
    before = [t.clone() for t in (master, m, v)]
    with pytest.raises(RuntimeError, match="misaligned"):
        native.fused_update(grads, native.GRAD_BF16, master, m, v, outs, optimizer="adamw", step=1)
    torch.cuda.synchronize()
    assert all(torch.equal(a, b) for a, b in zip((master, m, v), before)), "a refused launch wrote state"


BAD_ARGUMENTS = {
    "no_slots": lambda a: a.update(grads=[]),
    "nine_slots": lambda a: a.update(grads=a["grads"] * 9),
    "ten_outputs": lambda a: a.update(outs=a["outs"] * 10),
    "short_bf16_slot": lambda a: a.update(grads=[a["grads"][0][:-1]]),
    "short_f32_slot": lambda a: a.update(grad_format="f32", grads=[torch.zeros(a["n"] - 1)]),
    "short_fp8_slot": lambda a: a.update(grad_format="fp8", grads=[torch.zeros(_slot_bytes("fp8", a["n"]) - 1,
                                                                               dtype=torch.uint8)]),
    "bad_format": lambda a: a.update(grad_format=7),
    "short_m": lambda a: a.update(m=a["m"][:-1]),
    "short_v_adamw": lambda a: a.update(v=a["v"][:-1]),
    "short_output": lambda a: a.update(outs=[a["outs"][0][:-1]]),
    "mixed_output_dtypes": lambda a: a.update(outs=[a["outs"][0], torch.zeros(a["n"])]),
    "fp16_output": lambda a: a.update(outs=[torch.zeros(a["n"], dtype=torch.float16)]),
    "strided_output": lambda a: a.update(outs=[torch.zeros(2 * a["n"], dtype=torch.bfloat16)[::2]]),
    "strided_slot": lambda a: a.update(grads=[torch.zeros(2 * a["n"], dtype=torch.bfloat16)[::2]]),
    "strided_m": lambda a: a.update(m=torch.zeros(2 * a["n"])[::2]),
    "slot_on_other_device": lambda a: a.update(grads=[torch.empty(a["n"], dtype=torch.bfloat16, device="meta")]),
    "output_on_other_device": lambda a: a.update(outs=[torch.empty(a["n"], dtype=torch.bfloat16, device="meta")]),
    "m_on_other_device": lambda a: a.update(m=torch.empty(a["n"], device="meta")),
    "adamw_step_0": lambda a: a.update(step=0),
    "unknown_optimizer": lambda a: a.update(optimizer="adam"),
}


@pytest.mark.parametrize("bad", sorted(BAD_ARGUMENTS))
def test_fused_update_binding_refuses_bad_arguments(native, bad):
    """every size the kernel and its twin trust is checked before either runs (on the CPU here, where
    an undersized buffer would be a heap overrun)"""
    n = 1000
    grads, master, m, v, outs = _small_update_args("cpu", n)
    a = dict(n=n, grads=grads, grad_format="bf16", master=master, m=m, v=v, outs=outs, step=1, optimizer="adamw")
    BAD_ARGUMENTS[bad](a)
    fmt = {"bf16": native.GRAD_BF16, "f32": native.GRAD_F32, "fp8": native.GRAD_FP8BLOCK}.get(a["grad_format"],
                                                                                            a["grad_format"])
    before = master.clone()
    with pytest.raises(RuntimeError, match="fused_update"):
        native.fused_update(a["grads"], fmt, a["master"], a["m"], a["v"], a["outs"], optimizer=a["optimizer"],
                            step=a["step"])
    assert torch.equal(master, before)


def test_fused_update_binding_accepts_sgd_without_v_and_no_outputs(native):
    """SGD never reads v, and fan-out 0 is legal: the checks must not refuse either"""
    n = 1000
    grads, master, m, _, _ = _small_update_args("cpu", n)
    p0 = master.clone()
    native.fused_update(grads, native.GRAD_BF16, master, m, torch.empty(0), [], optimizer="sgd", lr=0.5,
                        beta1=0.0)
    torch.testing.assert_close(master, p0 - 0.5 * grads[0].float(), rtol=1e-6, atol=1e-7)


@pytest.mark.gpu
def test_tma_update_on_every_device_of_one_process(native):
    """the shared-memory attribute of k_update_tma is set per device: a process that drives several
    GPUs (one GpuServer per device) must be able to run the TMA flavour on each of them"""
    if not torch.cuda.is_available() or torch.cuda.device_count() < 2:
        pytest.skip("needs 2 or more GPUs")
    from torch.profiler import ProfilerActivity, profile

    for d in range(torch.cuda.device_count()):
        with torch.cuda.device(d):
            S = _sm_count("cuda")
            n = 3 * S * T
            g = [(torch.randn(n, device=f"cuda:{d}") * 0.01).to(torch.bfloat16) for _ in range(2)]
            master = torch.randn(n, device=f"cuda:{d}")
            m, v = torch.zeros_like(master), torch.zeros_like(master)
            out = torch.empty(n, dtype=torch.bfloat16, device=f"cuda:{d}")
            p0 = master.clone()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                native.fused_update(g, native.GRAD_BF16, master, m, v, [out], optimizer="sgd", lr=0.5, beta1=0.0,
                                    grad_scale=0.5)
                torch.cuda.synchronize()
            assert "tma" in _kernel_flavours(prof), f"cuda:{d}: the TMA flavour did not run"
            ref = p0 - 0.5 * 0.5 * (g[0].float() + g[1].float())
            torch.testing.assert_close(master, ref, rtol=1e-6, atol=1e-7)
            assert torch.equal(out, master.to(torch.bfloat16))


# ---------------------------------------------------------------------------------------------
# fp8 block codec
# ---------------------------------------------------------------------------------------------
def ref_fp8_exact(x, scale):
    """exact block-scaled e4m3 encoding of x * scale (scale applied in fp32, as the kernels do):
    returns (scale bytes, fp32 value the wire decodes to). The block exponent comes from torch.frexp:
    amax = f * 2^k with f in [0.5, 1), i.e. (2f) * 2^(k-1); the smallest e with amax / 2^e <= 448 =
    1.75 * 2^8 is k - 9 + (2f > 1.75), clamped to [-126, 127]. An infinite amax has exponent field 255
    (k - 1 = 128) and no mantissa: e = 120. NaN does not take part in amax."""
    x32 = x.detach().cpu().float() * torch.tensor(scale, dtype=torch.float32)
    n = x32.numel()
    npad = (n + 31) // 32 * 32
    xb = torch.cat([x32, torch.zeros(npad - n)]).view(-1, 32)
    amax = torch.where(torch.isnan(xb), torch.zeros_like(xb), xb.abs()).amax(dim=1)
    f, k = torch.frexp(amax)
    e = (k.long() - 9 + (2 * f > 1.75).long()).clamp(-126, 127)
    e = torch.where(torch.isinf(amax), torch.full_like(e, 120), e)
    byte = torch.where(amax > 0, e + 127, torch.zeros_like(e))
    y = (xb.double() * torch.exp2(-e.double())[:, None]).clamp(-448.0, 448.0)  # exact; satfinite
    q = y.to(torch.float8_e4m3fn).float().double()
    dec = (q * torch.exp2(byte.double() - 127.0)[:, None]).float()  # fp32, like every decoder
    return byte.to(torch.uint8), dec.view(-1)[:n]


def _encode(native, x, bf16_src, scale, device, max_ctas=0):
    codec = native.CODEC_BF16_TO_FP8BLOCK if bf16_src else native.CODEC_F32_TO_FP8BLOCK
    src = x.to(device=device, dtype=torch.bfloat16 if bf16_src else torch.float32).contiguous()
    wire = torch.zeros(native.wire_bytes(codec, src.numel() * src.element_size()), dtype=torch.uint8, device=device)
    native.copy_codec(wire, src.view(torch.uint8), codec, scale, max_ctas)
    dec = torch.empty(src.numel(), dtype=torch.float32, device=device)
    native.decode(dec, wire, src.numel(), native.GRAD_FP8BLOCK)
    if device == "cuda":
        torch.cuda.synchronize()
    return src, wire.cpu(), dec.cpu()


def check_fp8_codec(native, x, bf16_src, device, scale=1.0, max_ctas=0):
    src, wire, dec = _encode(native, x, bf16_src, scale, device, max_ctas)
    n = src.numel()
    npad = (n + 31) // 32 * 32
    ref_bytes, ref_dec = ref_fp8_exact(src.float(), scale)
    assert torch.equal(wire[npad:], ref_bytes), (
        f"scale bytes differ in blocks {torch.nonzero(wire[npad:] != ref_bytes).view(-1)[:8].tolist()}")
    # the wire, read by the independent decoder, and the project's decoder agree with the reference
    ours = decode_slot(wire, "fp8", n).float()
    torch.testing.assert_close(ours, ref_dec, rtol=0, atol=0, equal_nan=True)
    torch.testing.assert_close(dec, ref_dec, rtol=0, atol=0, equal_nan=True)
    finite = bool(torch.isfinite(src.float()).all())
    if device == "cuda" and finite:  # the kernel and its CPU twin write the same bytes
        _, host_wire, _ = _encode(native, x, bf16_src, scale, "cpu")
        assert torch.equal(wire, host_wire)
    return src, dec


def _next_above(v, dtype):
    t = torch.tensor([v], dtype=dtype)
    bits = t.view(torch.int16 if dtype == torch.bfloat16 else torch.int32)
    return float((bits + 1).view(dtype))


EDGE_AMAX = [0.0, -0.0, 2.0 ** -149, 1e-38, 2.0 ** -119, 2.0 ** -118, 2.0 ** -117, 3e38]


def _edge_blocks(dtype):
    """one 32-element block per controlled amax; the maximum sits at a different position in each
    block and carries alternating signs, the other elements are up to 0.9 of it"""
    gen = torch.Generator().manual_seed(11)
    amaxes = list(EDGE_AMAX)
    for k in (-20, 0, 20):
        a = 448.0 * 2.0 ** k
        amaxes += [a, _next_above(a, dtype)]
    blocks = []
    for i, a in enumerate(amaxes):
        if a == 0.0:
            b = torch.full((32,), a, dtype=torch.float64)  # keeps the sign of -0
        else:
            b = (torch.rand(32, generator=gen, dtype=torch.float64) * 1.8 - 0.9) * a
            b[(5 * i) % 32] = -a if i % 2 else a
        blocks.append(b.to(dtype))
    return torch.cat(blocks)


@pytest.mark.parametrize("bf16_src", [False, True], ids=["f32", "bf16"])
@pytest.mark.parametrize("device", DEVICES)
def test_fp8_codec_edge_block_maxima(native, device, bf16_src):
    """zero, -0, denormal, tiny (2^-119 used to decode at twice its value), 448 * 2^k and the next
    value above it, and 3e38"""
    _require(device)
    dtype = torch.bfloat16 if bf16_src else torch.float32
    check_fp8_codec(native, _edge_blocks(dtype), bf16_src, device)


@pytest.mark.parametrize("bf16_src", [False, True], ids=["f32", "bf16"])
@pytest.mark.parametrize("device", DEVICES)
def test_fp8_codec_block_maximum_at_every_position(native, device, bf16_src):
    """amax is reduced over the four lanes of a block with shuffles: a maximum in any lane's eight
    elements must set the scale of all 32"""
    _require(device)
    gen = torch.Generator().manual_seed(3)
    x = (torch.rand(32, 32, generator=gen) * 2 - 1) * 0.01  # every other element is tiny
    for j in range(32):
        x[j, j] = 300.0 if j % 2 else -300.0
    check_fp8_codec(native, x.view(-1), bf16_src, device)


@pytest.mark.parametrize("bf16_src", [False, True], ids=["f32", "bf16"])
@pytest.mark.parametrize("device", DEVICES)
@pytest.mark.parametrize("n,scale,max_ctas", [(32 * 1000 + 1, 1.0, 0), (32 * 1000 + 7, 1.0, 0),
                                               (32 * 1000 + 8, 1.0, 0), (32 * 1000 + 9, 1.0, 0),
                                               (32 * 1000 + 31, 1.0, 0),
                                               # one CTA (2048 elements per pass): 3 passes, then a
                                               # warp with 24 live lanes of 32
                                               (3 * 2048 + 32 * 5 + 7, 1.0, 1),
                                               (100003, 0.37, 0)])
def test_fp8_codec_ragged_lengths_passes_and_scale(native, device, bf16_src, n, scale, max_ctas):
    _require(device)
    gen = torch.Generator().manual_seed(n)
    x = torch.randn(n, generator=gen) * torch.logspace(-30, 30, n)
    check_fp8_codec(native, x, bf16_src, device, scale=scale, max_ctas=max_ctas)


@pytest.mark.parametrize("bf16_src", [False, True], ids=["f32", "bf16"])
@pytest.mark.parametrize("device", DEVICES)
def test_fp8_codec_nan_and_inf(native, device, bf16_src):
    """NaN stays NaN (and does not set the block scale); +-Inf saturates to 448 at the largest scale
    an fp32 exponent gives, which decodes to +-Inf again"""
    _require(device)
    gen = torch.Generator().manual_seed(13)
    x = torch.randn(4, 32, generator=gen)
    x[0, 3] = float("nan")
    x[1, 17] = float("inf")
    x[2, 30] = float("-inf")
    x[3, 0], x[3, 9] = float("nan"), float("-inf")
    src, dec = check_fp8_codec(native, x.view(-1), bf16_src, device)
    s = src.float().cpu()
    assert torch.equal(torch.isnan(dec), torch.isnan(s))
    assert torch.equal(dec[torch.isinf(s)], s[torch.isinf(s)])
