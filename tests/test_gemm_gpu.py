"""otb_gemm_bf16 against a plain fp64 reference: every kernel family the host dispatch can choose, each operand layout,
each compiled epilogue class plus the generic one, and the shape tails where tiled kernels go wrong.

Reference: A.double() @ B.double().T on the device, then the epilogue in fp64 in the order include/otter_b200.h
documents (bias, aux_out = pre-activation, act or act'(aux_in), x alpha * (tanh(g) or g), + residual, + old value).
Every input is bf16 (fp32 where the ABI says so), so the reference sees exactly what the kernel sees.

Tolerance (gemm_tolerance) follows from the arithmetic instead of being picked: the tensor cores add each K=16 step
into an fp32 accumulator with truncation, so the accumulated product is off by at most
e_acc = C_ACC * ceil(K/16) * 2^-24 * (|A| |B|^T); the epilogue carries e_acc through |act'| * |scale|, adds a few fp32
roundings, and a bf16 output adds its own rounding (one bf16 ulp of the larger of |ref| and |got|).

Every operand is a view inside a larger buffer whose padding (extra columns, extra rows) is bf16 NaN, so a read past the
logical extent turns into NaN in the output.  Every output is a view inside a buffer pre-filled with a sentinel bit
pattern that must survive outside [M, N].  Each case names the kernel the dispatch should pick and checks it against
the kernel torch.profiler records (on a 148-SM B200; other SM counts skip only that assertion).

The read-once switches OTB_GEMM_EPI_TMA=0 (direct-store epilogue), OTB_GEMM_EPI_CLS=0 (generic TMA-store epilogue) and
OTB_GEMM_2CTA=0 (BN256 kernels instead of the cta_group::2 pair kernel) are covered by running this file again in a
child process under each of them (test_switch_configuration).

OTB_GEMM_TEST_REPORT=<file> appends one JSON line per case (configuration, kernel, largest error / tolerance, card).
"""
import ctypes as C
import json
import math
import os
import re
import subprocess
import sys
from dataclasses import dataclass

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEV = "cuda:0"
BF16 = torch.bfloat16
# Truncating fp32 accumulation loses less than 1 ulp = 2^-23 of the running sum per K=16 step.  Checked on a B200:
# fp32 outputs use at most 0.17 of the resulting tolerance (profiles/r03_gemm_parity.md).
C_ACC = 2.0
SM_EXPECTED = 148    # the dispatch expectations below hold for a B200 with 148 SMs
CHILD_ENV = "OTB_GEMM_TEST_CHILD"
REPORT_ENV = "OTB_GEMM_TEST_REPORT"
SWITCHES = ("OTB_GEMM_EPI_TMA=0", "OTB_GEMM_EPI_CLS=0", "OTB_GEMM_2CTA=0")


# ------------------------------------------------------------------------------------------------------------------
# fp64 reference and the tolerance derived from the arithmetic (device-agnostic: the CPU tests check the checker)
# ------------------------------------------------------------------------------------------------------------------
def ulp_bf16(x):
    """Spacing of bf16 numbers at |x| (fp64 tensor): 2^(e - 8) for |x| in [2^(e-1), 2^e); subnormals use 2^-133."""
    _, e = torch.frexp(x.abs().clamp_min(2.0 ** -126))
    return torch.ldexp(torch.ones_like(x), (e - 8).to(torch.int32))


def gemm_tolerance(K, S, dact, scale, mag, ref, got, out_fp32, c=C_ACC):
    """Largest error an fp32-accumulating bf16 GEMM + fp32 epilogue may show at each element.
    S = |A| |B|^T (fp64); dact = |d out / d accumulator| before the scale (act'(z), or act'(aux_in) in backward);
    mag = sum of the magnitudes the epilogue adds or multiplies (its fp32 rounding budget)."""
    e_acc = c * math.ceil(K / 16) * 2.0 ** -24 * S
    carried = e_acc * dact.abs() * abs(scale)
    if out_fp32:
        return carried + 2.0 ** -21 * (mag + ref.abs())          # a few fp32 ulps of |ref| and of the added terms
    return ulp_bf16(torch.maximum(ref.abs(), got.double().abs())) + carried + 2.0 ** -20 * mag


def gelu(x):
    return 0.5 * x * (1.0 + torch.erf(x / math.sqrt(2.0)))


def gelu_grad(x):
    return 0.5 * (1.0 + torch.erf(x / math.sqrt(2.0))) + x * torch.exp(-0.5 * x * x) / math.sqrt(2.0 * math.pi)


def act_and_grad(z, act):
    if act == 1:
        return gelu(z), gelu_grad(z)
    if act == 2:                                                  # quick-GELU z * sigmoid(1.702 z)
        s = torch.sigmoid(1.702 * z)
        return z * s, s + 1.702 * z * s * (1.0 - s)
    if act == 3:                                                  # relu(z)^2
        r = z.clamp_min(0.0)
        return r * r, 2.0 * r
    return z, torch.ones_like(z)


def reference(a, b, *, bias=None, act=0, aux_in=None, gate=None, scale_tanh=True, alpha=1.0, residual=None, old=None):
    """fp64 epilogue(a[M,K] @ b[N,K]^T) in the documented order -> (ref, pre-activation, S, dact, scale, mag)."""
    a, b = a.double(), b.double()
    z = a @ b.t()
    S = a.abs() @ b.abs().t()
    if bias is not None:
        z = z + bias.double()
    if aux_in is not None:
        x = aux_in.double()
        dact = 2.0 * x.clamp_min(0.0) if act == 3 else gelu_grad(x)
        y = z * dact
    else:
        y, dact = act_and_grad(z, act)
    scale = alpha * ((math.tanh(gate) if scale_tanh else gate) if gate is not None else 1.0)
    ref = y * scale
    mag = abs(scale) * (z.abs() + y.abs())
    if residual is not None:
        ref = ref + residual.double()
        mag = mag + residual.double().abs()
    if old is not None:
        ref = ref + old.double()
        mag = mag + old.double().abs()
    return ref, z, S, dact, scale, mag


def excess(got, ref, tol):
    """err / tol per element (NaN or inf in `got` -> inf)."""
    r = (got.double() - ref).abs() / tol
    return torch.where(torch.isfinite(r), r, torch.full_like(r, math.inf))


# ------------------------------------------------------------------------------------------------------------------
# the case matrix
# ------------------------------------------------------------------------------------------------------------------
# Epilogues by name.  Classes 0-13 are the compiled TMA-store classes kEpiCls of csrc/otb_gemm.cu; "g" = generic.
EPI = {
    "plain":          (0, {}),
    "gate":           (1, dict(gate=True)),
    "bias":           (2, dict(bias=True)),
    "bias_qgelu":     (3, dict(bias=True, act=2)),
    "bias_res":       (4, dict(bias=True, res=True)),
    "res":            (5, dict(res=True)),
    "gelu_aux":       (6, dict(act=1, aux_out=True)),
    "aux_gate_res":   (7, dict(aux_out=True, gate=True, res=True)),
    "dgelu_gate":     (8, dict(aux_in=True, act=1, gate=True)),
    "dgelu":          (9, dict(aux_in=True, act=1)),
    "f32":            (10, dict(out32=True)),
    "f32_gate":       (11, dict(out32=True, gate=True)),
    "f32_acc":        (12, dict(out32=True, acc=True)),
    "f32_acc_gate":   (13, dict(out32=True, acc=True, gate=True)),
    "bias_gelu_aux":  ("g", dict(bias=True, act=1, aux_out=True)),     # MPT up-projection
    "bias_relu2_aux": ("g", dict(bias=True, act=3, aux_out=True)),     # Persimmon up-projection
    "drelu2":         ("g", dict(aux_in=True, act=3)),                 # Persimmon down-projection dgrad
    "bias_res_gate":  ("g", dict(bias=True, res=True, gate=True)),     # no compiled class
    "alpha":          (1, dict(alpha=-1.25)),                          # alpha != 1 without a scale pointer
    "gate_notanh":    (1, dict(gate=True, scale_tanh=False)),
    "f32_res32":      ("direct", dict(out32=True, res32=True)),        # fp32 residual: always the direct epilogue
}


@dataclass(frozen=True)
class Case:
    M: int
    N: int
    K: int
    layout: tuple      # (a_mn_major, b_mn_major)
    epi: str
    kern: tuple        # intended kernel: (default, under OTB_GEMM_2CTA=0)

    @property
    def id(self):
        return f"{self.M}x{self.N}x{self.K}-L{self.layout[0]}{self.layout[1]}-{self.epi}"


BN128, MC128 = ("BN128", "BN128"), ("BN128 MC", "BN128 MC")
PAIR_256, PAIR_MC256 = ("pair", "BN256"), ("pair", "BN256 MC")
L00, L01, L11 = (0, 0), (0, 1), (1, 1)
KS = (8, 72, 384, 392, 1000)     # 1 k-block, a tail, the BN128 / pair ring depth (6 stages), one more, many wraps

CASES = []


def _add(*args):
    c = Case(*args)
    if all(c.id != o.id for o in CASES):          # the matrices below overlap in a few cases: keep one of each
        CASES.append(c)


# variant matrix, layout (0,0)
for (M, N, K), kern in [
        ((1, 8, 8), BN128), ((129, 136, 72), BN128), ((300, 520, 200), BN128),
        ((2056, 1024, 1024), BN128),            # CLIP out_proj: 136 tiles
        ((896, 2824, 200), BN128),              # 161 tiles on 148 CTAs; tiles_m = 7 (odd, < 9): no multicast
        ((1024, 2560, 200), MC128), ((1100, 4096, 64), MC128),   # the second: tiles_m = 9, the last pair padded
        ((2056, 4104, 200), PAIR_MC256),        # 8-row M tail (rank-1 CTA fully out of bounds), 8-column N tail
        ((1, 50432, 512), PAIR_256), ((8, 50432, 512), PAIR_256),    # decode LM head
        ((18944, 256, 64), PAIR_MC256), ((19200, 256, 64), PAIR_MC256),   # 74 pair tiles (one pass), then 75
        ((4104, 2056, 1000), PAIR_MC256),       # 16 k-blocks on a 6-stage ring
        ((896, 5640, 200), PAIR_256),           # BN256 without multicast under OTB_GEMM_2CTA=0
        ((264, 1032, 100), BN128)]:             # K not a multiple of 8 (rows of A / B padded to a 16 B pitch)
    _add(M, N, K, L00, "plain", kern)
# K sweep of every family in every layout (MN-major operands need M, N multiples of 8)
FAMILY = [((296, 520), BN128), ((1096, 4096), MC128), ((2056, 4104), PAIR_MC256), ((896, 5640), PAIR_256)]
for (M, N), kern in FAMILY:
    for layout, epi in ((L00, "plain"), (L01, "plain"), (L11, "f32")):
        for K in KS:
            _add(M, N, K, layout, epi, kern)
# epilogue matrix at layout (0,0) on one tail shape (M, N and K tails) per family
for (M, N, K), kern in [((300, 520, 200), BN128), ((1100, 4040, 200), MC128), ((2056, 4104, 200), PAIR_MC256)]:
    for epi in EPI:
        _add(M, N, K, L00, epi, kern)
_add(896, 5640, 200, L00, "f32_res32", PAIR_256)      # BN256 with the direct epilogue (2CTA=0)
# the classes each layout really uses: dgrad (0,1) and wgrad (1,1); "plain" at (1,1) = the bf16 wire format of dp.py
for (M, N, K), kern in [((296, 520, 72), BN128), ((1096, 4040, 392), MC128), ((2056, 4104, 200), PAIR_MC256),
                        ((896, 5640, 72), PAIR_256)]:
    for epi in ("plain", "res", "dgelu", "dgelu_gate", "drelu2"):
        _add(M, N, K, L01, epi, kern)
    for epi in ("f32", "f32_gate", "f32_acc", "f32_acc_gate", "plain"):
        _add(M, N, K, L11, epi, kern)


def dispatch_model(M, N, two_cta, sms=SM_EXPECTED):
    """The host dispatch rule of otb_gemm_bf16 (csrc/otb_gemm.cu), restated to check the cases' written intent."""
    tiles_m = -(-M // 128)
    tiles256 = tiles_m * -(-N // 256)
    bn128 = N <= 128 or tiles256 < sms
    tiles = tiles_m * -(-N // 128) if bn128 else tiles256
    mc = tiles_m >= 2 and (tiles_m % 2 == 0 or tiles_m >= 9) and tiles >= sms
    if two_cta and not bn128 and (-(-M // 256)) * (-(-N // 256)) >= sms // 2:
        return "pair"
    return ("BN128" if bn128 else "BN256") + (" MC" if mc else "")


def switches(env=os.environ):
    """The read-once switches of otb_gemm_bf16 as this process sees them."""
    return dict(epi_tma=not env.get("OTB_GEMM_EPI_TMA", "1").startswith("0"),
                two_cta=int(env.get("OTB_GEMM_2CTA", "1") or 0) != 0)


def intended_kernel(case, sw):
    """Normalised kernel name: ("gemm_bf16_kernel", BN, A_MN, B_MN, MC, TS) or ("gemm2_bf16_kernel", A_MN, B_MN, TS)."""
    fam = case.kern[0] if sw["two_cta"] else case.kern[1]
    ts = int(sw["epi_tma"] and not EPI[case.epi][1].get("res32", False))
    a, b = case.layout
    if fam == "pair":
        return ("gemm2_bf16_kernel", a, b, ts)
    return ("gemm_bf16_kernel", int(fam[2:5]), a, b, int(fam.endswith("MC")), ts)


_BOOL = {"true": 1, "1": 1, "(bool)1": 1, "false": 0, "0": 0, "(bool)0": 0}


def parse_kernel(name):
    m = re.search(r"(gemm2?_bf16_kernel)<([^>]*)>", name)
    if m is None:
        return None
    args = [s.strip() for s in m.group(2).split(",")]
    if m.group(1) == "gemm_bf16_kernel":
        return (m.group(1), int(args[0]), *[_BOOL[s] for s in args[1:]])
    return (m.group(1), *[_BOOL[s] for s in args])


# ------------------------------------------------------------------------------------------------------------------
# CPU: the checker itself
# ------------------------------------------------------------------------------------------------------------------
def _control_inputs(seed=3, M=64, N=64, K=72):
    g = torch.Generator().manual_seed(seed)
    a = torch.randn(M, K, generator=g).to(BF16)
    b = (torch.randn(N, K, generator=g) / math.sqrt(K)).to(BF16)
    bias = torch.randn(N, generator=g) * 0.5
    res = torch.randn(M, N, generator=g).to(BF16)
    return a, b, bias, res


@pytest.mark.parametrize("out_fp32", [False, True])
def test_tolerance_rejects_subtly_wrong_results(out_fp32):
    """The tolerance accepts the correctly rounded result and rejects the fp64 reference recomputed with the last 8
    columns of K dropped, with `gate` in place of tanh(gate), or with the bias shifted by 8 columns."""
    a, b, bias, res = _control_inputs()
    K = a.shape[1]
    kw = dict(bias=bias, gate=0.5, residual=res)
    ref, _, S, dact, scale, mag = reference(a, b, **kw)
    cast = torch.float32 if out_fp32 else BF16

    def worst(got):
        tol = gemm_tolerance(K, S, dact, scale, mag, ref, got, out_fp32)
        r = excess(got, ref, tol).max().item()
        print(f"[gemm tol control] out_fp32={out_fp32} max err/tol {r:.3g}")
        return r

    assert worst(ref.to(cast)) <= 1.0
    wrong = {
        "K-8": reference(a[:, :K - 8], b[:, :K - 8], **kw)[0],
        "gate": reference(a, b, **{**kw, "scale_tanh": False})[0],
        "bias>>8": reference(a, b, **{**kw, "bias": bias.roll(8)})[0],
    }
    for what, w in wrong.items():
        assert worst(w.to(cast)) > 1.0, what


def test_case_matrix_intent_and_coverage():
    """Each case's written kernel matches the dispatch rule; across the default configuration and the three switch
    configurations the matrix reaches gemm_bf16_kernel in every (BN, MC, TS) combination and gemm2_bf16_kernel with
    TS 0 and 1, in layouts (0,0), (0,1) and (1,1) (BN256 with the direct epilogue: layout (0,0), via res_fp32)."""
    for c in CASES:
        assert (dispatch_model(c.M, c.N, True), dispatch_model(c.M, c.N, False)) == c.kern, c.id
        if 1 in c.layout:
            assert c.N % 8 == 0 and (c.layout[0] == 0 or c.M % 8 == 0), c.id
    seen = set()
    for env in ({}, *({s.split("=")[0]: "0"} for s in SWITCHES)):
        for c in CASES:
            seen.add((intended_kernel(c, switches(env)), c.layout))
    need = set()
    for layout in (L00, L01, L11):
        a, b = layout
        for ts in (0, 1):
            need.add((("gemm2_bf16_kernel", a, b, ts), layout))
            for mc in (0, 1):
                need.add((("gemm_bf16_kernel", 128, a, b, mc, ts), layout))
                if ts == 1 or layout == L00:
                    need.add((("gemm_bf16_kernel", 256, a, b, mc, ts), layout))
    assert need - seen == set()


def test_parse_kernel_accepts_both_bool_spellings():
    assert parse_kernel("void otb::gemm_bf16_kernel<128, false, true, (bool)1, 1>(CUtensorMap, ...)") == \
        ("gemm_bf16_kernel", 128, 0, 1, 1, 1)
    assert parse_kernel("void otb::gemm2_bf16_kernel<true, true, false>(CUtensorMap)") == ("gemm2_bf16_kernel", 1, 1, 0)
    assert parse_kernel("void otb::layernorm_fwd_kernel<4>(...)") is None


class _Recorder:
    def __init__(self):
        self.calls = 0

    def __call__(self, *args):
        self.calls += 1
        return 0


def _meta_tensor(shape, dtype, stride=None):
    """A tensor that claims to live on the GPU without touching one: _gemm_raw validates shapes before any launch."""
    t = torch.empty(shape, dtype=dtype, device="meta")
    if stride is not None:
        t = t.as_strided(shape, stride)
    return t


@pytest.mark.parametrize("what", ["out_shape", "out_dtype", "bias_len", "bias_dtype", "bias_strided", "res_shape",
                                  "res_dtype", "res32_dtype", "aux_in_shape", "aux_out_shape", "aux_out_dtype"])
def test_gemm_wrapper_validates_epilogue_operands(what, monkeypatch):
    """_gemm_raw raises OtbError for an epilogue operand that is not (M, N) of the right type — a wrong-shaped one would
    be written or read past its buffer.  otb_gemm_bf16 is replaced by a recording stub that must never be called."""
    from otter_b200 import _lib
    from otter_b200 import functional as F
    rec = _Recorder()

    class Lib:
        otb_gemm_bf16 = rec

    monkeypatch.setattr(_lib, "load", lambda: Lib)
    monkeypatch.setattr(F, "_stream", lambda: None)
    monkeypatch.setattr(torch.Tensor, "is_cuda", property(lambda self: True))
    M, N, K = 24, 40, 16
    A, B = _meta_tensor((M, K), BF16), _meta_tensor((N, K), BF16)
    out = _meta_tensor((M, N), BF16)
    epi = {}
    if what == "out_shape":
        out = _meta_tensor((M, N + 8), BF16)
    elif what == "out_dtype":
        out = _meta_tensor((M, N), torch.float16)
    elif what == "bias_len":
        epi["bias"] = _meta_tensor((N - 8,), torch.float32)
    elif what == "bias_dtype":
        epi["bias"] = _meta_tensor((N,), BF16)
    elif what == "bias_strided":
        epi["bias"] = _meta_tensor((N,), torch.float32, (2,))
    elif what == "res_shape":
        epi["residual"] = _meta_tensor((M - 1, N), BF16)
    elif what == "res_dtype":
        epi["residual"] = _meta_tensor((M, N), torch.float32)
    elif what == "res32_dtype":
        out = _meta_tensor((M, N), torch.float32)
        epi.update(residual=_meta_tensor((M, N), BF16), res_fp32=True)
    elif what == "aux_in_shape":
        epi["aux_in"] = _meta_tensor((2, M, N), BF16)
    elif what == "aux_out_shape":
        epi["aux_out"] = _meta_tensor((N, M), BF16)
    elif what == "aux_out_dtype":
        epi["aux_out"] = _meta_tensor((M, N), torch.float32)
    with pytest.raises(_lib.OtbError, match="otb_gemm_bf16|must (be|have)"):
        F._gemm_raw(A, 0, K, B, 0, K, M, N, K, out, **epi)
    assert rec.calls == 0
    # the same call with well-formed operands reaches the (stubbed) library exactly once
    ok = dict(bias=_meta_tensor((N,), torch.float32), residual=_meta_tensor((M, N), BF16),
              aux_out=_meta_tensor((M, N), BF16))
    F._gemm_raw(A, 0, K, B, 0, K, M, N, K, _meta_tensor((M, N), BF16), **ok)
    assert rec.calls == 1


# ------------------------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------------------------
SENT16, SENT32 = 0x5A5A, 0x5A5A5A5A


def _ceil8(n):
    return (n + 7) // 8 * 8


def _nan_view(rows, cols, dtype):
    """[rows, cols] view inside a buffer with 8+ extra NaN columns (pitch a multiple of 8) and 8 extra NaN rows."""
    buf = torch.full((rows + 8, _ceil8(cols) + 8), float("nan"), dtype=dtype, device=DEV)
    return buf[:rows, :cols]


def _canary_view(rows, cols, dtype):
    """[rows, cols] view inside a buffer pre-filled with a sentinel bit pattern."""
    ity = torch.int16 if dtype == BF16 else torch.int32
    buf = torch.full((rows + 8, _ceil8(cols) + 8), SENT16 if dtype == BF16 else SENT32, dtype=ity, device=DEV)
    return buf.view(dtype), buf.view(dtype)[:rows, :cols]


def _canary_intact(buf, rows, cols):
    ity = torch.int16 if buf.dtype == BF16 else torch.int32
    bits = buf.view(ity).clone()
    sent = SENT16 if buf.dtype == BF16 else SENT32
    bits[:rows, :cols] = sent
    return bool((bits == sent).all().item())


def _kernels_of(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [k for k in (parse_kernel(e.name) for e in prof.events()) if k is not None]


class Problem:
    """One case's operands (inside NaN-padded buffers), outputs (inside canary buffers) and fp64 reference."""

    def __init__(self, case, seed=0):
        self.case = case
        M, N, K = case.M, case.N, case.K
        cls, spec = EPI[case.epi]
        self.spec = spec
        g = torch.Generator(device=DEV).manual_seed(1000003 * M + 1009 * N + 7 * K + seed)

        def randn(*shape, s=1.0):
            return (torch.randn(*shape, generator=g, device=DEV) * s)

        a = randn(M, K).to(BF16)
        b = randn(N, K, s=1.0 / math.sqrt(K)).to(BF16)
        a_mn, b_mn = case.layout
        self.A = _nan_view(K, M, BF16) if a_mn else _nan_view(M, K, BF16)
        self.A.copy_(a.t() if a_mn else a)
        self.B = _nan_view(K, N, BF16) if b_mn else _nan_view(N, K, BF16)
        self.B.copy_(b.t() if b_mn else b)
        self.kw = {}
        ref_kw = {}
        if spec.get("bias"):
            bias_buf = torch.full((N + 8,), float("nan"), device=DEV)
            bias_buf[:N] = randn(N, s=0.5)
            self.kw["bias"] = ref_kw["bias"] = bias_buf[:N]
        act = spec.get("act", 0)
        self.kw["act"] = ref_kw["act"] = act
        if spec.get("aux_in"):
            self.kw["aux_in"] = _nan_view(M, N, BF16)
            self.kw["aux_in"].copy_(randn(M, N, s=2.0).to(BF16))
            ref_kw["aux_in"] = self.kw["aux_in"]
        if spec.get("gate"):
            gate = 0.7
            self.kw["scale_ptr"] = torch.tensor([gate], device=DEV)
            self.kw["scale_tanh"] = ref_kw["scale_tanh"] = spec.get("scale_tanh", True)
            ref_kw["gate"] = gate
        if "alpha" in spec:
            self.kw["alpha"] = ref_kw["alpha"] = spec["alpha"]
        if spec.get("res") or spec.get("res32"):
            rdt = torch.float32 if spec.get("res32") else BF16
            self.kw["residual"] = _nan_view(M, N, rdt)
            self.kw["residual"].copy_(randn(M, N).to(rdt))
            self.kw["res_fp32"] = bool(spec.get("res32"))
            ref_kw["residual"] = self.kw["residual"]
        self.out_fp32 = bool(spec.get("out32"))
        self.out_buf, self.out = _canary_view(M, N, torch.float32 if self.out_fp32 else BF16)
        self.old = None
        if spec.get("acc"):
            self.old = randn(M, N)
            self.kw["accumulate"] = True
            ref_kw["old"] = self.old
        self.aux_buf = None
        if spec.get("aux_out"):
            self.aux_buf, self.kw["aux_out"] = _canary_view(M, N, BF16)
        self.reset()
        self.ref, self.pre, self.S, self.dact, self.scale, self.mag = reference(a, b, **ref_kw)

    def reset(self):
        if self.old is not None:
            self.out.copy_(self.old)

    def run(self):
        from otter_b200 import functional as F
        c = self.case
        F._gemm_raw(self.A, c.layout[0], self.A.stride(0), self.B, c.layout[1], self.B.stride(0), c.M, c.N, c.K,
                    self.out, **self.kw)

    def check(self):
        """-> (max err/tol of out, of aux_out or None); asserts the canaries and every element."""
        c = self.case
        torch.cuda.synchronize()
        assert _canary_intact(self.out_buf, c.M, c.N), f"{c.id}: out written outside [M, N]"
        got = self.out.double()
        tol = gemm_tolerance(c.K, self.S, self.dact, self.scale, self.mag, self.ref, self.out, self.out_fp32)
        ratio = self._assert_within(got, self.ref, tol, "out")
        aux_ratio = None
        if self.aux_buf is not None:
            assert _canary_intact(self.aux_buf, c.M, c.N), f"{c.id}: aux_out written outside [M, N]"
            aux = self.kw["aux_out"]
            tol_a = gemm_tolerance(c.K, self.S, torch.ones_like(self.pre), 1.0, self.pre.abs(), self.pre, aux, False)
            aux_ratio = self._assert_within(aux.double(), self.pre, tol_a, "aux_out")
        return ratio, aux_ratio

    def _assert_within(self, got, ref, tol, what):
        r = excess(got, ref, tol)
        bad = r > 1.0
        if bool(bad.any().item()):
            idx = bad.nonzero()[:6].tolist()
            rows = [f"(m={i}, n={j}) got {got[i, j].item():.6g} ref {ref[i, j].item():.6g} tol {tol[i, j].item():.3g}"
                    for i, j in idx]
            raise AssertionError(f"{self.case.id}: {what}: {int(bad.sum().item())}/{r.numel()} elements outside the "
                                 f"tolerance (max err/tol {r.max().item():.3g}); first: " + "; ".join(rows))
        return r.max().item()


def _config_name():
    on = [s for s in SWITCHES if os.environ.get(s.split("=")[0], "").startswith("0")]
    return ",".join(on) or "default"


def _report(record):
    path = os.environ.get(REPORT_ENV)
    if path:
        with open(path, "a") as f:
            f.write(json.dumps(record) + "\n")


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=lambda c: c.id)
def test_gemm_matches_fp64_reference(case):
    p = Problem(case)
    kernels = _kernels_of(p.run)
    ratio, aux_ratio = p.check()
    want = intended_kernel(case, switches())
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    print(f"[gemm] {_config_name():18s} {case.id:34s} {str(kernels):48s} max err/tol {ratio:.3f}"
          + (f" aux {aux_ratio:.3f}" if aux_ratio is not None else ""))
    _report(dict(config=_config_name(), case=case.id, cls=str(EPI[case.epi][0]), kernel=kernels, want=want,
                 ratio=ratio, aux_ratio=aux_ratio, card=torch.cuda.get_device_name(0), sms=sms))
    assert len(kernels) == 1, kernels
    if sms == SM_EXPECTED:
        assert kernels[0] == want, (case.id, kernels[0], want)


@pytest.mark.gpu
@pytest.mark.parametrize("case", [Case(300, 520, 200, L00, "bias_gelu_aux", BN128),
                                  Case(1100, 4040, 200, L00, "aux_gate_res", MC128),
                                  Case(2056, 4104, 1000, L01, "dgelu_gate", PAIR_MC256),
                                  Case(1096, 4040, 392, L11, "f32_acc_gate", MC128)], ids=lambda c: c.id)
def test_gemm_is_deterministic(case):
    """Two calls on the same inputs give bitwise-equal outputs (and side outputs)."""
    p = Problem(case)
    p.run()
    p.check()
    first = p.out.clone()
    first_aux = p.kw["aux_out"].clone() if "aux_out" in p.kw else None
    p.reset()
    p.run()
    torch.cuda.synchronize()
    assert torch.equal(p.out.view(torch.int16 if p.out.dtype == BF16 else torch.int32),
                       first.view(torch.int16 if first.dtype == BF16 else torch.int32))
    if first_aux is not None:
        assert torch.equal(p.kw["aux_out"].view(torch.int16), first_aux.view(torch.int16))


@pytest.mark.gpu
def test_descriptor_cache_keys_on_shape_and_pitch():
    """TMA descriptors are cached by (base, shape, pitch, box): views with the same base pointer but a different M or
    row pitch must miss the cache and compute their own product."""
    from otter_b200 import _lib
    from otter_b200 import functional as F
    lib = _lib.load()
    K, N = 200, 520
    g = torch.Generator(device=DEV).manual_seed(7)
    store = torch.randn(600 * 264, generator=g, device=DEV).to(BF16)
    w = (torch.randn(N, K, generator=g, device=DEV) / math.sqrt(K)).to(BF16)
    for M, ld in ((256, 208), (520, 208), (520, 264)):          # same base; then more rows; then a wider pitch
        a = store[:M * ld].view(M, ld)[:, :K]
        assert a.data_ptr() == store.data_ptr()
        misses = lib.otb_tmap_cache_stat(1)
        y = F.linear_fwd(a, w)
        torch.cuda.synchronize()
        assert lib.otb_tmap_cache_stat(1) > misses, (M, ld)
        ref, _, S, dact, scale, mag = reference(a, w)
        tol = gemm_tolerance(K, S, dact, scale, mag, ref, y, False)
        assert excess(y, ref, tol).max().item() <= 1.0, (M, ld)


@pytest.mark.gpu
def test_layout_a_mn_b_k_is_unsupported_before_any_launch():
    """Layout (A MN-major, B K-major) has no kernel: OTB_ERR_UNSUPPORTED, and nothing is launched."""
    from otter_b200 import _lib
    lib = _lib.load()
    A = torch.zeros(64, 128, dtype=BF16, device=DEV)        # [K][M]
    B = torch.zeros(128, 64, dtype=BF16, device=DEV)        # [N][K]
    out = torch.zeros(128, 128, dtype=BF16, device=DEV)
    e = _lib.GemmEpilogue()
    e.out, e.ld_out, e.alpha = out.data_ptr(), 128, 1.0
    n0 = lib.otb_launch_count()
    rc = lib.otb_gemm_bf16(A.data_ptr(), 1, 128, B.data_ptr(), 0, 64, 128, 128, 64, C.byref(e), None)
    assert rc == 3 and b"not instantiated" in lib.otb_last_error()
    assert lib.otb_launch_count() == n0


@pytest.mark.gpu
@pytest.mark.parametrize("setting", SWITCHES)
def test_switch_configuration(setting):
    """This file again, in a child process whose otb_gemm_bf16 reads `setting` at its first call: the whole GPU matrix
    with that configuration's intended kernels.  The child does not start children of its own."""
    if os.environ.get(CHILD_ENV):
        pytest.skip("already a switch-configuration child")
    key, val = setting.split("=")
    env = dict(os.environ, **{key: val, CHILD_ENV: "1"})
    for other in SWITCHES:
        if other != setting:
            env.pop(other.split("=")[0], None)
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + \
        ["-m", "pytest", os.path.abspath(__file__), "-q", "-m", "gpu", "-p", "no:cacheprovider", "-x"]
    r = subprocess.run(cmd, cwd=ROOT, env=env, capture_output=True, text=True, timeout=900)
    tail = "\n".join((r.stdout + r.stderr).splitlines()[-40:])
    print(f"[gemm child {setting}]\n{tail}")
    assert r.returncode == 0, f"{setting}: child exited {r.returncode}\n{tail}"
    assert " passed" in tail and " failed" not in tail
