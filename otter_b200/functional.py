"""Thin torch-tensor wrappers over the C ABI (include/otter_b200.h).

PyTorch is plumbing only here: it owns device memory and the current CUDA stream; every arithmetic
operation on the hot path is a kernel of libotter_b200.so.  All activations are bf16, row-major with
unit column stride (row pitch may exceed the logical width so column slices work in place).
"""
import ctypes as C
import functools

import torch

from . import _lib
from ._lib import AttnDesc, AttnGrads, GemmEpilogue, LmAttnDesc, LmAttnGrads, check

BF16 = torch.bfloat16


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _device_of(args, kwargs):
    """Device index shared by every tensor argument (OtbError if they disagree); None if there is no tensor."""
    dev = None
    for a in (*args, *kwargs.values()):
        if isinstance(a, AttnSpec):
            a = a.q
        if isinstance(a, torch.Tensor) and a.is_cuda:
            i = a.device.index
            if dev is None:
                dev = i
            elif i != dev:
                raise _lib.OtbError(f"tensors live on different devices (cuda:{dev} and cuda:{i})")
    return dev


def _on_device(fn):
    """The C library launches on the CURRENT device and stream.  The reference places models with
    device_map="auto" (pipeline/demos/demo_models.py:37), so an op may be called with tensors of a non-current GPU:
    switch to the tensors' device for the duration of the call (the stream is then that device's current stream)."""
    @functools.wraps(fn)
    def wrapped(*args, **kwargs):
        dev = _device_of(args, kwargs)
        if dev is None or dev == torch.cuda.current_device():
            return fn(*args, **kwargs)
        with torch.cuda.device(dev):
            return fn(*args, **kwargs)
    return wrapped


def _p(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _req(t, dtype=None, name="tensor"):
    if not t.is_cuda:
        raise _lib.OtbError(f"{name} must be a CUDA tensor (otter_b200 has no CPU path)")
    if dtype is not None and t.dtype != dtype:
        raise _lib.OtbError(f"{name} must be {dtype}, got {t.dtype}")
    if t.dim() >= 1 and t.stride(-1) != 1:
        raise _lib.OtbError(f"{name} must have unit stride in its last dim")
    return t


def _mat(t, name="matrix", dtype=BF16):
    """2-D view [rows, cols] with unit column stride (leading dims flattened when contiguous)."""
    _req(t, dtype, name)
    if t.dim() == 2:
        return t
    return t.reshape(-1, t.shape[-1])


# ------------------------------------------------------------------------------------------------
# GEMM
# ------------------------------------------------------------------------------------------------
_GEMM_PROF = None


def set_gemm_profiler(sink):
    """bench.py: when `sink` is a list, every GEMM launch appends (2*M*N*K, start_event, end_event)."""
    global _GEMM_PROF
    _GEMM_PROF = sink


def _epi_mat(t, name, M, N, dtype):
    """Epilogue matrices are addressed as [M][N] with row pitch stride(0): anything else would be read or written
    outside its buffer, so it is rejected before the launch."""
    _req(t, dtype, name)
    if t.dim() != 2 or tuple(t.shape) != (M, N):
        raise _lib.OtbError(f"otb_gemm_bf16: {name} must be ({M}, {N}), got {tuple(t.shape)}")


def _gemm_raw(A, a_mn, lda, B, b_mn, ldb, M, N, K, out, *, bias=None, act=0, aux_out=None, aux_in=None,
              scale_ptr=None, scale_tanh=False, alpha=1.0, residual=None, accumulate=False, res_fp32=False):
    if out.dtype not in (BF16, torch.float32):
        raise _lib.OtbError(f"otb_gemm_bf16: out must be bf16 or fp32, got {out.dtype}")
    _epi_mat(out, "out", M, N, out.dtype)
    if bias is not None:
        _req(bias, torch.float32, "bias")
        if bias.numel() != N or not bias.is_contiguous():
            raise _lib.OtbError(f"otb_gemm_bf16: bias must be {N} contiguous fp32 values, got {tuple(bias.shape)}")
    if residual is not None:
        _epi_mat(residual, "residual", M, N, torch.float32 if res_fp32 else BF16)
    if aux_in is not None:
        _epi_mat(aux_in, "aux_in", M, N, BF16)
    if aux_out is not None:
        _epi_mat(aux_out, "aux_out", M, N, BF16)
    lib = _lib.load()
    e = GemmEpilogue()
    e.bias = _p(bias)
    e.aux_in = _p(aux_in)
    e.aux_out = _p(aux_out)
    e.scale_ptr = _p(scale_ptr)
    e.residual = _p(residual)
    e.out = _p(out)
    e.ld_out = out.stride(0)
    e.ld_aux_in = aux_in.stride(0) if aux_in is not None else 0
    e.ld_aux_out = aux_out.stride(0) if aux_out is not None else 0
    e.ld_res = residual.stride(0) if residual is not None else 0
    e.act = act
    e.scale_tanh = 1 if scale_tanh else 0
    e.out_fp32 = 1 if out.dtype == torch.float32 else 0
    e.accumulate = 1 if accumulate else 0
    e.alpha = alpha
    e.res_fp32 = 1 if res_fp32 else 0
    if _GEMM_PROF is not None:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
    check(lib.otb_gemm_bf16(_p(A), int(a_mn), lda, _p(B), int(b_mn), ldb, M, N, K, C.byref(e), _stream()),
          "otb_gemm_bf16")
    if _GEMM_PROF is not None:
        e1.record()
        _GEMM_PROF.append((2.0 * M * N * K, e0, e1, (M, N, K, int(a_mn), int(b_mn))))
    return out


@_on_device
def linear_fwd(x, w, *, out=None, out_dtype=BF16, **epi):
    """y[M,N] = epilogue(x[M,K] @ w[N,K]^T)   (nn.Linear forward)."""
    x, w = _mat(x, "x"), _mat(w, "w")
    M, K = x.shape
    N = w.shape[0]
    assert w.shape[1] == K, (x.shape, w.shape)
    if out is None:
        out = torch.empty((M, N), device=x.device, dtype=out_dtype)
    if epi.get("bias") is not None:
        _req(epi["bias"], torch.float32, "bias")
    return _gemm_raw(x, 0, x.stride(0), w, 0, w.stride(0), M, N, K, out, **epi)


@_on_device
def linear_dgrad(dy, w, *, out=None, out_dtype=BF16, **epi):
    """dx[M,K] = epilogue(dy[M,N] @ w[N,K])   — w is consumed MN-major in place (no transpose copy)."""
    dy, w = _mat(dy, "dy"), _mat(w, "w")
    M, N = dy.shape
    K = w.shape[1]
    assert w.shape[0] == N, (dy.shape, w.shape)
    if out is None:
        out = torch.empty((M, K), device=dy.device, dtype=out_dtype)
    return _gemm_raw(dy, 0, dy.stride(0), w, 1, w.stride(0), M, K, N, out, **epi)


@_on_device
def linear_wgrad(dy, x, *, out=None, accumulate=False, **epi):
    """dW[N,K] (fp32) (+)= dy[M,N]^T @ x[M,K]   — both operands consumed MN-major in place."""
    dy, x = _mat(dy, "dy"), _mat(x, "x")
    M, N = dy.shape
    K = x.shape[1]
    assert x.shape[0] == M, (dy.shape, x.shape)
    if out is None:
        out = torch.empty((N, K), device=dy.device, dtype=torch.float32)
        accumulate = False
    return _gemm_raw(dy, 1, dy.stride(0), x, 1, x.stride(0), N, K, M, out, accumulate=accumulate, **epi)


# ------------------------------------------------------------------------------------------------
# Causal self-attention of the frozen LM layers (head dim 128) — SURVEY.md §8f rank 1
# ------------------------------------------------------------------------------------------------
def _lm_desc(qkv, out, lse, slopes, B, S, H, causal, scale):
    d = LmAttnDesc()
    d.qkv, d.out, d.lse, d.alibi_slopes = _p(qkv), _p(out), _p(lse), _p(slopes)
    d.ld_qkv, d.ld_out = qkv.stride(0), out.stride(0)
    D = H * 128
    d.qkv_cols, d.q_col0, d.k_col0, d.v_col0, d.out_col0 = qkv.shape[1], 0, D, 2 * D, 0
    d.B, d.H, d.S, d.head_dim, d.causal = B, H, S, 128, 1 if causal else 0
    d.scale = scale
    return d


@_on_device
def lm_attn_fwd(qkv, B, S, H, *, slopes=None, causal=True, scale=None):
    """qkv bf16 [B*S, 3*H*128] (fused Wqkv output, [q|k|v]) -> (out bf16 [B*S, H*128], lse fp32 [B, H, S])."""
    qkv = _mat(qkv, "qkv")
    assert qkv.shape == (B * S, 3 * H * 128), qkv.shape
    if slopes is not None:
        _req(slopes, torch.float32, "alibi slopes")
    out = torch.empty((B * S, H * 128), device=qkv.device, dtype=BF16)
    lse = torch.empty((B, H, S), device=qkv.device, dtype=torch.float32)
    scale = (128 ** -0.5) if scale is None else scale
    d = _lm_desc(qkv, out, lse, slopes, B, S, H, causal, scale)
    check(_lib.load().otb_lm_attn_fwd(C.byref(d), _stream()), "otb_lm_attn_fwd")
    return out, lse


@_on_device
def lm_attn_bwd(dout, qkv, out, lse, B, S, H, *, slopes=None, causal=True, scale=None):
    """-> dqkv bf16 [B*S, 3*H*128] ([dq|dk|dv], the layout of qkv)."""
    dout, qkv, out = _mat(dout, "dout"), _mat(qkv, "qkv"), _mat(out, "out")
    scale = (128 ** -0.5) if scale is None else scale
    d = _lm_desc(qkv, out, lse, slopes, B, S, H, causal, scale)
    dqkv = torch.empty_like(qkv)
    g = LmAttnGrads()
    ws = torch.empty((B * S, H * 128), device=qkv.device, dtype=torch.float32) if S > 128 else None
    D = H * 128
    g.dout, g.dqkv, g.dq_ws = _p(dout), _p(dqkv), _p(ws)
    g.ld_dout, g.ld_dqkv = dout.stride(0), dqkv.stride(0)
    g.dout_cols, g.dout_col0, g.dq_col0, g.dk_col0, g.dv_col0 = dout.shape[1], 0, 0, D, 2 * D
    check(_lib.load().otb_lm_attn_bwd(C.byref(d), C.byref(g), _stream()), "otb_lm_attn_bwd")
    return dqkv


# ------------------------------------------------------------------------------------------------
# LayerNorm
# ------------------------------------------------------------------------------------------------
@_on_device
def layernorm_fwd(x, gamma, beta, eps=1e-5, want_stats=True, out=None):
    x2 = _mat(x, "x")
    _req(gamma, torch.float32, "gamma"), _req(beta, torch.float32, "beta")
    rows, D = x2.shape
    y = out if out is not None else torch.empty((rows, D), device=x.device, dtype=BF16)
    assert y.shape == (rows, D) and y.stride(1) == 1
    mean = torch.empty(rows, device=x.device, dtype=torch.float32) if want_stats else None
    rstd = torch.empty(rows, device=x.device, dtype=torch.float32) if want_stats else None
    check(_lib.load().otb_layernorm_fwd(_p(x2), x2.stride(0), _p(gamma), _p(beta), _p(y), y.stride(0), _p(mean),
                                        _p(rstd), rows, D, eps, _stream()), "otb_layernorm_fwd")
    return (y if out is not None else y.view(x.shape)), mean, rstd


@_on_device
def layernorm_bwd(dy, x, mean, rstd, gamma, *, add=None, want_dx=True, dgamma=None, dbeta=None, accumulate=False,
                  want_param_grads=True):
    """Returns (dx or None, dgamma, dbeta). `add` (bf16, same shape) is summed into dx (fused residual grad)."""
    lib = _lib.load()
    dy2, x2 = _mat(dy, "dy"), _mat(x, "x")
    rows, D = x2.shape
    dx = torch.empty((rows, D), device=x.device, dtype=BF16) if want_dx else None
    add2 = _mat(add, "add") if add is not None else None
    ws = None
    if want_param_grads:
        if dgamma is None:
            dgamma = torch.empty(D, device=x.device, dtype=torch.float32)
            dbeta = torch.empty(D, device=x.device, dtype=torch.float32)
            accumulate = False
        ws = torch.empty(2 * lib.otb_ln_chunks(rows, D) * D, device=x.device, dtype=torch.float32)
    else:
        dgamma = dbeta = None
    check(lib.otb_layernorm_bwd(_p(dy2), dy2.stride(0), _p(x2), x2.stride(0), _p(mean), _p(rstd), _p(gamma),
                                _p(add2), add2.stride(0) if add2 is not None else 0, _p(dx),
                                dx.stride(0) if dx is not None else 0, _p(dgamma), _p(dbeta), int(accumulate), _p(ws),
                                rows, D, _stream()), "otb_layernorm_bwd")
    return (dx.view(x.shape) if dx is not None else None), dgamma, dbeta


# ------------------------------------------------------------------------------------------------
# attention
# ------------------------------------------------------------------------------------------------
class AttnSpec:
    """Where Q / K / V / O live inside their 2-D buffers (see otb_attn_desc)."""

    def __init__(self, q, q_col0, kv1, k1_col0, v1_col0, P, H, Sq, Sk1, scale, kv2=None, k2_col0=0, v2_col0=0, Sk2=0,
                 text_time=None, n_per_media=0, T_img=0, dtype=BF16, mask_ge=False, causal=False):
        self.q, self.q_col0 = _mat(q, "q", dtype), q_col0
        self.kv1, self.k1_col0, self.v1_col0 = _mat(kv1, "kv1", dtype), k1_col0, v1_col0
        self.kv2 = _mat(kv2, "kv2", dtype) if kv2 is not None else None
        self.k2_col0, self.v2_col0 = k2_col0, v2_col0
        self.P, self.H, self.Sq, self.Sk1, self.Sk2, self.scale = P, H, Sq, Sk1, Sk2, scale
        self.text_time, self.n_per_media, self.T_img = text_time, n_per_media, T_img
        self.mask_ge, self.causal = bool(mask_ge), bool(causal)
        assert self.q.shape[0] == P * Sq and self.kv1.shape[0] == P * Sk1
        if text_time is not None:
            _req(text_time, torch.int32, "text_time")
            assert text_time.numel() == P * Sq

    def desc(self, out, out_col0, lse):
        d = AttnDesc()
        d.q, d.kv1, d.kv2, d.out, d.lse = _p(self.q), _p(self.kv1), _p(self.kv2), _p(out), _p(lse)
        d.text_time = _p(self.text_time)
        d.ldq, d.ldkv1 = self.q.stride(0), self.kv1.stride(0)
        d.ldkv2 = self.kv2.stride(0) if self.kv2 is not None else 0
        d.ld_out = out.stride(0)
        d.q_cols, d.kv1_cols = self.q.shape[1], self.kv1.shape[1]
        d.kv2_cols = self.kv2.shape[1] if self.kv2 is not None else 0
        d.q_col0, d.k1_col0, d.v1_col0 = self.q_col0, self.k1_col0, self.v1_col0
        d.k2_col0, d.v2_col0, d.out_col0 = self.k2_col0, self.v2_col0, out_col0
        d.n_per_media, d.T_img = self.n_per_media, self.T_img
        d.P, d.H, d.Sq, d.Sk1, d.Sk2, d.head_dim = self.P, self.H, self.Sq, self.Sk1, self.Sk2, 64
        d.scale = self.scale
        d.mask_ge, d.causal = int(self.mask_ge), int(self.causal)
        return d


@_on_device
def attn_fwd(spec, out=None, out_col0=0, want_lse=True):
    if out is None:
        out = torch.empty((spec.P * spec.Sq, spec.H * 64), device=spec.q.device, dtype=BF16)
    lse = torch.empty((spec.P, spec.H, spec.Sq), device=spec.q.device, dtype=torch.float32) if want_lse else None
    d = spec.desc(out, out_col0, lse)
    check(_lib.load().otb_attn_fwd(C.byref(d), _stream()), "otb_attn_fwd")
    return out, lse


@_on_device
def attn_bwd(spec, out, out_col0, lse, dout, dout_col0, dq, dq_col0, dkv1, dk1_col0, dv1_col0, dkv2=None, dk2_col0=0,
             dv2_col0=0):
    d = spec.desc(out, out_col0, lse)
    g = AttnGrads()
    dout = _mat(dout, "dout")
    g.dout, g.dq, g.dkv1, g.dkv2 = _p(dout), _p(dq), _p(dkv1), _p(dkv2)
    nkt = (spec.Sk1 + 127) // 128 + (spec.Sk2 + 127) // 128
    ws = torch.empty((spec.P * spec.Sq, spec.H * 64), device=dout.device, dtype=torch.float32) if nkt > 1 else None
    g.dq_ws = _p(ws)
    g.ld_dout, g.ld_dq, g.ld_dkv1 = dout.stride(0), dq.stride(0), dkv1.stride(0)
    g.ld_dkv2 = dkv2.stride(0) if dkv2 is not None else 0
    g.dout_cols, g.dout_col0, g.dq_col0 = dout.shape[1], dout_col0, dq_col0
    g.dk1_col0, g.dv1_col0, g.dk2_col0, g.dv2_col0 = dk1_col0, dv1_col0, dk2_col0, dv2_col0
    check(_lib.load().otb_attn_bwd(C.byref(d), C.byref(g), _stream()), "otb_attn_bwd")
    return dq, dkv1, dkv2


def xattn_out_fusable(spec, D):
    """The single fused kernel covers the training layout: one key source with T_img * n <= 64 keys, <= 8 heads."""
    return spec.kv2 is None and spec.Sk1 <= 64 and spec.H <= 8 and D % 512 == 0 and not spec.causal


@_on_device
def xattn_out_fused(spec, wo, gate, residual, want_aux=True, want_lse=True):
    """-> (y, aux, o, lse): y = (attn(spec) @ wo^T) * tanh(gate) + residual in ONE kernel (otb_xattn_out_fused)."""
    wo, residual = _mat(wo, "wo"), _mat(residual, "residual")
    D = wo.shape[0]
    rows = spec.P * spec.Sq
    assert wo.shape[1] == spec.H * 64 and residual.shape == (rows, D)
    o = torch.empty((rows, spec.H * 64), device=wo.device, dtype=BF16)
    lse = torch.empty((spec.P, spec.H, spec.Sq), device=wo.device, dtype=torch.float32) if want_lse else None
    y = torch.empty((rows, D), device=wo.device, dtype=BF16)
    aux = torch.empty((rows, D), device=wo.device, dtype=BF16) if want_aux else None
    d = spec.desc(o, 0, lse)
    check(_lib.load().otb_xattn_out_fused(C.byref(d), _p(wo), wo.stride(0), _p(_req(gate, torch.float32, "gate")),
                                          _p(residual), residual.stride(0), _p(aux), aux.stride(0) if aux is not None else D,
                                          _p(y), y.stride(0), D, _stream()), "otb_xattn_out_fused")
    return y, aux, o, lse


@_on_device
def text_time(media_locations, attend_previous=True):
    """bool/uint8 [B,L] -> int32 [B,L]  (bit-exact restatement of modeling_otter.py:298-311)."""
    ml = media_locations
    if ml.dtype == torch.bool:
        ml = ml.view(torch.uint8) if ml.is_contiguous() else ml.contiguous().view(torch.uint8)
    _req(ml, torch.uint8, "media_locations")
    ml = ml.contiguous()
    B, L = ml.shape
    out = torch.empty((B, L), device=ml.device, dtype=torch.int32)
    check(_lib.load().otb_text_time(_p(ml), B, L, int(bool(attend_previous)), _p(out), _stream()), "otb_text_time")
    return out


# ------------------------------------------------------------------------------------------------
# small passes
# ------------------------------------------------------------------------------------------------
@_on_device
def cast_bf16(src, out=None):
    _req(src, torch.float32, "src")
    src = src.contiguous()
    if out is None:
        out = torch.empty(src.shape, device=src.device, dtype=BF16)
    check(_lib.load().otb_cast_f32_bf16(_p(src), _p(out), src.numel(), _stream()), "otb_cast_f32_bf16")
    return out


CAST_MULTI_BLOCK = 4096      # elements per block of otb_cast_f32_bf16_multi (kCastSegElems)


@_on_device
def cast_bf16_multi(table, n_tensors, total_blocks):
    """table: int64 [n_tensors, 4] on the device = {src ptr, dst ptr, numel, first block} per tensor."""
    assert table.dtype == torch.int64 and table.is_contiguous() and table.shape == (n_tensors, 4)
    check(_lib.load().otb_cast_f32_bf16_multi(_p(table), n_tensors, total_blocks, _stream()), "otb_cast_f32_bf16_multi")


@_on_device
def cast_f32(src, out=None):
    _req(src, BF16, "src")
    src = src.contiguous()
    if out is None:
        out = torch.empty(src.shape, device=src.device, dtype=torch.float32)
    check(_lib.load().otb_cast_bf16_f32(_p(src), _p(out), src.numel(), _stream()), "otb_cast_bf16_f32")
    return out


@_on_device
def cast_f32_scaled(src, out, scale):
    """out fp32 = float(src bf16) * scale (flat buffers)."""
    _req(src, BF16, "src")
    _req(out, torch.float32, "out")
    assert src.is_contiguous() and out.is_contiguous() and src.numel() == out.numel()
    check(_lib.load().otb_cast_bf16_f32_scale(_p(src), _p(out), src.numel(), float(scale), _stream()), "otb_cast_bf16_f32_scale")
    return out


@_on_device
def bcast_rows(src, rows, div, mod):
    _req(src, torch.float32, "src")
    D = src.shape[-1]
    out = torch.empty((rows, D), device=src.device, dtype=BF16)
    check(_lib.load().otb_bcast_rows(_p(src), div, mod, _p(out), rows, D, _stream()), "otb_bcast_rows")
    return out


@_on_device
def add_rowbias(x, bias, div, mod):
    x2 = _mat(x, "x")
    assert x2.is_contiguous()
    rows, D = x2.shape
    out = torch.empty_like(x2)
    check(_lib.load().otb_add_rowbias(_p(x2), _p(_req(bias, torch.float32, "bias")), div, mod, _p(out), rows, D,
                                      _stream()), "otb_add_rowbias")
    return out


@_on_device
def grouped_colsum(x, div, mod, out=None, accumulate=False):
    x2 = _mat(x, "x")
    rows, D = x2.shape
    if out is None:
        out = torch.empty((mod, D), device=x.device, dtype=torch.float32)
        accumulate = False
    check(_lib.load().otb_grouped_colsum(_p(x2), x2.stride(0), rows, D, div, mod, _p(out), int(accumulate), _stream()),
          "otb_grouped_colsum")
    return out


@_on_device
def gate_grad(dy, a, gate, dgate=None, accumulate=False):
    lib = _lib.load()
    _req(dy, BF16, "dy"), _req(a, BF16, "a"), _req(gate, torch.float32, "gate")
    assert dy.is_contiguous() and a.is_contiguous() and dy.numel() == a.numel()
    if dgate is None:
        dgate = torch.empty(1, device=dy.device, dtype=torch.float32)
        accumulate = False
    ws = torch.empty(lib.otb_dot_blocks(), device=dy.device, dtype=torch.float32)
    check(lib.otb_gate_grad(_p(dy), _p(a), dy.numel(), _p(gate), _p(dgate), int(accumulate), _p(ws), _stream()),
          "otb_gate_grad")
    return dgate


@_on_device
def sqmean_loss(x, want_grad=True):
    lib = _lib.load()
    _req(x, BF16, "x")
    assert x.is_contiguous()
    loss = torch.empty(1, device=x.device, dtype=torch.float32)
    dx = torch.empty_like(x) if want_grad else None
    ws = torch.empty(lib.otb_dot_blocks(), device=x.device, dtype=torch.float32)
    check(lib.otb_sqmean_loss(_p(x), x.numel(), _p(loss), _p(dx), _p(ws), _stream()), "otb_sqmean_loss")
    return loss, dx


@_on_device
def im2col_patches(pixels, patch, Kpad):
    assert pixels.is_cuda and pixels.dim() == 4 and pixels.shape[1] == 3
    pixels = pixels.contiguous()
    if pixels.dtype not in (torch.float32, BF16):
        pixels = pixels.float()
    N, _, H, W = pixels.shape
    out = torch.empty((N * (H // patch) * (W // patch), Kpad), device=pixels.device, dtype=BF16)
    check(_lib.load().otb_im2col_patches(_p(pixels), int(pixels.dtype == torch.float32), N, H, W, patch, _p(out), Kpad,
                                         _stream()), "otb_im2col_patches")
    return out


@_on_device
def clip_assemble(patch_emb, cls, pos, N, np_):
    D = patch_emb.shape[-1]
    out = torch.empty((N, np_ + 1, D), device=patch_emb.device, dtype=BF16)
    check(_lib.load().otb_clip_assemble(_p(_mat(patch_emb)), _p(_req(cls, torch.float32)), _p(_req(pos, torch.float32)),
                                        _p(out), N, np_, D, _stream()), "otb_clip_assemble")
    return out


@_on_device
def media_from_clip(hidden, frame_embs, F):
    """hidden bf16 [n_img, 1+v, D] -> bf16 [n_img*v, D] (CLS dropped, + frame_embs[img % F] if given)."""
    _req(hidden, BF16, "hidden")
    n_img, v1, D = hidden.shape
    out = torch.empty((n_img * (v1 - 1), D), device=hidden.device, dtype=BF16)
    check(_lib.load().otb_media_from_clip(_p(hidden.contiguous()), _p(frame_embs), F, _p(out), n_img, v1 - 1, D,
                                          _stream()), "otb_media_from_clip")
    return out


@_on_device
def fuyu_scatter(word, cont, idx, b_off):
    """b_off: int64 [B+1] prefix offsets of each sample's rows in `cont` (see otb_fuyu_scatter)."""
    _req(word, BF16, "word"), _req(cont, BF16, "cont")
    B, S, D = word.shape
    if b_off.numel() != B + 1 or b_off.dtype != torch.int64 or idx.dtype != torch.int64:
        raise _lib.OtbError("fuyu_scatter: b_off must be int64 [B+1] and idx int64 [B,S]")
    out = torch.empty_like(word)
    check(_lib.load().otb_fuyu_scatter(_p(word.contiguous()), _p(cont.contiguous()), _p(idx.contiguous()),
                                       _p(b_off.contiguous()), _p(out), B, S, D, _stream()), "otb_fuyu_scatter")
    return out


# ------------------------------------------------------------------------------------------------
# LLaMA layer: RMSNorm, rotary embedding, SwiGLU (csrc/otb_llama.cu)
# ------------------------------------------------------------------------------------------------
@_on_device
def rmsnorm_fwd(x, weight, eps, want_rstd=True):
    x2 = _mat(x, "x")
    rows, D = x2.shape
    y = torch.empty((rows, D), device=x.device, dtype=BF16)
    rstd = torch.empty(rows, device=x.device, dtype=torch.float32) if want_rstd else None
    check(_lib.load().otb_rmsnorm_fwd(_p(x2), x2.stride(0), _p(_req(weight, torch.float32, "weight")), _p(y), y.stride(0),
                                      _p(rstd), rows, D, float(eps), _stream()), "otb_rmsnorm_fwd")
    return y, rstd


@_on_device
def rmsnorm_bwd(dy, x, rstd, weight, add=None):
    dy2, x2 = _mat(dy, "dy"), _mat(x, "x")
    rows, D = x2.shape
    dx = torch.empty((rows, D), device=x.device, dtype=BF16)
    add2 = _mat(add, "add") if add is not None else None
    check(_lib.load().otb_rmsnorm_bwd(_p(dy2), dy2.stride(0), _p(x2), x2.stride(0), _p(rstd), _p(weight), _p(add2),
                                      add2.stride(0) if add2 is not None else 0, _p(dx), dx.stride(0), rows, D, _stream()),
          "otb_rmsnorm_bwd")
    return dx


@_on_device
def rope128_(buf, H, S, nblk, rope_theta, backward=False):
    """In place: rotary embedding (rotate_half convention) on the first `nblk` blocks of H x 128 columns of buf."""
    buf = _mat(buf, "buf")
    check(_lib.load().otb_rope128(_p(buf), buf.stride(0), buf.shape[0], H, S, nblk, float(rope_theta), int(bool(backward)),
                                  _stream()), "otb_rope128")
    return buf


@_on_device
def swiglu_fwd(g, u):
    g, u = _mat(g, "g"), _mat(u, "u")
    rows, I = g.shape
    h = torch.empty((rows, I), device=g.device, dtype=BF16)
    check(_lib.load().otb_swiglu_fwd(_p(g), g.stride(0), _p(u), u.stride(0), _p(h), h.stride(0), rows, I, _stream()),
          "otb_swiglu_fwd")
    return h


@_on_device
def swiglu_bwd(dh, g, u):
    dh, g, u = _mat(dh, "dh"), _mat(g, "g"), _mat(u, "u")
    rows, I = g.shape
    dg, du = torch.empty((rows, I), device=g.device, dtype=BF16), torch.empty((rows, I), device=g.device, dtype=BF16)
    check(_lib.load().otb_swiglu_bwd(_p(dh), dh.stride(0), _p(g), g.stride(0), _p(u), u.stride(0), _p(dg), dg.stride(0),
                                     _p(du), du.stride(0), rows, I, _stream()), "otb_swiglu_bwd")
    return dg, du


# ------------------------------------------------------------------------------------------------
# Persimmon / Fuyu layer: split + qk-LayerNorm + partial RoPE (csrc/otb_persimmon.cu)
# ------------------------------------------------------------------------------------------------
@_on_device
def qkln_rope_fwd(fused, H, S, q_gamma, q_beta, k_gamma, k_beta, rotary_dims, rope_theta, eps=1e-5):
    """fused bf16 [rows, H*3*64] -> (qkv bf16 [rows, 3*H*64] as q | k | v blocks, stats fp32 [rows, H, 4])."""
    fused = _mat(fused, "fused")
    rows = fused.shape[0]
    assert fused.shape[1] == H * 192, fused.shape
    qkv = torch.empty((rows, 3 * H * 64), device=fused.device, dtype=BF16)
    stats = torch.empty((rows, H, 4), device=fused.device, dtype=torch.float32)
    check(_lib.load().otb_qkln_rope_fwd(_p(fused), fused.stride(0), _p(_req(q_gamma, torch.float32)),
                                        _p(_req(q_beta, torch.float32)), _p(_req(k_gamma, torch.float32)),
                                        _p(_req(k_beta, torch.float32)), _p(qkv), qkv.stride(0), _p(stats), rows, H, S,
                                        int(rotary_dims), float(rope_theta), float(eps), _stream()), "otb_qkln_rope_fwd")
    return qkv, stats


@_on_device
def qkln_rope_bwd(dqkv, fused, stats, H, S, q_gamma, k_gamma, rotary_dims, rope_theta, dq_gamma, dq_beta, dk_gamma,
                  dk_beta, accumulate=False):
    """-> dfused bf16 [rows, H*3*64]; the four fp32 [64] parameter gradients are written / accumulated in place."""
    lib = _lib.load()
    dqkv, fused = _mat(dqkv, "dqkv"), _mat(fused, "fused")
    rows = fused.shape[0]
    dfused = torch.empty_like(fused)
    ws = torch.empty(lib.otb_qkln_rope_ws_floats(), device=fused.device, dtype=torch.float32)
    check(lib.otb_qkln_rope_bwd(_p(dqkv), dqkv.stride(0), _p(fused), fused.stride(0), _p(stats), _p(q_gamma), _p(k_gamma),
                                _p(dfused), dfused.stride(0), _p(dq_gamma), _p(dq_beta), _p(dk_gamma), _p(dk_beta),
                                int(bool(accumulate)), _p(ws), rows, H, S, int(rotary_dims), float(rope_theta), _stream()),
          "otb_qkln_rope_bwd")
    return dfused


# ------------------------------------------------------------------------------------------------
# fp32-grade forward path (parity mode; csrc/otb_fp32.cu)
# ------------------------------------------------------------------------------------------------
F32_KCHUNK = 512


@_on_device
def epilogue_f32(acc, *, bias=None, act=0, scale_ptr=None, scale_tanh=False, residual=None):
    """fp32 epilogue of the chunked fp32-grade GEMM: act(acc + bias) * gate + residual (otb_epilogue_f32)."""
    acc = _mat(acc, "acc", torch.float32)
    M, N = acc.shape
    out = torch.empty_like(acc)
    check(_lib.load().otb_epilogue_f32(_p(acc), _p(bias), act, _p(scale_ptr), int(bool(scale_tanh)), _p(residual),
                                       _p(out), M, N, _stream()), "otb_epilogue_f32")
    return out


@_on_device
def split3_concat(src, pattern):
    """fp32 [rows, K] -> bf16 [rows, 6K]: three-term bf16 split laid out for the 6-product GEMM."""
    src = _mat(src, "src", torch.float32)
    rows, K = src.shape
    out = torch.empty((rows, 6 * K), device=src.device, dtype=BF16)
    check(_lib.load().otb_split3_concat(_p(src), src.stride(0), rows, K, pattern, _p(out), _stream()), "otb_split3_concat")
    return out


@_on_device
def linear_f32(x, w6, N, *, bias=None, act=0, scale_ptr=None, scale_tanh=False, residual=None):
    """y fp32 [M,N] = epilogue(x fp32 [M,K] @ W^T) with fp32-grade accuracy; w6 = split3_concat(W, 1)."""
    x = _mat(x, "x", torch.float32)
    M, K = x.shape
    assert w6.shape == (N, 6 * K), (w6.shape, N, K)
    a6 = split3_concat(x, 0)
    out = torch.empty((M, N), device=x.device, dtype=torch.float32)
    if residual is not None:
        residual = _mat(residual, "residual", torch.float32)
    # The tensor core adds into its fp32 accumulator with truncation, so a long in-TMEM reduction drifts by
    # ~(#MMA steps) * 2^-24 of the running sum.  Keep each in-TMEM run short (F32_KCHUNK columns of K') and
    # carry the running sum in fp32 through the epilogue's round-to-nearest accumulate instead.
    K6, kc = 6 * K, F32_KCHUNK
    if K6 <= kc:
        return _gemm_raw(a6, 0, a6.stride(0), w6, 0, w6.stride(0), M, N, K6, out, bias=bias, act=act,
                         scale_ptr=scale_ptr, scale_tanh=scale_tanh, residual=residual, res_fp32=residual is not None)
    nchunk = (K6 + kc - 1) // kc
    for i in range(nchunk):
        k0, k1 = i * kc, min(K6, (i + 1) * kc)
        _gemm_raw(a6[:, k0:k1], 0, a6.stride(0), w6[:, k0:k1], 0, w6.stride(0), M, N, k1 - k0, out,
                  accumulate=(i > 0))
    if bias is not None or act or scale_ptr is not None or residual is not None:
        out = epilogue_f32(out, bias=bias, act=act, scale_ptr=scale_ptr, scale_tanh=scale_tanh, residual=residual)
    return out


@_on_device
def layernorm_fwd_f32(x, gamma, beta, eps=1e-5):
    x2 = _mat(x, "x", torch.float32)
    rows, D = x2.shape
    y = torch.empty((rows, D), device=x.device, dtype=torch.float32)
    check(_lib.load().otb_layernorm_fwd_f32(_p(x2), x2.stride(0), _p(_req(gamma, torch.float32)),
                                            _p(_req(beta, torch.float32)), _p(y), y.stride(0), rows, D, eps, _stream()),
          "otb_layernorm_fwd_f32")
    return y.view(x.shape)


@_on_device
def add_rowbias_f32(x, bias, div, mod):
    x2 = _mat(x, "x", torch.float32)
    assert x2.is_contiguous()
    rows, D = x2.shape
    out = torch.empty_like(x2)
    check(_lib.load().otb_add_rowbias_f32(_p(x2), _p(_req(bias, torch.float32)), div, mod, _p(out), rows, D, _stream()),
          "otb_add_rowbias_f32")
    return out


@_on_device
def attn_fwd_f32(spec):
    """spec: AttnSpec(dtype=torch.float32) -> fp32 [P*Sq, H*64]."""
    out = torch.empty((spec.P * spec.Sq, spec.H * 64), device=spec.q.device, dtype=torch.float32)
    d = spec.desc(out, 0, None)
    check(_lib.load().otb_attn_fwd_f32(C.byref(d), _stream()), "otb_attn_fwd_f32")
    return out


# ---- fp32-grade backward passes (csrc/otb_fp32_bwd.cu) ----
@_on_device
def layernorm_bwd_f32(dy, x, gamma, eps=1e-5, need_dx=True, need_params=True):
    dy2, x2 = _mat(dy, "dy", torch.float32), _mat(x, "x", torch.float32)
    rows, D = x2.shape
    dx = torch.empty((rows, D), device=x.device, dtype=torch.float32) if need_dx else None
    dg = torch.empty(D, device=x.device, dtype=torch.float32) if need_params else None
    db = torch.empty(D, device=x.device, dtype=torch.float32) if need_params else None
    ws = torch.empty(2 * rows, device=x.device, dtype=torch.float32)
    check(_lib.load().otb_layernorm_bwd_f32(_p(dy2), dy2.stride(0), _p(x2), x2.stride(0), _p(_req(gamma, torch.float32)),
                                            _p(dx), D, _p(dg), _p(db), _p(ws), rows, D, eps, _stream()),
          "otb_layernorm_bwd_f32")
    return dx, dg, db


@_on_device
def act_bwd_f32(dy, pre, act):
    dy, pre = _req(dy, torch.float32, "dy").contiguous(), _req(pre, torch.float32, "pre").contiguous()
    out = torch.empty_like(pre)
    check(_lib.load().otb_act_bwd_f32(_p(dy), _p(pre), act, _p(out), pre.numel(), _stream()), "otb_act_bwd_f32")
    return out


@_on_device
def gate_grad_f32(dy, f, gate):
    dy, f = _req(dy, torch.float32, "dy").contiguous(), _req(f, torch.float32, "f").contiguous()
    out = torch.empty(1, device=dy.device, dtype=torch.float32)
    check(_lib.load().otb_gate_grad_f32(_p(dy), _p(f), f.numel(), _p(_req(gate, torch.float32)), _p(out), _stream()),
          "otb_gate_grad_f32")
    return out


@_on_device
def rowbias_grad_f32(dy, div, mod, out_rows):
    dy2 = _mat(dy, "dy", torch.float32)
    assert dy2.is_contiguous()
    rows, D = dy2.shape
    out = torch.empty((out_rows, D), device=dy.device, dtype=torch.float32)
    check(_lib.load().otb_rowbias_grad_f32(_p(dy2), div, mod, rows, D, out_rows, _p(out), _stream()), "otb_rowbias_grad_f32")
    return out


@_on_device
def attn_bwd_f32(spec, out, dout):
    """spec: AttnSpec(dtype=torch.float32) of the forward problem (K at column 0, V at column H*64 of each key source),
    out: its forward output -> (dq [P*Sq, H*64], dkv1 [P*Sk1, 2*H*64], dkv2 or None), all fp32."""
    inner = spec.H * 64
    dev = spec.q.device
    dout = _mat(dout, "dout", torch.float32)
    dq = torch.empty((spec.P * spec.Sq, inner), device=dev, dtype=torch.float32)
    dkv1 = torch.empty((spec.P * spec.Sk1, 2 * inner), device=dev, dtype=torch.float32)
    dkv2 = torch.empty((spec.P * spec.Sk2, 2 * inner), device=dev, dtype=torch.float32) if spec.Sk2 else None
    ws = torch.empty(spec.P * spec.H * spec.Sq * 3, device=dev, dtype=torch.float32)
    d = spec.desc(out, 0, None)
    g = AttnGrads()
    g.dout, g.dq, g.dkv1, g.dkv2, g.dq_ws = _p(dout), _p(dq), _p(dkv1), _p(dkv2), _p(ws)
    g.ld_dout, g.ld_dq, g.ld_dkv1 = dout.stride(0), dq.stride(0), dkv1.stride(0)
    g.ld_dkv2 = dkv2.stride(0) if dkv2 is not None else 0
    g.dout_cols, g.dout_col0, g.dq_col0 = dout.shape[1], 0, 0
    g.dk1_col0, g.dv1_col0, g.dk2_col0, g.dv2_col0 = 0, inner, 0, inner
    check(_lib.load().otb_attn_bwd_f32(C.byref(d), C.byref(g), _stream()), "otb_attn_bwd_f32")
    return dq, dkv1, dkv2


def launch_count():
    return int(_lib.load().otb_launch_count())
