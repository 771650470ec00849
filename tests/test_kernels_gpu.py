"""GPU parity tests of the individual kernels, called through the C ABI (ctypes).

Reference for each op = the same op in plain torch fp32 on the bf16-rounded inputs (a floating-point
kernel: tolerance written at each assert; integer/index outputs are compared bit-exact against the
numpy oracle).
"""
import math

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def dev():
    return torch.device("cuda:0")


def rnd(*shape, scale=1.0, seed=0):
    g = torch.Generator(device="cpu").manual_seed(seed + sum(shape))
    return (torch.randn(*shape, generator=g) * scale).to(dev()).to(torch.bfloat16)


def assert_close(got, ref, rtol, atol, what=""):
    got, ref = got.float(), ref.float()
    err = (got - ref).abs()
    tol = atol + rtol * ref.abs()
    bad = (err > tol).sum().item()
    assert bad == 0, f"{what}: {bad}/{err.numel()} outside tol, max err {err.max().item():.4e}, max ref {ref.abs().max().item():.3f}"


# The GEMM (otb_gemm_bf16) has its own parity suite against an fp64 reference: tests/test_gemm_gpu.py.


@pytest.mark.parametrize("rows,D", [(37, 256), (512, 1024), (300, 4096), (101, 3072), (2, 2048)])
def test_layernorm_fwd_bwd(rows, D):
    from otter_b200 import functional as F
    x = rnd(rows, D, scale=2.0)
    g = (1 + 0.1 * torch.randn(D)).to(dev())
    b = (0.1 * torch.randn(D)).to(dev())
    y, mean, rstd = F.layernorm_fwd(x, g, b)
    xr = x.float().requires_grad_(True)
    gr, br = g.clone().requires_grad_(True), b.clone().requires_grad_(True)
    yr = torch.nn.functional.layer_norm(xr, (D,), gr, br, 1e-5)
    assert_close(y, yr, 1e-2, 1e-2, "ln fwd")
    dy = rnd(rows, D, seed=3)
    add = rnd(rows, D, seed=4)
    yr.backward(dy.float())
    dx, dg, db = F.layernorm_bwd(dy, x, mean, rstd, g, add=add)
    assert_close(dx, xr.grad + add.float(), 1e-2, 2e-2, "ln dx")
    assert_close(dg, gr.grad, 1e-3, 1e-2 * math.sqrt(rows), "ln dgamma")
    assert_close(db, br.grad, 1e-3, 1e-2 * math.sqrt(rows), "ln dbeta")


def test_text_time_bit_exact():
    from oracle.restatement import text_time_np
    from otter_b200 import functional as F
    rng = np.random.RandomState(0)
    for L in (1, 7, 32, 257, 2048):
        loc = rng.rand(5, L) < 0.1
        loc[0, :] = False
        if L > 3:
            loc[1, 0] = True
        for ap in (True, False):
            got = F.text_time(torch.from_numpy(loc).to(dev()), ap).cpu().numpy()
            ref = text_time_np(loc, ap)
            assert got.dtype == np.int32 and np.array_equal(got.astype(np.int64), ref), (L, ap)


def _attn_ref(q, k, v, scale, tt=None, n=64, T=1):
    """fp32 reference of the attention core with the reference's mask semantics. q [P,H,Sq,64] etc."""
    sim = (q * scale) @ k.transpose(-1, -2)
    if tt is not None:
        media_time = torch.arange(T, device=q.device).repeat_interleave(n) + 1
        keep = tt[:, None, :, None] == media_time[None, None, None, :]
        sim = sim.masked_fill(~keep, -torch.finfo(sim.dtype).max)
    sim = sim - sim.amax(dim=-1, keepdim=True).detach()
    attn = sim.softmax(dim=-1)
    if tt is not None:
        attn = attn.masked_fill((tt == 0)[:, None, :, None], 0.0)
    return attn @ v


def _heads(t, P, S, H):
    return t.float().reshape(P, S, H, 64).permute(0, 2, 1, 3)


@pytest.mark.parametrize("P,H,Sq,Sk1,Sk2", [(2, 8, 64, 256, 64), (1, 2, 64, 96, 64), (3, 4, 257, 257, 0),
                                             (2, 2, 64, 2048, 64), (2, 8, 300, 64, 0),
                                             # >= 119 (problem, head) pairs: one CTA walks ALL query tiles with K/V resident
                                             (8, 16, 257, 257, 0), (16, 8, 300, 64, 0), (15, 8, 700, 130, 64)])
def test_attention_fwd_bwd_unmasked(P, H, Sq, Sk1, Sk2):
    from otter_b200 import functional as F
    inner = H * 64
    q = rnd(P * Sq, inner, seed=1)
    kv1 = rnd(P * Sk1, 2 * inner, seed=2)
    kv2 = rnd(P * Sk2, 2 * inner, seed=3) if Sk2 else None
    spec = F.AttnSpec(q, 0, kv1, 0, inner, P, H, Sq, Sk1, 0.125, kv2=kv2, k2_col0=0, v2_col0=inner, Sk2=Sk2)
    out, lse = F.attn_fwd(spec)
    qr = q.float().requires_grad_(True)
    k1r = kv1.float().requires_grad_(True)
    k2r = kv2.float().requires_grad_(True) if Sk2 else None
    kk = _heads(k1r[:, :inner], P, Sk1, H)
    vv = _heads(k1r[:, inner:], P, Sk1, H)
    if Sk2:
        kk = torch.cat([kk, _heads(k2r[:, :inner], P, Sk2, H)], dim=2)
        vv = torch.cat([vv, _heads(k2r[:, inner:], P, Sk2, H)], dim=2)
    ref = _attn_ref(_heads(qr, P, Sq, H), kk, vv, 0.125).permute(0, 2, 1, 3).reshape(P * Sq, inner)
    assert_close(out, ref, 2e-2, 2e-2, "attn fwd")
    dout = rnd(P * Sq, inner, seed=5)
    ref.backward(dout.float())
    dq = torch.zeros_like(q)
    dkv1 = torch.zeros_like(kv1)
    dkv2 = torch.zeros_like(kv2) if Sk2 else None
    F.attn_bwd(spec, out, 0, lse, dout, 0, dq, 0, dkv1, 0, inner, dkv2, 0, inner)
    sc = max(1.0, math.sqrt(Sq / 64))
    assert_close(dq, qr.grad, 3e-2, 3e-2, "attn dq")
    assert_close(dkv1, k1r.grad, 3e-2, 3e-2 * sc, "attn dkv1")
    if Sk2:
        assert_close(dkv2, k2r.grad, 3e-2, 3e-2 * sc, "attn dkv2")


@pytest.mark.parametrize("T,L,pos,attend_previous", [
    (1, 256, [[0], [5]], True),
    (2, 160, [[0, 40], [3, 90]], True),
    (1, 64, [[0, 8, 16], [2, 9]], True),          # more <image> tokens than media -> uniform rows
    (3, 300, [[0, 100, 200], [10, 20, 290]], False),
    (2, 40, [[], [7]], True),                      # a sample without any <image>
])
def test_attention_media_mask(T, L, pos, attend_previous):
    from oracle.restatement import text_time_np
    from otter_b200 import functional as F
    P, H, n = 2, 8, 64
    inner = H * 64
    loc = np.zeros((P, L), dtype=bool)
    for b, ps in enumerate(pos):
        loc[b, ps] = True
    tt = F.text_time(torch.from_numpy(loc).to(dev()), attend_previous)
    assert np.array_equal(tt.cpu().numpy().astype(np.int64), text_time_np(loc, attend_previous))
    q = rnd(P * L, inner, seed=1)
    kv = rnd(P * T * n, 2 * inner, seed=2)
    spec = F.AttnSpec(q, 0, kv, 0, inner, P, H, L, T * n, 0.125, text_time=tt, n_per_media=n, T_img=T)
    out, lse = F.attn_fwd(spec)
    qr, kr = q.float().requires_grad_(True), kv.float().requires_grad_(True)
    ref = _attn_ref(_heads(qr, P, L, H), _heads(kr[:, :inner], P, T * n, H), _heads(kr[:, inner:], P, T * n, H), 0.125,
                    tt=tt.long(), n=n, T=T).permute(0, 2, 1, 3).reshape(P * L, inner)
    assert_close(out, ref, 2e-2, 2e-2, "masked attn fwd")
    # rows with text_time == 0 must be exactly zero
    zero_rows = (tt.reshape(-1) == 0)
    assert (out[zero_rows].float().abs().max().item() if zero_rows.any() else 0.0) == 0.0
    dout = rnd(P * L, inner, seed=5)
    ref.backward(dout.float())
    dq, dkv = torch.zeros_like(q), torch.zeros_like(kv)
    F.attn_bwd(spec, out, 0, lse, dout, 0, dq, 0, dkv, 0, inner)
    assert_close(dq, qr.grad, 3e-2, 3e-2, "masked attn dq")
    assert_close(dkv, kr.grad, 3e-2, 3e-2 * math.sqrt(L / 64), "masked attn dkv")


def test_small_passes():
    from otter_b200 import functional as F
    src = torch.randn(64, 1024, device=dev())
    out = F.bcast_rows(src, 64 * 5, 1, 64)
    assert torch.equal(out.view(5, 64, 1024), src.to(torch.bfloat16).expand(5, 64, 1024))
    x = rnd(5 * 64, 1024)
    cs = F.grouped_colsum(x, 1, 64)
    assert_close(cs, x.float().view(5, 64, 1024).sum(0), 1e-5, 1e-4, "grouped colsum latents")
    xf = rnd(2 * 3 * 16, 128)  # (img=6 -> F=3) x v=16
    cs = F.grouped_colsum(xf, 16, 3)
    assert_close(cs, xf.float().view(2, 3, 16, 128).sum((0, 2)), 1e-5, 1e-4, "grouped colsum frames")
    a, dy = rnd(1000, 512, seed=1), rnd(1000, 512, seed=2)
    gate = torch.tensor([0.3], device=dev())
    dg = F.gate_grad(dy, a, gate)
    ref = (1 - math.tanh(0.3) ** 2) * (dy.float() * a.float()).sum()
    assert abs(dg.item() - ref.item()) <= 1e-3 * abs(ref.item()) + 1e-2
    loss, dx = F.sqmean_loss(a)
    assert abs(loss.item() - a.float().pow(2).mean().item()) < 1e-4
    assert_close(dx, 2 * a.float() / a.numel(), 1e-2, 1e-9, "sqmean grad")
    w = torch.randn(1000, 333, device=dev())
    assert torch.equal(F.cast_bf16(w), w.to(torch.bfloat16))
    assert torch.equal(F.cast_f32(a), a.float())
    # CLIP embedding pieces
    px = torch.randn(2, 3, 56, 56, device=dev())
    cols = F.im2col_patches(px, 14, 592)
    ref = torch.nn.functional.unfold(px, 14, stride=14).transpose(1, 2).reshape(-1, 588)
    assert torch.equal(cols[:, :588], ref.to(torch.bfloat16)) and cols[:, 588:].abs().max().item() == 0
    pe = rnd(2 * 16, 256)
    cls, pos = torch.randn(256, device=dev()), torch.randn(17, 256, device=dev())
    h = F.clip_assemble(pe, cls, pos, 2, 16)
    ref = torch.cat([cls.expand(2, 1, 256), pe.float().view(2, 16, 256)], 1) + pos[None]
    assert_close(h, ref, 1e-2, 1e-2, "clip assemble")
    fe = torch.randn(4, 256, device=dev())
    hid = rnd(6, 17, 256)
    m = F.media_from_clip(hid, fe, 3)
    ref = hid.float()[:, 1:] + fe[:3].repeat(2, 1)[:, None, :]
    assert_close(m.view(6, 16, 256), ref, 1e-2, 1e-2, "media_from_clip")
    # fuyu scatter
    from oracle.restatement import fuyu_gather_continuous_embeddings
    word = rnd(2, 10, 64)
    cont = [rnd(3, 64, seed=1), rnd(4, 64, seed=2)]
    idx = torch.full((2, 10), -1, dtype=torch.int64)
    idx[0, 2:5] = torch.arange(3)
    idx[1, 1:5] = torch.tensor([3, 2, 1, 0])
    ref = fuyu_gather_continuous_embeddings(word.cpu().float(), [c.cpu().float() for c in cont], idx)
    got = F.fuyu_scatter(word, torch.cat(cont), idx.to(dev()), torch.tensor([0, 3, 7], device=dev()))
    assert torch.equal(got.cpu().float(), ref)
    idx[1, 9] = 4                                   # id == n_1: out of range -> never read out of bounds, word row kept
    got = F.fuyu_scatter(word, torch.cat(cont), idx.to(dev()), torch.tensor([0, 3, 7], device=dev()))
    assert torch.equal(got[1, 9], word[1, 9])


def test_label_mask_bit_exact_and_shifted_cross_entropy():
    """SURVEY.md §8f row 2: device label masking == the reference's masking() (golden, bit-exact) and the fused
    shifted cross-entropy (+ gradient) == F.cross_entropy on rolled labels (modeling_mpt.py:430-436)."""
    import os
    from oracle import restatement as R
    from otter_b200 import losses
    g = torch.load(os.path.join(os.path.dirname(__file__), "golden", "label_mask.pt"), weights_only=False)
    for name, c in g["cases"].items():
        got = losses.label_mask(c["input_ids"].to(dev()), g["eos"], g["answer"], g["eoc"])
        assert got.dtype == torch.int64 and torch.equal(got.cpu(), c["labels"]), name
    torch.manual_seed(0)
    for dtype, V, tol in ((torch.float32, 1000, 1e-5), (torch.bfloat16, 50432, 2e-3)):
        B, L = 3, 37
        logits = (torch.randn(B, L, V) * 2).to(dtype)
        labels = torch.randint(0, V, (B, L))
        labels[labels % 5 == 0] = -100
        labels[1, :] = -100                                   # a fully ignored sequence
        ref_in = logits.float().clone().requires_grad_(True)
        ref = R.shifted_cross_entropy(ref_in, labels.clone())
        (ref * 0.5).backward()
        x = logits.detach().to(dev()).requires_grad_(True)
        loss = losses.shifted_cross_entropy(x, labels.to(dev()))
        (loss * 0.5).backward()
        assert abs(loss.item() - ref.item()) <= tol * abs(ref.item()) + 1e-6, (dtype, loss.item(), ref.item())
        gerr = (x.grad.float().cpu() - ref_in.grad).abs().max().item()
        assert gerr <= (1e-7 if dtype == torch.float32 else 2e-4), (dtype, gerr)
    # nothing supervised: finite (0) loss, zero gradient
    x = torch.randn(1, 4, 64, device=dev(), requires_grad=True)
    loss = losses.shifted_cross_entropy(x, torch.full((1, 4), -100, device=dev()))
    loss.backward()
    assert loss.item() == 0.0 and x.grad.abs().max().item() == 0.0


def test_multi_tensor_cast_matches_per_tensor_cast():
    """params.refresh(): one launch for a list of fp32 weights == torch round-to-nearest-even bf16, bit for bit."""
    from otter_b200 import params as P
    torch.manual_seed(5)
    shapes = [(1,), (7,), (4096,), (4097,), (33, 129), (1024, 1024), (3, 5, 7), (2048, 4096)]
    ps = [torch.nn.Parameter(torch.randn(*s, device=dev()) * 3) for s in shapes]
    P.refresh(ps)
    for p in ps:
        got = P.bf16_of(p)
        assert got.shape == p.shape
        assert torch.equal(got, p.detach().to(torch.bfloat16)), p.shape
    with torch.no_grad():
        for p in ps:
            p.mul_(1.5)                                  # version bump: shadows stale
    P.refresh(ps)                                        # second call reuses the pointer table and the shadow buffers
    for p in ps:
        assert torch.equal(P.bf16_of(p), p.detach().to(torch.bfloat16)), p.shape


def test_upcast_with_folded_scale():
    """otb_cast_bf16_f32_scale: the up-cast after the bf16 all-reduce(SUM) with 1/world_size folded in (dp.py)."""
    from otter_b200 import functional as F
    g = torch.Generator().manual_seed(5)
    for n in (8, 4099, 1 << 20):
        src = torch.randn(n, generator=g).to(torch.bfloat16)
        out = torch.full((n,), 7.0, device=dev())
        F.cast_f32_scaled(src.to(dev()), out, 1.0 / 3.0)
        assert torch.equal(out.cpu(), src.float() * torch.tensor(1.0 / 3.0, dtype=torch.float32))
