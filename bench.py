#!/usr/bin/env python
"""bench.py — samples/sec of the vision-fusion hot path (harness mode M1, BASELINE.md §2 / SURVEY.md §8d).

One step = CLIP ViT-L/14 forward (frozen, no grad) -> PerceiverResampler (6 blocks, 64 latents) ->
8 x GatedCrossAttentionBlock(dim 4096) chained on a synthetic hidden state, loss = mean(out^2), backward
through the gated blocks and the perceiver (dgrad + wgrad, fp32 gradients into one flat buffer), and for
N > 1 the single NCCL all-reduce of that buffer.  Workload = BASELINE.json configs[1]
(OTTER-Image-MPT7B shape, per-GPU batch 8, 1 image/sample, L = 256, bf16), weak scaling over ranks.

  python bench.py [--gpus N --steps K --warmup W]            this repo's CUDA path (one rank per GPU)
  python bench.py --dump-outputs DIR [...]                    also writes the last timed step's loss and gradients
  python bench.py --impl reference [...]                      the reference's CPU implementation of the same path

Numerics of every GPU number printed here: production mode = bf16 operands, fp32 accumulation / softmax / LayerNorm
statistics (the reference's autocast(bf16) training recipe), held to the bf16 tolerances of tests/ (outputs 1.5e-2
rel-Frobenius, gradients 3-4e-2).  The north star's 1e-3 rel / 1e-5 abs is met by the forward-only fp32-grade mode
(`otter_b200.precision("fp32")`), which is a parity mode and is not what is timed.

The CPU arm (`--impl reference`, and the `cpu_baseline` leg of the GPU arm) times the reference's OWN modules (HF
CLIPVisionModel + OtterPerceiverResampler + 8 x OtterGatedCrossAttentionBlock, fp32, all host threads), imported from
/root/reference or from the archive oracle/build_ref.py packs into oracle/_ref (kind "reference"); without either it
falls back to oracle/restatement.py (kind "port").
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True       # the benchmark writes nothing into the tree it runs from (which may be read-only)

import torch  # noqa: E402

SEED = 0
BASE_CFG = dict(L=256, D=4096, n_gated=8, T=1, F=1, img=224, clip_layers=24, vis_dim=1024, latents=64,
                max_num_frames=None)
METRIC = "samples/sec perceiver+gated-xattn fwd+bwd"


# ---- algorithmic FLOPs (2*M*N*K per GEMM; SURVEY.md §8d) ---------------------------------------
def flops_per_sample(L=256, D=4096, T=1, Fr=1, n_gated=8):
    clip = 24 * (257 * (4 * 1024 ** 2 * 2 + 2 * 1024 * 4096 * 2) + 4 * 257 ** 2 * 1024) + 256 * 588 * 1024 * 2
    Nx = Fr * 256
    perc = 6 * (2 * (Nx + 64) * 1024 * 1024 + 2 * 64 * 1024 * 512 + 4 * 8 * 64 * (Nx + 64) * 64
                + 2 * 64 * 512 * 1024 + 4 * 64 * 1024 * 4096)
    gated = 2 * L * D * 512 + 2 * (T * 64) * 1024 * 1024 + 4 * 8 * L * (T * 64) * 64 + 2 * L * 512 * D + 4 * L * D * 4 * D
    return clip * T * Fr + 3 * perc * T + 3 * n_gated * gated


def host_cores():
    """CPU cores this process may actually use: min(affinity mask, cgroup quota, os.cpu_count())."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except Exception:
        pass
    return n


# ---- clocks sampler (nvidia-smi during the timed region) -----------------------------------------
class ClockSampler:
    def __init__(self, index):
        self.index, self.rows, self.proc, self.th = index, [], None, None

    def start(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i",
                                          str(self.index), "-lms", "100"], stdout=subprocess.PIPE, text=True)
        except Exception:
            self.proc = None
            return
        self.th = threading.Thread(target=self._read, daemon=True)
        self.th.start()

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            pass
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
            except Exception:
                continue
            for n, v in zip(names, r[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# ---- the CUDA arm -------------------------------------------------------------------------------
def build_modules(device, cfg):
    from transformers import CLIPVisionConfig
    from otter_b200.modeling_clip import CLIPVisionModel
    from otter_b200.modeling_otter import OtterGatedCrossAttentionBlock, OtterPerceiverResampler
    torch.manual_seed(SEED)       # identical weights on every rank (DDP semantics, no broadcast needed)
    vc = CLIPVisionConfig(hidden_size=1024, intermediate_size=4096, num_hidden_layers=cfg["clip_layers"],
                          num_attention_heads=16, image_size=cfg["img"], patch_size=14, hidden_act="quick_gelu")
    clip = CLIPVisionModel(vc).to(device).requires_grad_(False)
    perceiver = OtterPerceiverResampler(dim=cfg["vis_dim"], max_num_frames=cfg["max_num_frames"]).to(device)
    gated = torch.nn.ModuleList([OtterGatedCrossAttentionBlock(dim=cfg["D"], dim_visual=cfg["vis_dim"])
                                 for _ in range(cfg["n_gated"])]).to(device)
    with torch.no_grad():         # gates at 0 would make the path an identity (SURVEY.md §0)
        for g in gated:
            g.attn_gate.fill_(0.5)
            g.ff_gate.fill_(0.5)
    return clip, perceiver, gated


def host_batch(batch, rank, cfg, pin=True):
    g = torch.Generator().manual_seed(SEED + rank)     # rank r uses seed + r (train_utils.py:33-36)
    vision_x = torch.randn(batch, cfg["T"], cfg["F"], 3, cfg["img"], cfg["img"], generator=g).to(torch.bfloat16)
    hidden = torch.randn(batch, cfg["L"], cfg["D"], generator=g).to(torch.bfloat16)
    loc = torch.zeros(batch, cfg["L"], dtype=torch.bool)
    loc[:, 0] = True                                    # one <image> at position 0
    if pin:
        return vision_x.pin_memory(), hidden.pin_memory(), loc.pin_memory()
    return vision_x, hidden, loc


class HotPath:
    """The M1 step of one configuration on one rank: modules, flat gradient buffer, static device inputs, the two
    CUDA graphs (frozen CLIP forward | perceiver + gated fwd/bwd) and the timed loops."""

    def __init__(self, cfg, batch, dev, rank, world, args):
        from otter_b200.dp import FlatGradBuffer
        self.cfg, self.batch, self.dev, self.rank, self.world, self.args = cfg, batch, dev, rank, world, args
        self.clip, self.perceiver, self.gated = build_modules(dev, cfg)
        self.trainable = list(self.perceiver.parameters()) + list(self.gated.parameters())
        mode = args.grad_comm_dtype
        if mode == "auto":       # measured at N = 2 (profiles/r02_scale_sweep_n2.md): bf16-direct 713, fp32 688-705, bf16 664
            mode = "bf16-direct" if world > 1 else "fp32"
        self.comm_mode = mode
        comm_dtype = torch.bfloat16 if mode.startswith("bf16") else None
        direct = None
        if mode == "bf16-direct":                      # the Linear weights' wgrad epilogues write the wire buffer
            direct = [m.weight for mod in (self.perceiver, self.gated) for m in mod.modules()
                      if isinstance(m, torch.nn.Linear)]
        self.flat = FlatGradBuffer(self.trainable, device=dev, comm_dtype=comm_dtype,
                                   nccl_registered=args.nccl_registered and world > 1, direct_params=direct,
                                   reduce_op=args.reduce_op)
        self.h_vis, self.h_hid, self.h_loc = host_batch(batch, rank, cfg)
        self.d_vis, self.d_hid, self.d_loc = self.h_vis.to(dev), self.h_hid.to(dev), self.h_loc.to(dev)
        self.loss_host = torch.zeros(1).pin_memory()
        self.graphed = None
        self.hidden = None
        self.loss = None
        self.launches_per_step = None
        self.prefetch = None

    # -- the step ---------------------------------------------------------------------------------
    def clip_step(self, vis):
        """Frozen CLIP tower on this step's images (no grad, independent of the trainable weights)."""
        b_, T_, F_ = vis.shape[:3]
        return self.clip.last_hidden_bf16(vis.reshape(b_ * T_ * F_, *vis.shape[3:]))      # bf16 [bTF, 257, 1024]

    def train_step(self, hidden, hid, loc):
        """perceiver + gated blocks forward/backward on precomputed CLIP features."""
        from otter_b200 import functional as F
        from otter_b200 import params as P
        from otter_b200.blocks import MediaFromClipFn
        cfg = self.cfg
        B, L, D = hid.shape
        # weights "just updated by the optimizer": re-derive the bf16 compute copies (autocast-equivalent work)
        if self.args.multi_cast:
            P.refresh(self.trainable)                     # one multi-tensor launch
        else:
            P.invalidate(self.trainable)                  # one cast launch per weight, on first use
        self.flat.begin_step()
        media = MediaFromClipFn.apply(hidden, self.perceiver.frame_embs, cfg["F"])          # drop CLS (+frame_embs)
        media = self.perceiver.resample_media(media, B * cfg["T"])                           # [B*T*64, 1024] bf16
        tt = F.text_time(loc, True)
        x = hid.view(B * L, D).detach().requires_grad_(True)
        for g in self.gated:
            x = g.forward_2d(x, media, tt, B, L, cfg["T"], cfg["latents"])
        loss, dx = F.sqmean_loss(x)
        x.backward(dx)
        self.flat.finish_step()
        return loss

    def step_eager(self, vis, hid, loc):
        return self.train_step(self.clip_step(vis), hid, loc)

    def prepare(self):
        from otter_b200 import functional as F
        self.step_eager(self.d_vis, self.d_hid, self.d_loc)     # first step also builds the frozen CLIP weight shadows
        n0 = F.launch_count()
        self.step_eager(self.d_vis, self.d_hid, self.d_loc)
        self.launches_per_step = F.launch_count() - n0
        if not self.args.no_graph:
            from otter_b200.graph import GraphedStep
            ga = GraphedStep(self.clip_step, self.d_vis)
            gb = GraphedStep(self.train_step, ga.outputs, self.d_hid, self.d_loc)
            self.graphed = (ga, gb)
        self.run_clip()                                  # pipeline prologue: features of the first batch

    def run_clip(self):
        self.hidden = self.graphed[0].replay() if self.graphed is not None else self.clip_step(self.d_vis)

    def run_step(self):
        """One step = train_step on the CLIP features of this batch, then the ONE gradient all-reduce, overlapped
        with the frozen CLIP forward of the next batch (data prefetch: it does not depend on the weight update)."""
        import torch.distributed as dist
        loss = self.graphed[1].replay() if self.graphed is not None else \
            self.train_step(self.hidden, self.d_hid, self.d_loc)
        self.loss = loss
        work = self.flat.all_reduce(async_op=True)
        self.run_clip()
        if work is not None:
            work.wait()
            if dist.get_backend() == "gloo" and not getattr(work, "averaged", False):
                self.flat.flat.div_(self.world)
        return loss

    def enable_prefetch(self):
        """opt-in loader pipeline for the e2e leg: a copy stream fills device staging buffers with the next step's
        inputs while the current step computes; the step then starts with three device-to-device copies."""
        cs = torch.cuda.Stream(device=self.dev)
        pf = {"vis": torch.empty_like(self.d_vis), "hid": torch.empty_like(self.d_hid),
              "loc": torch.empty_like(self.d_loc), "landed": torch.cuda.Event(), "free": torch.cuda.Event()}

        def _issue():
            cs.wait_event(pf["free"])
            with torch.cuda.stream(cs):
                pf["vis"].copy_(self.h_vis, non_blocking=True)
                pf["hid"].copy_(self.h_hid, non_blocking=True)
                pf["loc"].copy_(self.h_loc, non_blocking=True)
                pf["landed"].record(cs)

        pf["issue"] = _issue
        pf["free"].record(torch.cuda.current_stream())
        _issue()                                         # prologue: inputs of the first timed step
        self.prefetch = pf

    def timed(self, n, e2e):
        import torch.distributed as dist
        start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        pf = self.prefetch
        if self.world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        start.record()
        for _ in range(n):
            if e2e and pf is not None:                   # same bytes per step, H2D of the NEXT step's inputs overlapped
                main = torch.cuda.current_stream()
                main.wait_event(pf["landed"])            # this step's inputs sit in the staging buffers
                self.d_vis.copy_(pf["vis"]); self.d_hid.copy_(pf["hid"]); self.d_loc.copy_(pf["loc"])   # D2D, us
                pf["free"].record(main)
                pf["issue"]()                            # pinned host -> staging on the copy stream, behind `free`
                loss = self.run_step()
                self.loss_host.copy_(loss, non_blocking=True)
                main.synchronize()                                          # the user reads the loss every step
            elif e2e:                                    # pinned host -> static device inputs, step, loss -> host
                self.d_vis.copy_(self.h_vis, non_blocking=True)
                self.d_hid.copy_(self.h_hid, non_blocking=True)
                self.d_loc.copy_(self.h_loc, non_blocking=True)
                loss = self.run_step()
                self.loss_host.copy_(loss, non_blocking=True)
                torch.cuda.current_stream().synchronize()                   # the user reads the loss every step
            else:
                self.run_step()
        end.record()
        if self.world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ms = start.elapsed_time(end)
        if self.world > 1:
            t = torch.tensor([ms], device=self.dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = t.item()
        return ms

    def h2d_bytes(self):
        return self.h_vis.numel() * 2 + self.h_hid.numel() * 2 + self.h_loc.numel()

    def close(self):
        from otter_b200 import params as P
        self.graphed = self.hidden = self.prefetch = None
        self.clip = self.perceiver = self.gated = self.trainable = self.flat = None
        self.d_vis = self.d_hid = self.d_loc = None
        P.clear_caches()
        import gc
        gc.collect()
        torch.cuda.empty_cache()


def graph_time_us(calls, reps=5):
    """Capture `calls` (a list of zero-argument launchers, each touching its own buffers) into one CUDA graph and
    time replays with CUDA events: microseconds per launch, back to back the way they run inside a step."""
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for c in calls:
            c()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, capture_error_mode="thread_local"):
        for c in calls:
            c()
    for _ in range(2):
        g.replay()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / (reps * len(calls))


def dominant_gemm_times(dev, M, D):
    from otter_b200 import functional as F
    g = torch.Generator(device=dev).manual_seed(1)

    def rn(*shape, scale=1.0):
        return (torch.randn(*shape, device=dev, generator=g) * scale).to(torch.bfloat16)

    x, h, dy, dz = rn(M, D), rn(M, 4 * D), rn(M, D), rn(M, 4 * D)
    w1, w2 = rn(4 * D, D, scale=D ** -0.5), rn(D, 4 * D, scale=(4 * D) ** -0.5)
    z, a2 = torch.empty(M, 4 * D, device=dev, dtype=torch.bfloat16), torch.empty(M, D, device=dev, dtype=torch.bfloat16)
    gw1 = torch.zeros(4 * D, D, device=dev)
    gw2 = torch.zeros(D, 4 * D, device=dev)
    gate = torch.full((1,), 0.5, device=dev)
    calls = {
        "fwd_up_gelu": lambda: F.linear_fwd(x, w1, act=1, aux_out=z),
        "fwd_down_gate_res": lambda: F.linear_fwd(h, w2, aux_out=a2, scale_ptr=gate, scale_tanh=True, residual=x),
        "dgrad_down_dgelu": lambda: F.linear_dgrad(dy, w2, aux_in=z, scale_ptr=gate, scale_tanh=True),
        "dgrad_up": lambda: F.linear_dgrad(dz, w1),
        "wgrad_down": lambda: F.linear_wgrad(dy, h, out=gw2, accumulate=False, scale_ptr=gate, scale_tanh=True),
        "wgrad_up": lambda: F.linear_wgrad(dz, x, out=gw1, accumulate=False),
    }
    F.linear_fwd(x, w1, act=1, aux_out=z)        # realistic pre-activations for the dGELU epilogue
    per, tot_ms = {}, 0.0
    flops = 2.0 * M * D * 4 * D
    for name, fn in calls.items():
        for _ in range(3):
            fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(10):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / 10
        per[name] = round(ms * 1e3, 1)
        tot_ms += ms
    return {"tflops": 6 * flops / (tot_ms * 1e-3) / 1e12, "per_class_us": per, "sum_ms": tot_ms, "flops_avg": flops}


def hbm_kernel_rooflines(dev, batch, cfg, hbm_gbs):
    """The HBM-bound kernels of the step against the measured copy bandwidth (SURVEY.md §8d): fused attention A
    (perceiver), B (gated cross-attention), their backward, the CLIP attention, LayerNorm and the weight cast.
    Each launch of a timed graph works on its own buffers (rotating sets, > 126 MB in total) so operands come from HBM,
    not from L2; `bytes` are the ALGORITHMIC bytes (every operand touched once, SURVEY.md §8d)."""
    from otter_b200 import functional as F
    BF = torch.bfloat16
    g = torch.Generator(device=dev).manual_seed(3)

    def rn(*shape):
        return torch.randn(*shape, device=dev, generator=g).to(BF)

    out = []

    def add(name, shape, nbytes, calls, note=""):
        us = graph_time_us(calls)
        gbs = nbytes / (us * 1e-6) / 1e9
        out.append({"kernel": name, "shape": shape, "algorithmic_bytes": int(nbytes), "us": round(us, 2),
                    "achieved_gbs": round(gbs, 1), "frac": round(gbs / hbm_gbs, 4), **({"note": note} if note else {})})

    def sets(nbytes):
        return max(2, int(math.ceil(256e6 / nbytes)))

    H, n, L, T = 8, cfg["latents"], cfg["L"], cfg["T"]
    inner = H * 64
    # ---- kernel A: perceiver attention, P = batch*T problems, 64 query latents, Nx + 64 keys (two key sources)
    Nx = cfg["F"] * 256
    P = batch * T
    bytesA = P * H * (2 * n * 64 + 2 * (Nx + n) * 64) * 2
    R = sets(bytesA)
    specs, bw = [], []
    for _ in range(R):
        q, kv = rn(P * n, inner), rn(P * (Nx + n), 2 * inner)
        specs.append(F.AttnSpec(q, 0, kv[:P * Nx], 0, inner, P, H, n, Nx, 0.125, kv2=kv[P * Nx:], k2_col0=0,
                                v2_col0=inner, Sk2=n))
    add("attention A fwd (perceiver latents x [media ; latents])", f"P={P} H=8 Sq={n} Sk={Nx}+{n}", bytesA,
        [(lambda s=s: F.attn_fwd(s)) for s in specs])
    for s in specs:
        o, lse = F.attn_fwd(s)
        do, dq, dkv = rn(P * n, inner), torch.empty(P * n, inner, device=dev, dtype=BF), \
            torch.empty(P * (Nx + n), 2 * inner, device=dev, dtype=BF)
        bw.append((s, o, lse, do, dq, dkv))
    add("attention A bwd", f"P={P} H=8 Sq={n} Sk={Nx}+{n}", 2 * bytesA + P * H * n * 64 * 2,
        [(lambda t=t: F.attn_bwd(t[0], t[1], 0, t[2], t[3], 0, t[4], 0, t[5][:P * Nx], 0, inner, t[5][P * Nx:], 0, inner))
         for t in bw], note="reads Q,K,V,O,dO, writes dQ,dK,dV")
    del specs, bw
    # ---- kernel B: gated cross-attention, P = batch problems, L query rows, T*64 keys, media mask
    bytesB = batch * H * (2 * L * 64 + 2 * (T * n) * 64) * 2
    R = sets(bytesB)
    loc = torch.zeros(batch, L, dtype=torch.bool, device=dev)
    loc[:, 0] = True
    tt = F.text_time(loc, True)
    specs, bw = [], []
    for _ in range(R):
        q, kv = rn(batch * L, inner), rn(batch * T * n, 2 * inner)
        specs.append(F.AttnSpec(q, 0, kv, 0, inner, batch, H, L, T * n, 0.125, text_time=tt, n_per_media=n, T_img=T))
    add("attention B fwd (text x latents, media mask)", f"P={batch} H=8 Sq={L} Sk={T * n}", bytesB,
        [(lambda s=s: F.attn_fwd(s)) for s in specs])
    for s in specs:
        o, lse = F.attn_fwd(s)
        do, dq, dkv = rn(batch * L, inner), torch.empty(batch * L, inner, device=dev, dtype=BF), \
            torch.empty(batch * T * n, 2 * inner, device=dev, dtype=BF)
        bw.append((s, o, lse, do, dq, dkv))
    add("attention B bwd", f"P={batch} H=8 Sq={L} Sk={T * n}", 2 * bytesB + batch * H * L * 64 * 2,
        [(lambda t=t: F.attn_bwd(t[0], t[1], 0, t[2], t[3], 0, t[4], 0, t[5], 0, inner)) for t in bw],
        note="reads Q,K,V,O,dO, writes dQ,dK,dV")
    del specs, bw
    # ---- CLIP self-attention: N images, 16 heads, 257 tokens, q|k|v fused
    N, S, Dc = batch * T * cfg["F"], 257, 1024
    bytesC = N * 16 * 4 * S * 64 * 2
    qkvs = [rn(N * S, 3 * Dc) for _ in range(sets(bytesC))]
    add("attention CLIP fwd", f"P={N} H=16 S={S}", bytesC,
        [(lambda x=x: F.attn_fwd(F.AttnSpec(x, 0, x, Dc, 2 * Dc, N, 16, S, S, 0.125), want_lse=False)) for x in qkvs])
    del qkvs
    # ---- LayerNorm fwd / bwd at the gated blocks' shape, weight cast at the FFN weight's size
    rows, D = batch * L, cfg["D"]
    gam, bet = torch.ones(D, device=dev), torch.zeros(D, device=dev)
    xs = [rn(rows, D) for _ in range(sets(rows * D * 4))]
    add("layernorm fwd", f"{rows}x{D}", rows * D * 4, [(lambda x=x: F.layernorm_fwd(x, gam, bet)) for x in xs])
    st = [F.layernorm_fwd(x, gam, bet) for x in xs]
    dys = [rn(rows, D) for _ in xs]
    add("layernorm bwd (dx + dgamma/dbeta, residual-gradient add)", f"{rows}x{D}", rows * D * 2 * 4,
        [(lambda x=x, s=s, dy=dy: F.layernorm_bwd(dy, x, s[1], s[2], gam, add=dy)) for x, s, dy in zip(xs, st, dys)],
        note="reads dy, x, add; writes dx")
    del xs, st, dys
    w = torch.randn(4 * D, D, device=dev)
    wb = torch.empty(4 * D, D, device=dev, dtype=BF)
    add("fp32 -> bf16 weight cast", f"{4 * D}x{D}", 4 * D * D * 6, [lambda: F.cast_bf16(w, wb)] * 2)
    return out


def self_check(hp):
    """Outside the timed region: the timed configuration's modules (same weights) at batch 1 — loss and two gradient
    norms of the CUDA path against the CPU oracle (oracle/restatement.py, fp32).  Catches a wrong-but-fast step."""
    from oracle import restatement as R
    cfg = hp.cfg
    hv, hh, hl = host_batch(1, 1000, cfg, pin=False)
    dev = hp.dev
    loss = hp.step_eager(hv.to(dev), hh.to(dev), hl.to(dev))
    torch.cuda.synchronize()
    w1 = hp.gated[0].feed_forward[1].weight
    got = {"loss": loss.item(), "gnorm_gated0_ff1": w1.grad.float().norm().item(),
           "gnorm_latents": hp.perceiver.latents.grad.float().norm().item()}
    t0 = time.perf_counter()
    clip_p = {k: v.detach().float().cpu() for k, v in hp.clip.state_dict().items()}
    perc_p = {k: v.detach().float().cpu().requires_grad_(True) for k, v in hp.perceiver.state_dict().items()}
    gated_ps = [{k: v.detach().float().cpu().requires_grad_(True) for k, v in g.state_dict().items()} for g in hp.gated]
    torch.set_num_threads(host_cores())
    out, _ = R.m1_forward(hv.float(), hh.float(), hl, clip_p, perc_p, gated_ps)
    ref_loss = out.float().pow(2).mean()
    ref_loss.backward()
    want = {"loss": ref_loss.item(), "gnorm_gated0_ff1": gated_ps[0]["feed_forward.1.weight"].grad.norm().item(),
            "gnorm_latents": perc_p["latents"].grad.norm().item()}
    rel = {k: abs(got[k] - want[k]) / max(abs(want[k]), 1e-30) for k in got}
    tol = {"loss": 1e-2, "gnorm_gated0_ff1": 3e-2, "gnorm_latents": 3e-2}
    return {"ok": all(rel[k] <= tol[k] for k in rel), "batch": 1, "cuda": got, "oracle_fp32": want,
            "rel_err": {k: float(f"{v:.3e}") for k, v in rel.items()}, "tol": tol,
            "oracle_seconds": round(time.perf_counter() - t0, 1)}


DUMP_SAMPLE = 65536                 # gradient entries kept per parameter by --dump-outputs


def dump_outputs(hp, out_dir):
    """What the last step handed its caller, the loss and the fp32 gradient of every trainable parameter, as
    <out_dir>/<name>.npy in float32.  A gradient with more than DUMP_SAMPLE entries is sampled at positions drawn from a
    generator seeded with the parameter's name, so that two builds of the project can be compared entry for entry."""
    import zlib

    import numpy as np
    torch.cuda.synchronize()
    arrays = {"loss": hp.loss}
    for prefix, mod in (("perceiver", hp.perceiver), ("gated", hp.gated)):
        for pname, p in mod.named_parameters():
            name = f"grad.{prefix}.{pname}"
            g = p.grad.detach().reshape(-1)
            if g.numel() > DUMP_SAMPLE:
                gen = torch.Generator().manual_seed(zlib.crc32(name.encode()))
                g = g[torch.randint(g.numel(), (DUMP_SAMPLE,), generator=gen).sort().values.to(g.device)]
            arrays[name] = g
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.float().cpu().numpy())
    return len(arrays), sum(t.numel() * 4 for t in arrays.values())


def fuyu_patch_linear_times(dev):
    """BASELINE configs[4] (OtterHD/Fuyu patch-linear, no vision encoder): Linear(2700 -> 4096, bias) on N_p patches +
    scatter into the word embeddings, through otter_b200.modeling_fuyu (reference signature)."""
    from otter_b200 import modeling_fuyu as MF
    res = {}
    lin = torch.nn.Linear(2700, 4096).to(dev)
    emb = torch.nn.Embedding(1024, 4096).to(dev).to(torch.bfloat16)
    for n_p in (1225, 4096):
        S = n_p + 64
        patches = [torch.randn(1, n_p, 2700, device=dev).to(torch.bfloat16)]
        ids = torch.randint(0, 1024, (1, S), device=dev)
        idx = torch.full((1, S), -1, dtype=torch.int64, device=dev)
        idx[0, 32:32 + n_p] = torch.arange(n_p, device=dev)
        with torch.no_grad():
            for _ in range(3):
                MF.embed_inputs(emb, lin, ids, image_patches=patches, image_patches_indices=idx)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            for _ in range(10):
                MF.embed_inputs(emb, lin, ids, image_patches=patches, image_patches_indices=idx)
            e1.record()
            torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / 10
        res[f"N_p={n_p}"] = {"ms": round(ms, 3), "images_per_s": round(1e3 / ms, 1),
                             "gemm_gflop": round(2 * n_p * 2700 * 4096 / 1e9, 1), "seq": S,
                             "note": "eager (host launches + the reference's index checks included)"}
    return res


def allreduce_alone(hp, dev, world, iters=10):
    """The step's one collective timed on its own (SURVEY.md §8d "NCCL all-reduce timed separately"): CUDA events on the
    current stream around `iters` back-to-back FlatGradBuffer.all_reduce() calls — cast of the fp32-produced tail, the NCCL
    all-reduce, the up-cast into the fp32 `.grad` views — nothing overlapped with it, max over ranks.  Bus bandwidth =
    2 (N-1)/N x wire bytes / time, the figure nccl-tests quotes, to hold against NVLink 5's 900 GB/s per direction."""
    import torch.distributed as dist
    for _ in range(2):
        hp.flat.all_reduce()
    torch.cuda.synchronize()
    dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        hp.flat.all_reduce()
    e1.record()
    torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1) / iters], device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    nbytes = hp.flat.comm_nbytes()
    return {"ms": round(ms, 3), "wire_bytes": int(nbytes), "iters": iters,
            "busbw_gbs": round(2.0 * (world - 1) / world * nbytes / (ms * 1e-3) / 1e9, 1),
            "includes": "tail cast + NCCL all-reduce + up-cast to the fp32 .grad views; not overlapped with compute "
                        "(inside the step it overlaps the next batch's CLIP forward)"}


class _BenchTokenizer:
    """Offline stand-in for the HF tokenizer the model constructor downloads (no network on the box): ids only."""
    pad_token = None

    def __init__(self, base=50277):
        self.vocab, self.base = {}, base

    @classmethod
    def from_pretrained(cls, *a, **k):
        return cls()

    def add_special_tokens(self, d):
        for tok in d.get("additional_special_tokens", []):
            self.vocab.setdefault(tok, self.base + len(self.vocab))
        if "pad_token" in d:
            self.pad_token = d["pad_token"]
            self.vocab.setdefault(d["pad_token"], self.base + len(self.vocab))
        return len(self.vocab)

    def encode(self, text):
        return [self.vocab[text]]

    def __len__(self):
        return self.base + len(self.vocab)


class _BenchLlamaTokenizer(_BenchTokenizer):
    def __init__(self):
        super().__init__(base=32000)


def m2_dropin_times(dev, batch, L, steps=5, lm="mpt", frames=1):
    """Harness mode M2 (SURVEY.md §8d): the full drop-in OtterForConditionalGeneration through the reference's forward()
    signature, forward + backward, eager launches (the HF module plumbing is not graph-captured).
      lm="mpt":   OTTER-Image-MPT7B shape — CLIP ViT-L/14 + perceiver + 32 frozen MPT layers (D 4096, 32 heads, ALiBi) with a
                  gated block before every 4th, tied 50432-token LM head, shifted cross-entropy (otter_b200.lm_mpt).
      lm="llama": OTTER-Video-LLaMA7B shape (BASELINE configs[2]) — `frames` frames per sample, 32 frozen LLaMA layers
                  (otter_b200.lm_llama inside HF's LlamaForCausalLM shell; trainable embeddings + LM head as in the
                  reference, modeling_otter.py:897-905), under autocast(bf16) like the reference's accelerate recipe."""
    from otter_b200 import otter_hf
    otter_hf.AutoTokenizer = _BenchTokenizer if lm == "mpt" else _BenchLlamaTokenizer
    torch.manual_seed(SEED)
    extra = {}
    if lm == "mpt":
        text = dict(d_model=4096, n_heads=32, n_layers=32, expansion_ratio=4, max_seq_len=2048, vocab_size=50432, no_bias=True,
                    attn_config=dict(attn_impl="torch", alibi=True, alibi_bias_max=8), architectures=["MPTForCausalLM"],
                    tie_word_embeddings=True, init_device="cpu")
        vocab_hi, head_vocab, mlp_mult = 50000, 50432, 8
    else:
        text = dict(model_type="llama", hidden_size=4096, intermediate_size=11008, num_hidden_layers=32,
                    num_attention_heads=32, num_key_value_heads=32, vocab_size=32004, max_position_embeddings=2048,
                    architectures=["LlamaForCausalLM"], tie_word_embeddings=False)
        vocab_hi, head_vocab, mlp_mult = 31000, 32004, 3 * 11008 / 4096
        extra = dict(max_num_frames=128)
    vis = dict(hidden_size=1024, intermediate_size=4096, num_hidden_layers=24, num_attention_heads=16, image_size=224,
               patch_size=14, hidden_act="quick_gelu")
    with torch.device(dev):
        model = otter_hf.OtterForConditionalGeneration(otter_hf.OtterConfig(vision_config=vis, text_config=text,
                                                                             cross_attn_every_n_layers=4, **extra))
    if lm == "llama":
        from otter_b200.lm_llama import FrozenLlamaDecoderLayer
        n_native = sum(isinstance(m_, FrozenLlamaDecoderLayer) for m_ in model.modules())
        assert n_native == 32, f"expected 32 otter_b200 LLaMA layers, found {n_native}"
    with torch.no_grad():
        for n_, p_ in model.named_parameters():
            if n_.endswith("attn_gate") or n_.endswith("ff_gate"):
                p_.fill_(0.5)
            elif "lang_encoder" in n_ and "gated_cross_attn" not in n_ and p_.dim() == 2:
                p_.normal_(0.0, 0.02)
    model.train()
    g = torch.Generator().manual_seed(SEED)
    vision_x = torch.randn(batch, 1, frames, 3, 224, 224, generator=g).to(torch.bfloat16).to(dev)
    lang_x = torch.randint(3, vocab_hi, (batch, L), generator=g).to(dev)
    lang_x[:, 0] = model.media_token_id
    labels = lang_x.clone()
    labels[:, 0] = -100
    mask = torch.ones_like(lang_x)
    trainable = [p_ for p_ in model.parameters() if p_.requires_grad]

    def one():
        for p_ in trainable:
            p_.grad = None
        with torch.autocast("cuda", dtype=torch.bfloat16, enabled=(lm == "llama")):
            out = model(vision_x=vision_x, lang_x=lang_x, attention_mask=mask, labels=labels)
        out.loss.backward()
        return out.loss

    for _ in range(3):
        loss = one()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(steps):
        loss = one()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    # per token: fwd + dgrad of the 32 frozen layers (4 + mlp_mult D x D matrices each) + LM head fwd + dgrad + wgrad
    lm_flops = 2 * 32 * (4 + mlp_mult) * 4096 * 4096 * 2 + 2 * 3 * head_vocab * 4096
    res = {"samples_per_s": round(batch / (ms * 1e-3), 1), "ms_per_step": round(ms, 2), "per_gpu_batch": batch, "L": L,
           "steps": steps, "loss": round(float(loss), 4), "launch": "eager",
           "trainable_params": sum(p_.numel() for p_ in trainable),
           "lm": lm, "frames": frames,
           "algorithmic_tflops": round((flops_per_sample(L, Fr=frames) + lm_flops * L) * batch / (ms * 1e-3) / 1e12, 1)}
    del model, trainable
    return res


def run_extras(dev, rank, world, args, log):
    """Other BASELINE.json configurations / sweep points, measured the same way (device-timed, CUDA graphs, W >= 3),
    reported as extra fields: they do not change `value`."""
    extras = {}
    steps = max(5, min(args.steps, 10))
    points = []
    if world == 1:
        points += [("c3_video_llama7b_b4_F8", dict(BASE_CFG, F=8, max_num_frames=128), 4),
                   ("c2_L128", dict(BASE_CFG, L=128), 8), ("c2_L512", dict(BASE_CFG, L=512), 8),
                   ("c2_L1024", dict(BASE_CFG, L=1024), 8)]
    points += [("c4_shape_per_gpu_batch32", dict(BASE_CFG), 32)]
    for name, cfg, b in points:
        try:
            hp = HotPath(cfg, b, dev, rank, world, args)
            hp.prepare()
            for _ in range(3):
                hp.run_step()
            ms = hp.timed(steps, e2e=False) / steps
            fl = flops_per_sample(cfg["L"], cfg["D"], cfg["T"], cfg["F"], cfg["n_gated"])
            extras[name] = {"samples_per_s": round(b * world / (ms * 1e-3), 1), "ms_per_step": round(ms, 3),
                            "per_gpu_batch": b, "L": cfg["L"], "frames": cfg["F"], "steps": steps,
                            "algorithmic_tflops_per_gpu": round(fl * b / (ms * 1e-3) / 1e12, 1)}
            log(f"extra {name}: {ms:.2f} ms/step")
            hp.close()
            del hp
        except Exception as e:                      # an extra point must never take the headline line down
            extras[name] = {"error": f"{type(e).__name__}: {e}"[:200]}
            log(f"extra {name} failed: {e}")
    if world == 1 and rank == 0:
        try:
            extras["c5_fuyu_patch_linear"] = fuyu_patch_linear_times(dev)
        except Exception as e:
            extras["c5_fuyu_patch_linear"] = {"error": f"{type(e).__name__}: {e}"[:200]}
        try:
            from otter_b200 import params as P
            extras["m2_dropin_otter_mpt7b"] = m2_dropin_times(dev, 8, BASE_CFG["L"])
            log(f"extra M2 drop-in: {extras['m2_dropin_otter_mpt7b']['ms_per_step']} ms/step")
            P.clear_caches()
            torch.cuda.empty_cache()
        except Exception as e:
            extras["m2_dropin_otter_mpt7b"] = {"error": f"{type(e).__name__}: {e}"[:300]}
        try:
            from otter_b200 import params as P
            extras["m2_dropin_otter_video_llama7b"] = m2_dropin_times(dev, 4, BASE_CFG["L"], lm="llama", frames=8)
            log(f"extra M2 drop-in (LLaMA-7B, 8 frames): {extras['m2_dropin_otter_video_llama7b']['ms_per_step']} ms/step")
            P.clear_caches()
            torch.cuda.empty_cache()
        except Exception as e:
            extras["m2_dropin_otter_video_llama7b"] = {"error": f"{type(e).__name__}: {e}"[:300]}
    return extras


def run_cuda(args):
    import torch.distributed as dist
    from otter_b200 import functional as F

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torch.distributed.run --nproc-per-node N for --gpus N > 1")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    batch = args.per_gpu_batch
    cfg = dict(BASE_CFG, L=args.seq_len)

    def log(msg):
        if rank == 0:
            print(f"[bench] {msg}", file=sys.stderr, flush=True)

    hp = HotPath(cfg, batch, dev, rank, world, args)
    if args.e2e_prefetch:
        hp.enable_prefetch()
    log(f"modules built (world {world}, per-GPU batch {batch})")
    hp.prepare()
    if hp.graphed is not None:
        log("step captured as two CUDA graphs (CLIP forward | perceiver + gated fwd/bwd)")
    for _ in range(max(args.warmup, 3)):
        hp.run_step()
    torch.cuda.synchronize()

    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    ms = hp.timed(args.steps, e2e=False)
    log(f"timed region done: {ms / args.steps:.3f} ms/step")
    launches = hp.launches_per_step
    clocks = sampler.stop() if sampler else None
    ms_e2e = hp.timed(args.steps, e2e=True)
    if args.dump_outputs and rank == 0:
        n, nbytes = dump_outputs(hp, args.dump_outputs)
        log(f"last step's loss and gradients: {n} arrays, {nbytes / 2 ** 20:.1f} MiB in {args.dump_outputs}")

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_gbs = peaks.get("hbm_gbs", 6600.0)

    # ---- roofline of the dominant kernel: the six 4096<->16384 FFN GEMM launch classes of the gated blocks
    # (8 launches each per step, 86 % of the step's algorithmic FLOPs), each timed live with CUDA events over
    # 10 back-to-back launches on fresh N(0,1) operands (operands + outputs > L2) ----
    B, L, D = batch, cfg["L"], cfg["D"]
    dom = dominant_gemm_times(dev, B * L, D) if rank == 0 else None
    hbm_rows = None
    if rank == 0 and not args.no_kernel_rooflines:
        try:
            hbm_rows = hbm_kernel_rooflines(dev, batch, cfg, hbm_gbs)
        except Exception as e:
            hbm_rows = [{"error": f"{type(e).__name__}: {e}"[:300]}]
    # eager per-launch event timing of EVERY GEMM of one step (includes host launch gaps; kept as a cross-check)
    prof = []
    F.set_gemm_profiler(prof)
    hp.step_eager(hp.d_vis, hp.d_hid, hp.d_loc)
    hp.flat.all_reduce()
    F.set_gemm_profiler(None)
    torch.cuda.synchronize()
    g_ms = sum(r[1].elapsed_time(r[2]) for r in prof)
    if rank == 0 and os.environ.get("OTB_GEMM_BREAKDOWN"):
        agg = {}
        for f, a_, b_, shape in prof:
            t = agg.setdefault(shape, [0, 0.0, 0.0])
            t[0] += 1
            t[1] += a_.elapsed_time(b_)
            t[2] += f
        with open(os.environ["OTB_GEMM_BREAKDOWN"], "w") as fh:
            fh.write("M,N,K,a_mn,b_mn,launches,total_ms,avg_us,TFLOPs\n")
            for shape, (n, ms_, fl_) in sorted(agg.items(), key=lambda kv: -kv[1][1]):
                fh.write(",".join(map(str, shape)) + f",{n},{ms_:.3f},{ms_ / n * 1e3:.1f},{fl_ / ms_ / 1e9:.1f}\n")
    check = None
    if rank == 0 and world == 1 and not args.no_self_check:
        try:
            check = self_check(hp)
            log(f"self-check vs the CPU oracle at batch 1: {check['rel_err']} ok={check['ok']}")
        except Exception as e:
            check = {"ok": False, "error": f"{type(e).__name__}: {e}"[:300]}
    comm_alone = None
    if world > 1:                                   # after every timed region: cannot disturb `value` / `e2e`
        try:
            comm_alone = allreduce_alone(hp, dev, world)
            log(f"all-reduce alone: {comm_alone['ms']} ms, bus bandwidth {comm_alone['busbw_gbs']} GB/s")
        except Exception as e:
            comm_alone = {"error": f"{type(e).__name__}: {e}"[:200]}
    h2d = hp.h2d_bytes()
    comm_mode = hp.comm_mode
    comm_bytes = hp.flat.comm_nbytes() if world > 1 else 0
    hp.close()
    del hp
    extras = None
    if not args.no_extras:
        extras = run_extras(dev, rank, world, args, log)
    if world > 1:
        dist.barrier()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    peak_tf = peaks.get("bf16_tflops", 1590.0)                # kernel timed alone -> burst figure
    peak_sus = peaks.get("bf16_tflops_sustained", 1400.0)
    peak_src = "MEASURED_PEAKS.json bf16_tflops (burst; kernel timed alone)" if peaks else \
        "fallback 1590 TFLOP/s (B200_PROFILING.md)"
    step_ms = ms / args.steps
    value = batch * world * args.steps / (ms / 1e3)
    e2e_value = batch * world * args.steps / (ms_e2e / 1e3)
    fl = flops_per_sample(cfg["L"], cfg["D"], cfg["T"], cfg["F"], cfg["n_gated"])
    ach = dom["tflops"]
    out = {
        "metric": METRIC, "value": round(value, 2), "unit": "samples/s",
        "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": round(step_ms, 3),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": "OTTER-Image-MPT7B shape (BASELINE configs[1]), M1 hot path: CLIP ViT-L/14 fwd -> "
                               "perceiver(6x64 latents) -> 8 gated x-attn blocks D=4096, fwd+bwd",
                   "per_gpu_batch": batch, "global_batch": batch * world, "L": cfg["L"], "images_per_sample": 1,
                   "parallelism": f"dp{world}", "random_init": True, "gates": 0.5,
                   "numerics": "bf16 operands, fp32 accumulate / softmax / LayerNorm stats (reference's autocast(bf16) "
                               "recipe; bf16-level tolerances in tests/, the 1e-3/1e-5 fp32-grade mode is not timed)",
                   "launch": "eager" if args.no_graph else "two CUDA graphs per step (frozen CLIP forward | perceiver + gated "
                             "fwd/bwd), replayed" + ("; the single NCCL gradient all-reduce runs between them, overlapped "
                             "with the CLIP forward of the next batch" if world > 1 else ""),
                   "weights": "fp32 master, bf16 compute copies re-cast every step; fp32 `.grad` views of one flat buffer" +
                              ("; the Linear weights' wgrad epilogues write the bf16 wire buffer of the all-reduce, one up-cast "
                               "after it" if comm_mode == "bf16-direct" else ""),
                   "cache": "per-step working set (2.4 GB bf16 weights + activations) >> 126 MB L2; no explicit flush",
                   "grad_allreduce_bytes": comm_bytes,
                   "grad_allreduce_dtype": comm_mode, "nccl_registered_buffer": bool(args.nccl_registered),
                   "grad_allreduce_op": ("sum, 1/N folded into the up-cast" if (args.reduce_op == "sum" and comm_mode != "fp32") else "avg")},
        "e2e": {"value": round(e2e_value, 2), "unit": "samples/s", "ms_per_step": round(ms_e2e / args.steps, 3),
                "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": 4, "h2d_overlapped_with_previous_step": bool(args.e2e_prefetch)},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "roofline": {"bound": "tensor",
                     "kernel": "otb::gemm2_bf16_kernel (tcgen05 cta_group::2 / TMA) — the six 4096<->16384 FFN GEMM classes "
                               "(fwd, dgrad, wgrad) of the gated blocks, 48 launches/step",
                     "achieved": round(ach, 1), "peak": peak_tf, "unit": "TFLOP/s",
                     "frac": round(ach / peak_tf, 4) if peak_tf else None,
                     "traffic": 259.1e6, "traffic_note": "dram read+write of one 2048x16384x4096 GELU+aux launch of "
                                                         "gemm2_bf16_kernel (shipped epilogue), ncu --set full, "
                                                         "profiles/r02_final_ncu_gemm_and_fused.md (algorithmic 285 MB; "
                                                         "tensor pipe 82.7 % active)",
                     "peak_source": peak_src, "frac_of_sustained_peak": round(ach / peak_sus, 4),
                     "per_class_us": dom["per_class_us"], "flops_per_launch_avg": dom["flops_avg"],
                     "share_of_step": round(8 * dom["sum_ms"] / step_ms, 3),
                     "all_gemms_eager_event_ms": round(g_ms, 3), "all_gemm_launches": len(prof),
                     "step_algorithmic_tflops": round(fl * batch / (step_ms * 1e-3) / 1e12, 1),
                     "step_frac_of_sustained_peak": round(fl * batch / (step_ms * 1e-3) / 1e12 / peak_sus, 4),
                     "hbm_bound_kernels": {"peak_gbs": hbm_gbs, "peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks
                                           else "fallback 6600 GB/s", "timing": "CUDA-graph replay, CUDA events, "
                                           "rotating operand sets > L2 (cold operands)", "kernels": hbm_rows}},
    }
    if comm_alone is not None:
        out["allreduce_alone"] = comm_alone
    if check is not None:
        out["self_check"] = check
    if extras is not None:
        out["extras"] = extras
    if world == 1 and not args.no_cpu_baseline:
        out["cpu_baseline"] = cpu_sample(steps=3, warmup=1, batch=batch, budget_s=120.0)
    print(json.dumps(out), flush=True)
    if world > 1:
        dist.destroy_process_group()


# ---- the CPU arm: the reference's modules (or the oracle port) on the host cores -----------------
def _cpu_inputs(batch, g):
    vision_x = torch.randn(batch, BASE_CFG["T"], BASE_CFG["F"], 3, BASE_CFG["img"], BASE_CFG["img"], generator=g)
    hidden = torch.randn(batch, BASE_CFG["L"], BASE_CFG["D"], generator=g).requires_grad_(True)
    loc = torch.zeros(batch, BASE_CFG["L"], dtype=torch.bool)
    loc[:, 0] = True
    return vision_x, hidden, loc


def _cpu_reference_step(batch):
    """One M1 step built from the reference's own classes (BASELINE.md §2): returns a zero-argument callable."""
    from oracle import ref_shims
    mod = ref_shims.load_reference_otter()
    from transformers import CLIPVisionConfig, CLIPVisionModel
    torch.manual_seed(SEED)
    vc = CLIPVisionConfig(hidden_size=1024, intermediate_size=4096, num_hidden_layers=BASE_CFG["clip_layers"],
                          num_attention_heads=16, image_size=BASE_CFG["img"], patch_size=14, hidden_act="quick_gelu")
    clip = CLIPVisionModel(vc).requires_grad_(False).eval()
    perceiver = mod.OtterPerceiverResampler(dim=BASE_CFG["vis_dim"])
    gated = [mod.OtterGatedCrossAttentionBlock(dim=BASE_CFG["D"], dim_visual=BASE_CFG["vis_dim"])
             for _ in range(BASE_CFG["n_gated"])]
    with torch.no_grad():
        for gb in gated:
            gb.attn_gate.fill_(0.5)
            gb.ff_gate.fill_(0.5)
    params = list(perceiver.parameters()) + [p for gb in gated for p in gb.parameters()]
    vision_x, hidden, loc = _cpu_inputs(batch, torch.Generator().manual_seed(SEED))

    def one():
        for p in params:
            p.grad = None
        b, T, Fr = vision_x.shape[:3]
        with torch.no_grad():                                               # modeling_otter.py:989-992
            feats = clip(vision_x.reshape(b * T * Fr, *vision_x.shape[3:]))[0][:, 1:, :]
        feats = feats.reshape(b, T, Fr, feats.shape[1], feats.shape[2])
        media = perceiver(feats)                                            # :994
        x = hidden
        for gb in gated:                                                    # :380-393 per block
            x = gb(x, media, media_locations=loc, attend_previous=True)
        loss = x.float().pow(2).mean()
        loss.backward()
        return loss.item()

    return one


def _cpu_port_step(batch):
    from oracle import restatement as R
    g = torch.Generator().manual_seed(SEED)
    D, Dv = BASE_CFG["D"], BASE_CFG["vis_dim"]

    def lin(o, i):
        return torch.randn(o, i, generator=g) / i ** 0.5

    def ln(d):
        return torch.ones(d), torch.zeros(d)

    clip_p = {}
    pre = "vision_model."
    clip_p[pre + "embeddings.patch_embedding.weight"] = torch.randn(Dv, 3, 14, 14, generator=g) * 0.02
    clip_p[pre + "embeddings.class_embedding"] = torch.randn(Dv, generator=g) * 0.02
    clip_p[pre + "embeddings.position_embedding.weight"] = torch.randn(257, Dv, generator=g) * 0.02
    clip_p[pre + "pre_layrnorm.weight"], clip_p[pre + "pre_layrnorm.bias"] = ln(Dv)
    for i in range(BASE_CFG["clip_layers"]):
        lp = f"{pre}encoder.layers.{i}."
        for nm in ("q_proj", "k_proj", "v_proj", "out_proj"):
            clip_p[lp + f"self_attn.{nm}.weight"], clip_p[lp + f"self_attn.{nm}.bias"] = lin(Dv, Dv), torch.zeros(Dv)
        clip_p[lp + "layer_norm1.weight"], clip_p[lp + "layer_norm1.bias"] = ln(Dv)
        clip_p[lp + "layer_norm2.weight"], clip_p[lp + "layer_norm2.bias"] = ln(Dv)
        clip_p[lp + "mlp.fc1.weight"], clip_p[lp + "mlp.fc1.bias"] = lin(4 * Dv, Dv), torch.zeros(4 * Dv)
        clip_p[lp + "mlp.fc2.weight"], clip_p[lp + "mlp.fc2.bias"] = lin(Dv, 4 * Dv), torch.zeros(Dv)
    perc_p = {"latents": torch.randn(64, Dv, generator=g)}
    perc_p["norm.weight"], perc_p["norm.bias"] = ln(Dv)
    for i in range(6):
        lp = f"layers.{i}."
        for nm in ("norm_media", "norm_latents", "feed_forward.0"):
            perc_p[lp + nm + ".weight"], perc_p[lp + nm + ".bias"] = ln(Dv)
        perc_p[lp + "to_q.weight"], perc_p[lp + "to_kv.weight"], perc_p[lp + "to_out.weight"] = lin(512, Dv), lin(1024, Dv), lin(Dv, 512)
        perc_p[lp + "feed_forward.1.weight"], perc_p[lp + "feed_forward.3.weight"] = lin(4 * Dv, Dv), lin(Dv, 4 * Dv)
    gated_ps = []
    for _ in range(BASE_CFG["n_gated"]):
        gp = {"attn_gate": torch.tensor([0.5]), "ff_gate": torch.tensor([0.5])}
        gp["attn.norm.weight"], gp["attn.norm.bias"] = ln(D)
        gp["feed_forward.0.weight"], gp["feed_forward.0.bias"] = ln(D)
        gp["attn.to_q.weight"], gp["attn.to_kv.weight"], gp["attn.to_out.weight"] = lin(512, D), lin(1024, Dv), lin(D, 512)
        gp["feed_forward.1.weight"], gp["feed_forward.3.weight"] = lin(4 * D, D), lin(D, 4 * D)
        gated_ps.append(gp)
    train = [t for t in perc_p.values()] + [t for gp in gated_ps for t in gp.values()]
    for t in train:
        t.requires_grad_(True)
    vision_x, hidden, loc = _cpu_inputs(batch, g)

    def one():
        for t in train:
            t.grad = None
        out, _ = R.m1_forward(vision_x, hidden, loc, clip_p, perc_p, gated_ps)
        loss = out.float().pow(2).mean()
        loss.backward()
        return loss.item()

    return one


def cpu_sample(steps, warmup, batch, budget_s=None, force_port=False):
    """Time M1 steps of the reference math on the host cores (fp32, every usable thread) at the GPU arm's batch.
    `budget_s` bounds the timed part: after the first (warm-up) step the step count is cut to fit, never below 1
    (3 when the budget allows) — the count actually run is reported."""
    from oracle import ref_shims
    cores = host_cores()               # affinity / cgroup quota aware (the GPU box: 128 visible, quota 16)
    torch.set_num_threads(cores)
    kind, origin = "port", "oracle/restatement.py"
    one = None
    if not force_port and ref_shims.reference_available():
        try:
            one = _cpu_reference_step(batch)
            kind, origin = "reference", ref_shims.reference_origin()
        except Exception as e:          # e.g. a transformers version the reference cannot import against
            print(f"[bench] reference modules unavailable ({type(e).__name__}: {e}); timing the oracle port",
                  file=sys.stderr, flush=True)
    if one is None:
        one = _cpu_port_step(batch)
    t_warm = None
    for _ in range(warmup):
        t0 = time.perf_counter()
        one()
        t_warm = time.perf_counter() - t0
    if budget_s is not None and t_warm:
        steps = max(1, min(steps, int(budget_s / t_warm)))
    t0 = time.perf_counter()
    for _ in range(steps):
        one()
    dt = time.perf_counter() - t0
    return {"value": round(batch * steps / dt, 4), "unit": "samples/s", "cores": cores, "kind": kind, "steps": steps,
            "warmup": warmup, "batch": batch,
            "sample": f"{steps} timed step(s) after {warmup} warm-up of the same M1 workload at batch {batch}, L "
                      f"{BASE_CFG['L']} (fp32, torch CPU, {cores} threads; {origin}), {dt / steps:.2f} s/step"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    batch = args.ref_batch if args.ref_batch else args.per_gpu_batch
    res = cpu_sample(steps=args.steps, warmup=min(args.warmup, 1), batch=batch, budget_s=args.ref_budget_s,
                     force_port=args.ref_port)
    dt_ms = 1e3 * batch / res["value"]
    out = {"impl": "reference", "metric": METRIC, "value": res["value"],
           "unit": "samples/s", "n_gpus": args.gpus, "steps": res["steps"], "steps_requested": args.steps,
           "warmup": min(args.warmup, 1),
           "ms_per_step": round(dt_ms, 1), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
           "dtype": "f32", "data": "synthetic",
           "config": {"workload": "OTTER-Image-MPT7B shape (BASELINE configs[1]), M1 hot path: CLIP ViT-L/14 fwd -> "
                                  "perceiver(6x64 latents) -> 8 gated x-attn blocks D=4096, fwd+bwd — the reference's "
                                  "CPU path on the host cores (rank 0 only; CPU work does not scale with --gpus)",
                      "per_gpu_batch": batch, "global_batch": batch, "L": BASE_CFG["L"], "images_per_sample": 1,
                      "random_init": True, "gates": 0.5,
                      "bounded": f"timed steps cut to fit {args.ref_budget_s:.0f} s after one warm-up step"},
           "cpu_baseline": res,
           "e2e": {"value": res["value"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    print(json.dumps(out), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="otter_b200", choices=["otter_b200", "reference"])
    ap.add_argument("--per-gpu-batch", type=int, default=8)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the extra configurations (c3, L sweep, batch 32, c5)")
    ap.add_argument("--no-self-check", action="store_true", help="skip the post-timing oracle check at batch 1")
    ap.add_argument("--no-kernel-rooflines", action="store_true", help="skip the HBM-bound kernel timings")
    ap.add_argument("--no-graph", action="store_true", help="launch every kernel eagerly instead of replaying a CUDA graph")
    ap.add_argument("--no-multi-cast", dest="multi_cast", action="store_false",
                    help="re-derive the bf16 weight copies with one cast launch per weight instead of one multi-tensor launch")
    ap.set_defaults(multi_cast=True)
    ap.add_argument("--grad-comm-dtype", default="auto", choices=["auto", "fp32", "bf16", "bf16-direct"],
                    help="wire format of the single gradient all-reduce (`.grad` is fp32 either way).  bf16 halves the "
                         "payload to SURVEY.md §8e's 2.36 GB at the cost of two cast passes; bf16-direct lets the wgrad "
                         "epilogues write the wire buffer (one up-cast after the collective).  auto = bf16-direct for N > 1")
    ap.add_argument("--e2e-prefetch", action="store_true",
                    help="e2e leg: copy the next step's inputs host->device on a copy stream while this step computes")
    ap.add_argument("--reduce-op", default="sum", choices=["sum", "avg"],
                    help="reduction of the wire-format all-reduce: sum (1/N folded into the up-cast; lets NCCL use its "
                         "in-switch NVLS algorithms) or avg (ncclAvg = pre-multiplied sum, RING only)")
    ap.add_argument("--nccl-registered", action="store_true",
                    help="allocate the flat gradient buffer from NCCL's allocator and register it (zero-copy / NVLS)")
    ap.add_argument("--seq-len", type=int, default=256, help="text length L (SURVEY.md §8d sweeps 128/256/512/1024)")
    ap.add_argument("--ref-batch", type=int, default=0, help="reference arm: batch per step (default: --per-gpu-batch)")
    ap.add_argument("--ref-budget-s", type=float, default=150.0, help="reference arm: wall-clock bound of the timed steps")
    ap.add_argument("--ref-port", action="store_true", help="reference arm: time oracle/restatement.py instead")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the last step's loss and (sampled) parameter gradients to "
                         "DIR/<name>.npy, to compare the outputs of two builds on identical inputs")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "otter_b200":
        ap.error("--dump-outputs writes what the CUDA arm computed; it does not apply to --impl reference")
    BASE_CFG["L"] = args.seq_len
    if args.impl == "reference":
        run_reference(args)
    else:
        run_cuda(args)


if __name__ == "__main__":
    main()
