"""CPU: bench.py's contract pieces that need no GPU — the reference arm (CPU port of the M1 step) prints one JSON line
with the required keys, and non-zero ranks of a torchrun launch exit quietly."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_host_cores_is_positive_and_bounded():
    sys.path.insert(0, ROOT)
    import bench
    n = bench.host_cores()
    assert 1 <= n <= (os.cpu_count() or 1)


def test_reference_arm_nonzero_rank_is_silent():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2",
                          "--steps", "1", "--warmup", "0"], capture_output=True, text=True, env=env, timeout=300)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_reference_arm_json_line(tmp_path):
    """One bounded step of the CPU arm (batch 1 of the c2 workload here to keep the CPU suite short; the driver's run
    uses the GPU arm's batch 8): the reference's own modules when /root/reference or oracle/_ref is present."""
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "0", "--ref-batch", "1"], capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads(out.stdout.strip().splitlines()[-1])
    assert d["impl"] == "reference" and d["unit"] == "samples/s" and d["higher_is_better"] is True
    assert d["metric"] == "samples/sec perceiver+gated-xattn fwd+bwd" and d["value"] > 0
    sys.path.insert(0, ROOT)
    from oracle import ref_shims
    want_kind = "reference" if ref_shims.reference_available() else "port"
    assert d["cpu_baseline"]["kind"] == want_kind and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["config"]["per_gpu_batch"] == 1 and d["cpu_baseline"]["batch"] == 1
    assert d["e2e"] == {"value": d["value"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["gpu_launches"] == 0 and d["steps"] == 1


def test_allreduce_alone_record(monkeypatch):
    """bench.allreduce_alone (N > 1 only): field names and the bus-bandwidth formula, with CUDA events and the process
    group replaced by stand-ins (the real thing needs NCCL)."""
    import torch
    import torch.distributed as dist
    import bench

    class _Ev:
        def __init__(self, enable_timing=True):
            pass

        def record(self):
            pass

        def elapsed_time(self, other):
            return 50.0                     # ms for the 10 iterations

    class _Flat:
        calls = 0

        def all_reduce(self):
            _Flat.calls += 1

        def comm_nbytes(self):
            return 2_000_000_000

    class _HP:
        flat = _Flat()

    monkeypatch.setattr(torch.cuda, "Event", _Ev)
    monkeypatch.setattr(torch.cuda, "synchronize", lambda *a, **k: None)
    monkeypatch.setattr(dist, "barrier", lambda *a, **k: None)
    monkeypatch.setattr(dist, "all_reduce", lambda t, op=None: None)
    r = bench.allreduce_alone(_HP(), "cpu", 8, iters=10)
    assert _Flat.calls == 12                                    # 2 warm-up + 10 timed
    assert r["ms"] == 5.0 and r["wire_bytes"] == 2_000_000_000 and r["iters"] == 10
    assert abs(r["busbw_gbs"] - 2 * 7 / 8 * 2e9 / 5e-3 / 1e9) < 0.1      # 700 GB/s


def test_dump_outputs_files(tmp_path, monkeypatch):
    """--dump-outputs: one float32 .npy per array (the loss, every trainable parameter's gradient), large gradients
    sampled at the same positions on every run, and at the timed workload's parameter shapes under the 64 MB bound."""
    import types

    import numpy as np
    import torch
    import bench
    from otter_b200.modeling_otter import OtterGatedCrossAttentionBlock, OtterPerceiverResampler

    monkeypatch.setattr(torch.cuda, "synchronize", lambda *a, **k: None)
    monkeypatch.setattr(bench, "DUMP_SAMPLE", 1000)
    torch.manual_seed(0)
    hp = types.SimpleNamespace(loss=torch.tensor([0.25]), perceiver=OtterPerceiverResampler(dim=32, depth=1),
                               gated=torch.nn.ModuleList([OtterGatedCrossAttentionBlock(dim=64, dim_visual=32)]))
    params = [(f"grad.{pre}.{n}", p) for pre, m in (("perceiver", hp.perceiver), ("gated", hp.gated))
              for n, p in m.named_parameters()]
    for _, p in params:
        p.grad = torch.randn_like(p)
    n, nbytes = bench.dump_outputs(hp, str(tmp_path / "a"))
    bench.dump_outputs(hp, str(tmp_path / "b"))
    names = sorted(f[:-4] for f in os.listdir(tmp_path / "a"))
    assert n == len(names) == len(params) + 1 and names == sorted(["loss"] + [k for k, _ in params])
    assert np.array_equal(np.load(tmp_path / "a" / "loss.npy"), hp.loss.numpy())
    total = 4
    for name, p in params:
        a, b = np.load(tmp_path / "a" / f"{name}.npy"), np.load(tmp_path / "b" / f"{name}.npy")
        assert a.dtype == np.float32 and np.array_equal(a, b) and a.size == min(p.numel(), 1000)
        g = p.grad.reshape(-1).numpy()
        assert np.array_equal(a, g) if p.numel() <= 1000 else np.isin(a, g).all()
        total += a.nbytes
    assert any(p.numel() > 1000 for _, p in params) and nbytes == total
    monkeypatch.undo()
    with torch.device("meta"):                                  # the timed workload's modules, shapes only
        per = OtterPerceiverResampler(dim=bench.BASE_CFG["vis_dim"])
        gated = [OtterGatedCrossAttentionBlock(dim=bench.BASE_CFG["D"], dim_visual=bench.BASE_CFG["vis_dim"])
                 for _ in range(bench.BASE_CFG["n_gated"])]
    sizes = [p.numel() for m in [per] + gated for p in m.parameters()]
    assert 4 * (1 + sum(min(s, bench.DUMP_SAMPLE) for s in sizes)) <= 64 * 2 ** 20
