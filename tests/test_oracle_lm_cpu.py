"""CPU: the frozen-LM oracle (oracle/restatement_lm.py, SURVEY.md §8f rank 1) against golden fixtures generated from the
unmodified reference MPTBlock (oracle/make_golden_lm.py, oracle/make_golden_live.py)."""
import os

import torch

from oracle import restatement_lm as R
from oracle.seeded import seeded_state, seeded_tensor

GOLD = os.path.join(os.path.dirname(__file__), "golden", "mpt_block_tiny.pt")
GOLD_LIVE = os.path.join(os.path.dirname(__file__), "golden", "mpt_block_live.pt")


def test_alibi_slopes_power_of_two_and_not():
    s8 = R.alibi_slopes(8)
    assert torch.allclose(s8, torch.tensor([2.0 ** -(i + 1) for i in range(8)]))
    s6 = R.alibi_slopes(6)                      # 8 slopes computed, odd-indexed first, then even, truncated
    full = torch.tensor([2.0 ** -(i + 1) for i in range(8)])
    assert torch.allclose(s6, torch.cat([full[1::2], full[::2]])[:6])
    b = R.alibi_key_bias(4, 5)
    assert b.shape == (4, 5) and torch.all(b[:, -1] == 0) and torch.all(b[:, 0] < 0)


def test_block_forward_and_input_grad_match_reference_golden():
    gold = torch.load(GOLD)
    for name, g in gold.items():
        B, S, D, H = g["shape"]
        x = g["x"].clone().requires_grad_(True)
        y = R.mpt_block(x, g["params"], H)
        assert torch.allclose(y, g["y"], rtol=1e-5, atol=1e-5), name
        (gx,) = torch.autograd.grad(y, x, g["gy"])
        assert torch.allclose(gx, g["gx"], rtol=1e-4, atol=1e-5), name


def test_causality_and_shift_property():
    """Outputs at position i do not depend on later tokens; the key-only ALiBi bias equals the relative-distance form."""
    g = torch.load(GOLD)["a"]
    B, S, D, H = g["shape"]
    y = R.mpt_block(g["x"], g["params"], H)
    x2 = g["x"].clone()
    x2[:, S // 2:] += 1.0
    y2 = R.mpt_block(x2, g["params"], H)
    assert torch.equal(y[:, :S // 2], y2[:, :S // 2])
    assert not torch.allclose(y[:, S // 2:], y2[:, S // 2:])


def test_against_live_reference_block():
    """Head dim 16 without biases, and with biases (generic MPT configs), vs the reference block's outputs."""
    gold = torch.load(GOLD_LIVE)
    assert any(not c["no_bias"] for c in gold.values())
    for name, c in gold.items():
        x = seeded_tensor(f"in.live.mpt.{name}", c["x_shape"], c["seed"], "randn")
        got = R.mpt_block(x, seeded_state(c["shapes"], c["seed"]), c["H"])
        assert torch.allclose(got, c["y"], rtol=1e-5, atol=1e-5), name
