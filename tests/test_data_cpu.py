"""CPU: SURVEY.md §8f rank 4 — the oracle of the image transform is pinned against Pillow + torchvision themselves
(the third-party arithmetic the reference calls: mimicit_dataset.py:132-143), the coefficient tables the CUDA kernels
consume equal the oracle's, and the host-side collate / checkpoint helpers equal the reference's own functions
(their outputs, stored by oracle/make_golden_live.py)."""
import os

import numpy as np
import pytest
import torch

from oracle import preprocess as PP

GOLD = os.path.join(os.path.dirname(__file__), "golden")
SIZES = [(480, 640), (224, 224), (100, 333), (1000, 750), (37, 41), (225, 223), (64, 2048)]


def _img(h, w, seed):
    rng = np.random.default_rng(seed)
    base = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    yy, xx = np.mgrid[0:h, 0:w]
    smooth = (127 + 100 * np.sin(xx / 17.0)[..., None] * np.cos(yy / 11.0)[..., None]).astype(np.uint8)
    return np.where(rng.random((h, w, 1)) < 0.5, base, np.broadcast_to(smooth, (h, w, 3))).astype(np.uint8)


@pytest.mark.parametrize("hw", SIZES)
def test_oracle_resize_is_bit_exact_vs_pillow_and_torchvision(hw):
    from PIL import Image
    from torchvision import transforms
    img = _img(*hw, seed=sum(hw))
    pil = Image.fromarray(img)
    assert np.array_equal(np.asarray(pil.resize((224, 224), Image.BICUBIC)), PP.resize_bicubic_u8(img, 224, 224))
    t = transforms.Compose([transforms.Resize((224, 224), interpolation=transforms.InterpolationMode.BICUBIC),
                            transforms.ToTensor(), transforms.Normalize(mean=PP.FLAMINGO_MEAN, std=PP.FLAMINGO_STD)])
    assert np.array_equal(t(pil).numpy(), PP.patch_resize_transform(img))          # fp32, bit for bit


def test_kernel_coefficient_tables_equal_the_oracle():
    from otter_b200 import data as D
    for i in (16, 37, 100, 223, 224, 225, 333, 480, 640, 750, 1000, 2048, 4000):
        b0, k0 = PP.precompute_coeffs(i, 224)
        b1, k1 = D.resample_coeffs(i, 224)
        assert np.array_equal(b0, b1) and np.array_equal(k0, k1), i
    assert D.FLAMINGO_MEAN == PP.FLAMINGO_MEAN and D.FLAMINGO_STD == PP.FLAMINGO_STD


def test_collate_and_checkpoint_helpers_equal_the_reference_functions():
    from otter_b200 import checkpoint as CK
    from otter_b200 import data as D
    g = torch.load(os.path.join(GOLD, "caller_functions.pt"), weights_only=False)
    for c in g["collate_tokens"]:
        assert torch.equal(c["out"], D.collate_tokens(c["values"], **c["kw"])), c["kw"]
    m = torch.nn.Sequential(torch.nn.Linear(4, 4), torch.nn.LayerNorm(4), torch.nn.Linear(4, 2))
    m[0].requires_grad_(False)
    assert g["get_checkpoint_keys"] == list(CK.get_checkpoint(m)) == ["1.weight", "1.bias", "2.weight", "2.bias"]
    assert D.resample_frames_fn(list(range(37)), 8) == [list(range(37))[i] for i in np.linspace(0, 36, 8, dtype=int)]


def test_trainable_checkpoint_round_trip(tmp_path):
    from otter_b200 import checkpoint as CK
    from otter_b200.modeling_otter import OtterGatedCrossAttentionBlock
    torch.manual_seed(0)
    holder = torch.nn.Module()
    holder.frozen = torch.nn.Linear(8, 8).requires_grad_(False)
    holder.gated_cross_attn_layer = OtterGatedCrossAttentionBlock(dim=64, dim_visual=32)
    path = CK.save_final_weights(holder, str(tmp_path))
    sd = torch.load(path, weights_only=True)
    assert all(k.startswith("gated_cross_attn_layer.") for k in sd) and "gated_cross_attn_layer.attn_gate" in sd
    other = torch.nn.Module()
    other.frozen = torch.nn.Linear(8, 8).requires_grad_(False)
    other.gated_cross_attn_layer = OtterGatedCrossAttentionBlock(dim=64, dim_visual=32)
    with torch.no_grad():
        other.gated_cross_attn_layer.attn_gate.fill_(3.0)
    CK.load_trainable_checkpoint(other, path)
    for (k, a), (_, b) in zip(holder.gated_cross_attn_layer.state_dict().items(),
                              other.gated_cross_attn_layer.state_dict().items()):
        assert torch.equal(a, b), k
    sd["nope.weight"] = torch.zeros(1)
    torch.save(sd, path)
    with pytest.raises(KeyError):
        CK.load_trainable_checkpoint(other, path)
