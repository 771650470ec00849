"""GPU: the drop-in boundary exercised the way the reference's own callers use it.

  * the reference's `forward_pass` (pipeline/train/instruction_following.py:73-103): the model call it makes for an Otter
    model (recorded by oracle/make_golden_live.py in caller_functions.pt: which inputs reach which keyword, in which
    dtype, which output element is the loss) replayed on otter_b200's OtterForConditionalGeneration — the loss must
    equal the one the same function returned for the reference model (fixture forward_pass_otter.pt);
  * the OpenFlamingo twin classes (modeling_flamingo.py:87-985) under their own names, against a reference Flamingo
    golden and the reference's state-dict keys / trainable set;
  * OtterForConditionalGeneration over an MPT text config (class-name dispatch modeling_otter.py:500-509), with this
    repo's MPTForCausalLM (frozen decoder layers on the otter_b200 kernels) — SURVEY.md §8f rank 1, harness mode M2.
Production numerics (bf16 operands): tolerances as in tests/test_modules_gpu.py.
"""
import os
import types

import pytest
import torch

from oracle.ref_shims import FakeTokenizer
from oracle.seeded import load_seeded_, seeded_tensor

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")
DEV = "cuda:0"
EMB_KINDS = {"perceiver.latents": "randn",
             "vision_encoder.vision_model.embeddings.class_embedding": "emb",
             "vision_encoder.vision_model.embeddings.position_embedding.weight": "emb",
             "lang_encoder.model.embed_tokens.weight": "emb",
             "lang_encoder.transformer.wte.weight": "emb"}
VKEYS = ("hidden_size", "intermediate_size", "num_hidden_layers", "num_attention_heads", "image_size", "patch_size",
         "hidden_act")
LKEYS = ("vocab_size", "hidden_size", "intermediate_size", "num_hidden_layers", "num_attention_heads",
         "num_key_value_heads", "max_position_embeddings")


def gold(name):
    return torch.load(os.path.join(GOLD, name), map_location="cpu", weights_only=False)


def _llama_cfg(g, cfg_cls, **kw):
    from transformers import LlamaConfig
    td = LlamaConfig(**{k: v for k, v in g["text_config"].items() if k in LKEYS}).to_dict()
    td["_name_or_path"] = "llama-tiny"
    td["architectures"] = ["LlamaForCausalLM"]
    cfg = cfg_cls(vision_config={k: v for k, v in g["vision_config"].items() if k in VKEYS}, text_config=td,
                  cross_attn_every_n_layers=2, **kw)
    cfg.text_config._name_or_path = "llama-tiny"
    cfg.text_config.architectures = ["LlamaForCausalLM"]
    return cfg


def _check(model, out, g, what, loss_tol=2e-2):
    from test_modules_gpu import check_grads, check_out
    assert abs(out.loss.item() - g["loss"].item()) <= loss_tol * abs(g["loss"].item()), (what, out.loss.item(), g["loss"].item())
    if "logits" in g:
        check_out(out.logits, g["logits"], f"{what} logits", fro=2e-2, mx=6e-2)
    out.loss.backward()
    check_grads(model.named_parameters(), g["grads"], what, norm_tol=5e-2, samp_tol=1e-1, gate_tol=0.12)


def test_reference_forward_pass_runs_on_the_drop_in(monkeypatch):
    from otter_b200 import otter_hf
    monkeypatch.setattr(otter_hf, "AutoTokenizer", FakeTokenizer)
    call = gold("caller_functions.pt")["forward_pass"]     # the call the reference's forward_pass makes
    assert call["model_name"] == "otter" and call["autocast_type"] == "bfloat16"   # the training recipe's cast (:99)
    g = gold("forward_pass_otter.pt")
    model = otter_hf.OtterForConditionalGeneration(_llama_cfg(g, otter_hf.OtterConfig))
    load_seeded_(model, g["seed"], kinds=EMB_KINDS)
    model.to(DEV)
    vision_x = seeded_tensor("in.fp.vision_x", (2, 1, 1, 3, 224, 224), g["input_seed"], "randn").to(DEV)
    lang_x, labels = g["lang_x"].to(DEV), g["labels"].to(DEV)
    inputs = {"images": vision_x, "input_ids": lang_x, "attention_mask": torch.ones_like(lang_x), "labels": labels}
    out = model(**{k: inputs[a["from"]].to(getattr(torch, a["dtype"])) for k, a in call["kwargs"].items()})
    loss = out[call["output_index"]]
    _check(model, types.SimpleNamespace(loss=loss), g, "forward_pass")


def test_flamingo_twin_golden_and_keys(monkeypatch):
    from otter_b200 import modeling_flamingo as MF
    from otter_b200 import otter_hf
    monkeypatch.setattr(otter_hf, "AutoTokenizer", FakeTokenizer)
    g = gold("tiny_flamingo_model.pt")
    model = MF.FlamingoForConditionalGeneration(_llama_cfg(g, MF.FlamingoConfig, use_media_placement_augmentation=False))
    assert model.media_token_id == g["media_token_id"]
    # the reference's state-dict keys / shapes and trainable set, under the Flamingo names
    ours = {k: list(v.shape) for k, v in model.state_dict().items()}
    assert ours == g["state_dict_shapes"], (sorted(set(ours) ^ set(g["state_dict_shapes"]))[:8])
    assert sorted(k for k, p in model.named_parameters() if p.requires_grad) == g["trainable"]
    assert type(model.perceiver).__name__ == "FlamingoPerceiverResampler"
    assert type(model.lang_encoder._get_decoder_layers()[1]).__name__ == "FlamingoLayer"
    assert type(model.lang_encoder._get_decoder_layers()[1].gated_cross_attn_layer).__name__ == "FlamingoGatedCrossAttentionBlock"
    load_seeded_(model, g["seed"], kinds=EMB_KINDS)
    model.to(DEV).train()
    vision_x = seeded_tensor("in.full.vision_x", (2, 1, 1, 3, 224, 224), g["seed"], "randn").to(DEV)
    lang_x, labels = g["lang_x"].to(DEV), g["labels"].to(DEV)
    out = model(vision_x=vision_x, lang_x=lang_x, attention_mask=torch.ones_like(lang_x), labels=labels)
    _check(model, out, g, "flamingo tiny")


def test_otter_over_mpt_golden(monkeypatch):
    """M2 at tiny size: CLIP -> perceiver -> [gated block + frozen MPT layer] x 2 -> norm_f -> tied LM head -> shifted CE,
    backward into the perceiver, the gated block and the tied embedding; vs the reference over ITS MPTForCausalLM."""
    from otter_b200 import otter_hf
    monkeypatch.setattr(otter_hf, "AutoTokenizer", FakeTokenizer)
    g = gold("tiny_mpt_model.pt")
    cfg = otter_hf.OtterConfig(vision_config={k: v for k, v in g["vision_config"].items() if k in VKEYS},
                               text_config=dict(g["text_config"]), cross_attn_every_n_layers=2)
    model = otter_hf.OtterForConditionalGeneration(cfg)
    assert model.lang_encoder.__class__.__name__ == "MPTForCausalLM"
    assert model.media_token_id == g["media_token_id"]
    ref_shapes = g["state_dict_shapes"]
    ours = {k: list(v.shape) for k, v in model.state_dict().items()}
    assert ours == ref_shapes, sorted(set(ours) ^ set(ref_shapes))[:8]
    assert sorted(k for k, p in model.named_parameters() if p.requires_grad) == g["trainable"]
    load_seeded_(model, g["seed"], kinds=EMB_KINDS)
    model.to(DEV).train()
    vision_x = seeded_tensor("in.mpt.vision_x", (2, 1, 1, 3, 224, 224), g["input_seed"], "randn").to(DEV)
    lang_x, labels = g["lang_x"].to(DEV), g["labels"].to(DEV)
    out = model(vision_x=vision_x, lang_x=lang_x, attention_mask=torch.ones_like(lang_x), labels=labels)
    assert out.logits.shape == (2, 32, 72)
    _check(model, out, g, "otter over mpt", loss_tol=2e-2)
