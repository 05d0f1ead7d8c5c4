"""Checkpoint plumbing for the encoders: state-dict loading and random initialisation.

The engine consumes parameters under their checkpoint names (open_clip state_dict names for CLIP, HF BertModel names
for BERT, HF MPNetModel names for MPNet), so a real checkpoint loads unchanged: open_clip `*.pt/*.bin` state dicts, HF `pytorch_model.bin`, or an
`.npz` with the same keys.  `random_*` build seeded random-init weights of a given architecture (bench.py and the
service's self-test use them — there is no network for real checkpoints in the build environment)."""
from __future__ import annotations

import math
from typing import Dict

import numpy as np


def load_state_dict(path: str) -> Dict[str, np.ndarray]:
    """.npz, torch .pt/.bin/.pth or .safetensors -> {name: fp32 ndarray}."""
    p = str(path)
    if p.endswith(".npz"):
        with np.load(p) as z:
            return {k: np.asarray(z[k], dtype=np.float32) for k in z.files}
    if p.endswith(".safetensors"):
        from safetensors.numpy import load_file  # optional dependency
        return {k: np.asarray(v, dtype=np.float32) for k, v in load_file(p).items()}
    import torch
    sd = torch.load(p, map_location="cpu", weights_only=True)
    if isinstance(sd, dict) and "state_dict" in sd and isinstance(sd["state_dict"], dict):
        sd = sd["state_dict"]
    out = {}
    for k, v in sd.items():
        if hasattr(v, "is_floating_point") and v.is_floating_point():
            out[k[len("module."):] if k.startswith("module.") else k] = v.float().numpy()
    return out


def strip_hf_prefix(sd: Dict[str, np.ndarray], prefix: str = "bert.") -> Dict[str, np.ndarray]:
    """HF checkpoints saved from BertForXxx / MPNetForXxx carry a 'bert.' / 'mpnet.' prefix; BertModel and MPNetModel
    checkpoints do not."""
    if any(k.startswith(prefix) for k in sd):
        return {k[len(prefix):]: v for k, v in sd.items() if k.startswith(prefix)}
    return sd


def _rng(seed):
    return np.random.default_rng(seed)


def _lin(g, out_f, in_f, gain=1.0):
    return (g.standard_normal((out_f, in_f), dtype=np.float32) * np.float32(gain / math.sqrt(in_f)))


def _vec(g, n, std=0.1, mean=0.0):
    return (mean + std * g.standard_normal(n, dtype=np.float32)).astype(np.float32)


def _clip_blocks(g, prefix, t, sd):
    w, mlp, L = t["width"], t["mlp"], t["layers"]
    rg = 1.0 / math.sqrt(2.0 * L)
    for i in range(L):
        p = f"{prefix}transformer.resblocks.{i}."
        sd[p + "ln_1.weight"] = _vec(g, w, 0.1, 1.0)
        sd[p + "ln_1.bias"] = _vec(g, w)
        sd[p + "attn.in_proj_weight"] = _lin(g, 3 * w, w, 1.5)
        sd[p + "attn.in_proj_bias"] = _vec(g, 3 * w)
        sd[p + "attn.out_proj.weight"] = _lin(g, w, w, rg)
        sd[p + "attn.out_proj.bias"] = _vec(g, w)
        sd[p + "ln_2.weight"] = _vec(g, w, 0.1, 1.0)
        sd[p + "ln_2.bias"] = _vec(g, w)
        sd[p + "mlp.c_fc.weight"] = _lin(g, mlp, w)
        sd[p + "mlp.c_fc.bias"] = _vec(g, mlp)
        sd[p + "mlp.c_proj.weight"] = _lin(g, w, mlp, rg)
        sd[p + "mlp.c_proj.bias"] = _vec(g, w)


def random_clip_weights(arch: dict, seed: int = 1234) -> Dict[str, np.ndarray]:
    g = _rng(seed)
    sd: Dict[str, np.ndarray] = {}
    v, t, E = arch.get("vision"), arch.get("text"), arch["embed_dim"]
    if v:
        w, p = v["width"], v["patch"]
        grid = v.get("image_size", 224) // p
        sd["visual.conv1.weight"] = g.standard_normal((w, 3, p, p), dtype=np.float32) / np.float32(math.sqrt(3 * p * p))
        sd["visual.class_embedding"] = _vec(g, w, 0.5)
        sd["visual.positional_embedding"] = 0.5 * g.standard_normal((grid * grid + 1, w), dtype=np.float32)
        sd["visual.ln_pre.weight"] = _vec(g, w, 0.1, 1.0)
        sd["visual.ln_pre.bias"] = _vec(g, w)
        _clip_blocks(g, "visual.", v, sd)
        sd["visual.ln_post.weight"] = _vec(g, w, 0.1, 1.0)
        sd["visual.ln_post.bias"] = _vec(g, w)
        sd["visual.proj"] = g.standard_normal((w, E), dtype=np.float32) / np.float32(math.sqrt(w))
    if t:
        w = t["width"]
        sd["token_embedding.weight"] = g.standard_normal((t["vocab"], w), dtype=np.float32)
        sd["positional_embedding"] = 0.5 * g.standard_normal((t["ctx"], w), dtype=np.float32)
        _clip_blocks(g, "", t, sd)
        sd["ln_final.weight"] = _vec(g, w, 0.1, 1.0)
        sd["ln_final.bias"] = _vec(g, w)
        sd["text_projection"] = g.standard_normal((w, E), dtype=np.float32) / np.float32(math.sqrt(w))
    return sd


def random_bert_weights(arch: dict, seed: int = 1234) -> Dict[str, np.ndarray]:
    g = _rng(seed)
    w, mlp = arch["width"], arch["mlp"]
    sd: Dict[str, np.ndarray] = {}
    sd["embeddings.word_embeddings.weight"] = g.standard_normal((arch["vocab"], w), dtype=np.float32)
    sd["embeddings.position_embeddings.weight"] = 0.5 * g.standard_normal((arch.get("max_pos", 512), w), dtype=np.float32)
    sd["embeddings.token_type_embeddings.weight"] = 0.5 * g.standard_normal((arch.get("type_vocab", 2), w), dtype=np.float32)
    sd["embeddings.LayerNorm.weight"] = _vec(g, w, 0.1, 1.0)
    sd["embeddings.LayerNorm.bias"] = _vec(g, w)
    for i in range(arch["layers"]):
        p = f"encoder.layer.{i}."
        for nm in ("query", "key", "value"):
            sd[p + f"attention.self.{nm}.weight"] = _lin(g, w, w, 1.5)
            sd[p + f"attention.self.{nm}.bias"] = _vec(g, w)
        sd[p + "attention.output.dense.weight"] = _lin(g, w, w)
        sd[p + "attention.output.dense.bias"] = _vec(g, w)
        sd[p + "attention.output.LayerNorm.weight"] = _vec(g, w, 0.1, 1.0)
        sd[p + "attention.output.LayerNorm.bias"] = _vec(g, w)
        sd[p + "intermediate.dense.weight"] = _lin(g, mlp, w)
        sd[p + "intermediate.dense.bias"] = _vec(g, mlp)
        sd[p + "output.dense.weight"] = _lin(g, w, mlp)
        sd[p + "output.dense.bias"] = _vec(g, w)
        sd[p + "output.LayerNorm.weight"] = _vec(g, w, 0.1, 1.0)
        sd[p + "output.LayerNorm.bias"] = _vec(g, w)
    return sd


def random_mpnet_weights(arch: dict, seed: int = 1234) -> Dict[str, np.ndarray]:
    """Seeded random weights under HF MPNetModel parameter names (relative-attention bias [32, heads] included)."""
    g = _rng(seed)
    w, mlp = arch["width"], arch["mlp"]
    sd: Dict[str, np.ndarray] = {}
    sd["embeddings.word_embeddings.weight"] = g.standard_normal((arch["vocab"], w), dtype=np.float32)
    sd["embeddings.position_embeddings.weight"] = 0.5 * g.standard_normal((arch.get("max_pos", 514), w), dtype=np.float32)
    sd["embeddings.LayerNorm.weight"] = _vec(g, w, 0.1, 1.0)
    sd["embeddings.LayerNorm.bias"] = _vec(g, w)
    for i in range(arch["layers"]):
        p = f"encoder.layer.{i}."
        for nm in ("q", "k", "v"):
            sd[p + f"attention.attn.{nm}.weight"] = _lin(g, w, w, 1.5)
            sd[p + f"attention.attn.{nm}.bias"] = _vec(g, w)
        sd[p + "attention.attn.o.weight"] = _lin(g, w, w)
        sd[p + "attention.attn.o.bias"] = _vec(g, w)
        sd[p + "attention.LayerNorm.weight"] = _vec(g, w, 0.1, 1.0)
        sd[p + "attention.LayerNorm.bias"] = _vec(g, w)
        sd[p + "intermediate.dense.weight"] = _lin(g, mlp, w)
        sd[p + "intermediate.dense.bias"] = _vec(g, mlp)
        sd[p + "output.dense.weight"] = _lin(g, w, mlp)
        sd[p + "output.dense.bias"] = _vec(g, w)
        sd[p + "output.LayerNorm.weight"] = _vec(g, w, 0.1, 1.0)
        sd[p + "output.LayerNorm.bias"] = _vec(g, w)
    sd["encoder.relative_attention_bias.weight"] = _vec(g, 32 * arch["heads"], 1.0).reshape(32, arch["heads"])
    return sd
