"""ORACLE — TEST INFRASTRUCTURE ONLY.  CPU fp32 restatement of the encoder arithmetic the reference calls into.
The forwards take a `dtype` (default float32) and run on their input's device: the GPU tests run them in float64 on the
GPU as a high-precision reference for every item of the production batches.

The reference only *calls* third-party forwards (none of them vendored under /root/reference):
  * open_clip_torch==2.24.0 (requirements.dev.txt:33)  `model.encode_image` / `model.encode_text`, called at
    src/marqo/core/inference/embedding_models/open_clip_model.py:258,260,277,279
  * transformers==4.41.2 (requirements.dev.txt:19)     `AutoModel` (BertModel) forward, called at
    src/marqo/core/inference/embedding_models/hugging_face_model.py:188
so the published algorithms are restated here (SURVEY.md Appendix B) and anchored on the reference's own call
sites for everything around them:
  * fp32 cast + `outputs /= outputs.norm(dim=-1, keepdim=True)` (no eps)   open_clip_model.py:256-265,
    abstract_clip_model.py:83-85
  * masked mean pool / CLS pool + F.normalize(p=2, dim=1)                  hugging_face_model.py:172-214

PARITY STATUS: "parity unpinned" for open_clip/ViT-B-32, open_clip/ViT-L-14 and hf/e5-large-v2 — the reference holds
no known-answer vector for them, and its e5-base-v2 golden (tests/core/inference/embedding_models/
test_hugging_face_model.py:15-274) needs the intfloat/e5-base-v2 checkpoint, which is not available offline.  What IS
checked (tests/test_oracle_encoders.py): this restatement == transformers' independent implementations
(CLIPVisionModelWithProjection / CLIPTextModelWithProjection / BertModel instantiated from config, same weights)
to 1e-5, and — through tests/golden/ — == the reference's own HuggingFaceModel.encode code path run here on a
config-instantiated BertModel (script: tests/golden/make_reference_golden.py).

Weights are plain dicts name -> torch.float32 tensor using the checkpoint's own parameter names (open_clip
state_dict names for CLIP, HF BertModel names for BERT), so a real checkpoint loads unchanged.
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field
from typing import Dict, Optional

import torch
import torch.nn.functional as F

# Normalize() constants: src/marqo/s2_inference/clip_utils.py:32-33
OPENAI_CLIP_MEAN = (0.48145466, 0.4578275, 0.40821073)
OPENAI_CLIP_STD = (0.26862954, 0.26130258, 0.27577711)


@dataclass
class TowerCfg:
    width: int
    layers: int
    heads: int
    mlp: int
    ctx: int = 0          # text context length
    vocab: int = 0
    image_size: int = 224
    patch: int = 0


@dataclass
class ClipCfg:
    embed_dim: int
    vision: TowerCfg
    text: TowerCfg
    act: str = "gelu"     # "gelu" (laion2b_* tags) or "quickgelu" (openai tags)
    mean: tuple = OPENAI_CLIP_MEAN
    std: tuple = OPENAI_CLIP_STD


@dataclass
class BertCfg:
    width: int
    layers: int
    heads: int
    mlp: int
    vocab: int = 30522
    max_pos: int = 512
    type_vocab: int = 2
    pool: str = "mean"    # hugging_face_model.py:205-214
    ln_eps: float = 1e-12


# model shapes: SURVEY.md §8 (open_clip 2.24.0 model_configs / HF config.json of intfloat/e5-*)
CLIP_VIT_B_32 = ClipCfg(512, TowerCfg(768, 12, 12, 3072, patch=32), TowerCfg(512, 12, 8, 2048, ctx=77, vocab=49408))
CLIP_VIT_L_14 = ClipCfg(768, TowerCfg(1024, 24, 16, 4096, patch=14), TowerCfg(768, 12, 12, 3072, ctx=77, vocab=49408))
E5_BASE = BertCfg(768, 12, 12, 3072)
E5_LARGE = BertCfg(1024, 24, 16, 4096)


def tiny_clip(act: str = "gelu") -> ClipCfg:
    return ClipCfg(128, TowerCfg(128, 2, 2, 512, patch=32, image_size=224), TowerCfg(128, 2, 2, 512, ctx=77, vocab=1000),
                   act=act)


def tiny_bert(pool: str = "mean") -> BertCfg:
    return BertCfg(128, 2, 2, 512, vocab=1000, max_pos=64, pool=pool)


# ------------------------------------------------------------------------------------------------ weights
def _lin(g, out_f, in_f, gain=1.0):
    return torch.randn(out_f, in_f, generator=g) * (gain / math.sqrt(in_f))


def _vec(g, n, std=0.1, mean=0.0):
    return mean + std * torch.randn(n, generator=g)


def _clip_blocks(g, prefix: str, t: TowerCfg, sd: Dict[str, torch.Tensor]):
    w = t.width
    res_gain = 1.0 / math.sqrt(2.0 * t.layers)
    for i in range(t.layers):
        p = f"{prefix}transformer.resblocks.{i}."
        sd[p + "ln_1.weight"] = _vec(g, w, 0.1, 1.0)
        sd[p + "ln_1.bias"] = _vec(g, w)
        sd[p + "attn.in_proj_weight"] = _lin(g, 3 * w, w, 1.5)
        sd[p + "attn.in_proj_bias"] = _vec(g, 3 * w)
        sd[p + "attn.out_proj.weight"] = _lin(g, w, w, res_gain)
        sd[p + "attn.out_proj.bias"] = _vec(g, w)
        sd[p + "ln_2.weight"] = _vec(g, w, 0.1, 1.0)
        sd[p + "ln_2.bias"] = _vec(g, w)
        sd[p + "mlp.c_fc.weight"] = _lin(g, t.mlp, w)
        sd[p + "mlp.c_fc.bias"] = _vec(g, t.mlp)
        sd[p + "mlp.c_proj.weight"] = _lin(g, w, t.mlp, res_gain)
        sd[p + "mlp.c_proj.bias"] = _vec(g, w)


def make_clip_weights(cfg: ClipCfg, seed: int = 1234) -> Dict[str, torch.Tensor]:
    """Seeded O(1)-activation random weights under open_clip state_dict names."""
    g = torch.Generator().manual_seed(seed)
    sd: Dict[str, torch.Tensor] = {}
    v, t = cfg.vision, cfg.text
    grid = v.image_size // v.patch
    sd["visual.conv1.weight"] = torch.randn(v.width, 3, v.patch, v.patch, generator=g) / math.sqrt(3 * v.patch * v.patch)
    sd["visual.class_embedding"] = _vec(g, v.width, 0.5)
    sd["visual.positional_embedding"] = 0.5 * torch.randn(grid * grid + 1, v.width, generator=g)
    sd["visual.ln_pre.weight"] = _vec(g, v.width, 0.1, 1.0)
    sd["visual.ln_pre.bias"] = _vec(g, v.width)
    _clip_blocks(g, "visual.", v, sd)
    sd["visual.ln_post.weight"] = _vec(g, v.width, 0.1, 1.0)
    sd["visual.ln_post.bias"] = _vec(g, v.width)
    sd["visual.proj"] = torch.randn(v.width, cfg.embed_dim, generator=g) / math.sqrt(v.width)
    sd["token_embedding.weight"] = torch.randn(t.vocab, t.width, generator=g)
    sd["positional_embedding"] = 0.5 * torch.randn(t.ctx, t.width, generator=g)
    _clip_blocks(g, "", t, sd)
    sd["ln_final.weight"] = _vec(g, t.width, 0.1, 1.0)
    sd["ln_final.bias"] = _vec(g, t.width)
    sd["text_projection"] = torch.randn(t.width, cfg.embed_dim, generator=g) / math.sqrt(t.width)
    return sd


def make_bert_weights(cfg: BertCfg, seed: int = 1234) -> Dict[str, torch.Tensor]:
    """Seeded random weights under HF BertModel parameter names."""
    g = torch.Generator().manual_seed(seed)
    w = cfg.width
    sd: Dict[str, torch.Tensor] = {}
    sd["embeddings.word_embeddings.weight"] = torch.randn(cfg.vocab, w, generator=g)
    sd["embeddings.position_embeddings.weight"] = 0.5 * torch.randn(cfg.max_pos, w, generator=g)
    sd["embeddings.token_type_embeddings.weight"] = 0.5 * torch.randn(cfg.type_vocab, w, generator=g)
    sd["embeddings.LayerNorm.weight"] = _vec(g, w, 0.1, 1.0)
    sd["embeddings.LayerNorm.bias"] = _vec(g, w)
    for i in range(cfg.layers):
        p = f"encoder.layer.{i}."
        for nm in ("query", "key", "value"):
            sd[p + f"attention.self.{nm}.weight"] = _lin(g, w, w, 1.5)
            sd[p + f"attention.self.{nm}.bias"] = _vec(g, w)
        sd[p + "attention.output.dense.weight"] = _lin(g, w, w)
        sd[p + "attention.output.dense.bias"] = _vec(g, w)
        sd[p + "attention.output.LayerNorm.weight"] = _vec(g, w, 0.1, 1.0)
        sd[p + "attention.output.LayerNorm.bias"] = _vec(g, w)
        sd[p + "intermediate.dense.weight"] = _lin(g, cfg.mlp, w)
        sd[p + "intermediate.dense.bias"] = _vec(g, cfg.mlp)
        sd[p + "output.dense.weight"] = _lin(g, w, cfg.mlp)
        sd[p + "output.dense.bias"] = _vec(g, w)
        sd[p + "output.LayerNorm.weight"] = _vec(g, w, 0.1, 1.0)
        sd[p + "output.LayerNorm.bias"] = _vec(g, w)
    return sd


# ------------------------------------------------------------------------------------------------ forward
def _act(x: torch.Tensor, act: str) -> torch.Tensor:
    if act == "quickgelu":
        return x * torch.sigmoid(1.702 * x)
    return F.gelu(x)  # exact erf GELU


def _mha(x: torch.Tensor, w_in, b_in, w_out, b_out, heads: int, mask: Optional[torch.Tensor]) -> torch.Tensor:
    """nn.MultiheadAttention arithmetic: fused in_proj, softmax((q / sqrt(hd)) k^T + mask) v, out_proj."""
    B, S, W = x.shape
    hd = W // heads
    qkv = F.linear(x, w_in, b_in)
    q, k, v = qkv.split(W, dim=-1)
    q = q.view(B, S, heads, hd).transpose(1, 2)
    k = k.view(B, S, heads, hd).transpose(1, 2)
    v = v.view(B, S, heads, hd).transpose(1, 2)
    att = (q / math.sqrt(hd)) @ k.transpose(-1, -2)
    if mask is not None:
        att = att + mask
    att = att.softmax(dim=-1)
    o = (att @ v).transpose(1, 2).reshape(B, S, W)
    return F.linear(o, w_out, b_out)


def _clip_tower(x: torch.Tensor, sd, prefix: str, t: TowerCfg, act: str, mask: Optional[torch.Tensor]) -> torch.Tensor:
    for i in range(t.layers):
        p = f"{prefix}transformer.resblocks.{i}."
        h = F.layer_norm(x, (t.width,), sd[p + "ln_1.weight"], sd[p + "ln_1.bias"], 1e-5)
        x = x + _mha(h, sd[p + "attn.in_proj_weight"], sd[p + "attn.in_proj_bias"], sd[p + "attn.out_proj.weight"],
                     sd[p + "attn.out_proj.bias"], t.heads, mask)
        h = F.layer_norm(x, (t.width,), sd[p + "ln_2.weight"], sd[p + "ln_2.bias"], 1e-5)
        h = _act(F.linear(h, sd[p + "mlp.c_fc.weight"], sd[p + "mlp.c_fc.bias"]), act)
        x = x + F.linear(h, sd[p + "mlp.c_proj.weight"], sd[p + "mlp.c_proj.bias"])
    return x


def _l2_normalize_clip(out: torch.Tensor) -> torch.Tensor:
    # abstract_clip_model.py:83-85 + open_clip_model.py:262-265: no epsilon
    return out / out.norm(dim=-1, keepdim=True)


def _cast(sd, dtype: torch.dtype, device: torch.device):
    """The weights in the compute type on the input's device (no copy when they already are)."""
    return {k: v.to(device=device, dtype=dtype) for k, v in sd.items()}


@torch.no_grad()
def clip_encode_image(sd, cfg: ClipCfg, pixels: torch.Tensor, normalize: bool = True,
                      dtype: torch.dtype = torch.float32) -> torch.Tensor:
    """pixels: fp32 [B,3,S,S] already preprocessed.  open_clip VisionTransformer forward (eval), then Marqo's cast +
    L2 normalise.  dtype: the compute type (float64 gives a high-precision reference; the output keeps it); the
    weights are cast to it on the pixels' device."""
    v = cfg.vision
    sd = _cast(sd, dtype, pixels.device)
    x = F.conv2d(pixels.to(dtype), sd["visual.conv1.weight"], None, stride=v.patch)  # [B, W, g, g]
    B = x.shape[0]
    x = x.reshape(B, v.width, -1).permute(0, 2, 1)                                 # [B, g*g, W]
    cls = sd["visual.class_embedding"].expand(B, 1, v.width)
    x = torch.cat([cls, x], dim=1) + sd["visual.positional_embedding"]
    x = F.layer_norm(x, (v.width,), sd["visual.ln_pre.weight"], sd["visual.ln_pre.bias"], 1e-5)
    x = _clip_tower(x, sd, "visual.", v, cfg.act, None)
    pooled = F.layer_norm(x[:, 0], (v.width,), sd["visual.ln_post.weight"], sd["visual.ln_post.bias"], 1e-5)
    out = (pooled @ sd["visual.proj"]).to(dtype)
    return _l2_normalize_clip(out) if normalize else out


@torch.no_grad()
def clip_encode_text(sd, cfg: ClipCfg, ids: torch.Tensor, normalize: bool = True,
                     dtype: torch.dtype = torch.float32) -> torch.Tensor:
    """ids: int [B, ctx].  open_clip text tower: causal mask, ln_final, EOT (= arg-max id) pooling, projection.
    dtype: the compute type, on the ids' device (as for clip_encode_image)."""
    t = cfg.text
    ids = ids.long()
    B, S = ids.shape
    sd = _cast(sd, dtype, ids.device)
    x = sd["token_embedding.weight"][ids] + sd["positional_embedding"][:S]
    mask = torch.full((S, S), float("-inf"), dtype=dtype, device=ids.device).triu_(1)
    x = _clip_tower(x, sd, "", t, cfg.act, mask)
    x = F.layer_norm(x, (t.width,), sd["ln_final.weight"], sd["ln_final.bias"], 1e-5)
    pooled = x[torch.arange(B, device=ids.device), ids.argmax(dim=-1)]
    out = (pooled @ sd["text_projection"]).to(dtype)
    return _l2_normalize_clip(out) if normalize else out


@torch.no_grad()
def bert_encode(sd, cfg: BertCfg, ids: torch.Tensor, attn_mask: Optional[torch.Tensor] = None,
                normalize: bool = True, dtype: torch.dtype = torch.float32) -> torch.Tensor:
    """HF BertModel forward (post-LN, erf-GELU, additive key-padding mask) + Marqo's pooling / normalise
    (hugging_face_model.py:188-214).  dtype: the compute type, on the ids' device; the mask fill is that type's
    finfo.min, as BertModel's get_extended_attention_mask does for its own dtype."""
    ids = ids.long()
    B, S = ids.shape
    sd = _cast(sd, dtype, ids.device)
    if attn_mask is None:
        attn_mask = torch.ones(B, S, dtype=torch.long, device=ids.device)
    attn_mask = attn_mask.to(ids.device).long()
    w, hd = cfg.width, cfg.width // cfg.heads
    x = (sd["embeddings.word_embeddings.weight"][ids] + sd["embeddings.position_embeddings.weight"][:S]
         + sd["embeddings.token_type_embeddings.weight"][0])
    x = F.layer_norm(x, (w,), sd["embeddings.LayerNorm.weight"], sd["embeddings.LayerNorm.bias"], cfg.ln_eps)
    add_mask = (1.0 - attn_mask[:, None, None, :].to(dtype)) * torch.finfo(dtype).min
    for i in range(cfg.layers):
        p = f"encoder.layer.{i}."
        q = F.linear(x, sd[p + "attention.self.query.weight"], sd[p + "attention.self.query.bias"])
        k = F.linear(x, sd[p + "attention.self.key.weight"], sd[p + "attention.self.key.bias"])
        v = F.linear(x, sd[p + "attention.self.value.weight"], sd[p + "attention.self.value.bias"])
        q = q.view(B, S, cfg.heads, hd).transpose(1, 2)
        k = k.view(B, S, cfg.heads, hd).transpose(1, 2)
        v = v.view(B, S, cfg.heads, hd).transpose(1, 2)
        att = (q @ k.transpose(-1, -2)) / math.sqrt(hd) + add_mask
        att = att.softmax(dim=-1)
        o = (att @ v).transpose(1, 2).reshape(B, S, w)
        o = F.linear(o, sd[p + "attention.output.dense.weight"], sd[p + "attention.output.dense.bias"])
        x = F.layer_norm(o + x, (w,), sd[p + "attention.output.LayerNorm.weight"],
                         sd[p + "attention.output.LayerNorm.bias"], cfg.ln_eps)
        h = F.gelu(F.linear(x, sd[p + "intermediate.dense.weight"], sd[p + "intermediate.dense.bias"]))
        h = F.linear(h, sd[p + "output.dense.weight"], sd[p + "output.dense.bias"])
        x = F.layer_norm(h + x, (w,), sd[p + "output.LayerNorm.weight"], sd[p + "output.LayerNorm.bias"], cfg.ln_eps)
    if cfg.pool == "cls":
        emb = x[:, 0]                                               # _cls_pool_func, hugging_face_model.py:211-214
    else:                                                           # _average_pool_func, :205-209
        last = x.masked_fill(~attn_mask[..., None].bool(), 0.0)
        emb = last.sum(dim=1) / attn_mask.sum(dim=1)[..., None]
    if normalize:
        emb = F.normalize(emb, p=2, dim=1)                          # eps 1e-12, :194-195
    return emb


# ------------------------------------------------------------------------------------------------ preprocess
def clip_preprocess_pil(img, n_px: int = 224, mean=OPENAI_CLIP_MEAN, std=OPENAI_CLIP_STD) -> torch.Tensor:
    """The transform of src/marqo/s2_inference/clip_utils.py:48-67 (`_get_transform`), restated with the same
    torchvision ops: Resize(n_px, BICUBIC) -> CenterCrop(n_px) -> RGB -> ToTensor -> Normalize."""
    from torchvision.transforms import CenterCrop, Compose, InterpolationMode, Normalize, Resize, ToTensor
    tf = Compose([Resize(n_px, interpolation=InterpolationMode.BICUBIC), CenterCrop(n_px),
                  lambda im: im.convert("RGB"), ToTensor(), Normalize(mean, std)])
    return tf(img)


def clip_preprocess_u8(hwc_u8, n_px: int = 224, mean=OPENAI_CLIP_MEAN, std=OPENAI_CLIP_STD) -> torch.Tensor:
    """uint8 [n,H,W,3] numpy -> fp32 [n,3,n_px,n_px] through PIL exactly as the reference's download threads do
    (src/marqo/tensor_search/add_docs.py:129-134)."""
    from PIL import Image
    return torch.stack([clip_preprocess_pil(Image.fromarray(a), n_px, mean, std) for a in hwc_u8])
