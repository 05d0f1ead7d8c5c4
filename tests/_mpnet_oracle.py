"""TEST INFRASTRUCTURE ONLY.  Torch restatement of the MPNet sentence encoders (hf/all-mpnet-base-v2 family) next to
oracle/encoders.py: HF MPNetModel forward (transformers modeling_mpnet.py: MPNetEmbeddings, MPNetEncoder with its
relative-position bias, post-LN MPNetLayer) + Marqo's pooling and normalise (hugging_face_model.py:172-214).

Like the restatements in oracle/encoders.py, `mpnet_encode` takes a `dtype` and runs on its input's device, so the GPU
tests use it in float64 as the high-precision reference.  tests/test_mpnet_oracle.py pins it against
transformers.MPNetModel built from the same weights."""
from __future__ import annotations

import math
from dataclasses import dataclass
from typing import Dict, Optional

import torch
import torch.nn.functional as F

from oracle.encoders import _cast, _lin, _vec

PADDING_IDX = 1   # MPNetEmbeddings.padding_idx: position ids start at 2, pads take position 1


@dataclass
class MpnetCfg:
    width: int
    layers: int
    heads: int
    mlp: int
    vocab: int = 30527
    max_pos: int = 514
    buckets: int = 32
    pool: str = "mean"
    ln_eps: float = 1e-5


ALL_MPNET_BASE = MpnetCfg(768, 12, 12, 3072)


def tiny_mpnet(pool: str = "mean") -> MpnetCfg:
    return MpnetCfg(128, 2, 2, 512, vocab=1000, max_pos=130, pool=pool)


def arch_of(cfg: MpnetCfg) -> dict:
    """The Encoder("mpnet", ...) config of a restated model."""
    return {"family": "mpnet", "width": cfg.width, "layers": cfg.layers, "heads": cfg.heads, "mlp": cfg.mlp,
            "vocab": cfg.vocab, "max_pos": cfg.max_pos, "buckets": cfg.buckets, "ln_eps": cfg.ln_eps, "pool": cfg.pool}


def make_mpnet_weights(cfg: MpnetCfg, seed: int = 1234, bias_std: float = 1.0) -> Dict[str, torch.Tensor]:
    """Seeded random weights under HF MPNetModel parameter names."""
    g = torch.Generator().manual_seed(seed)
    w = cfg.width
    sd: Dict[str, torch.Tensor] = {}
    sd["embeddings.word_embeddings.weight"] = torch.randn(cfg.vocab, w, generator=g)
    sd["embeddings.position_embeddings.weight"] = 0.5 * torch.randn(cfg.max_pos, w, generator=g)
    sd["embeddings.LayerNorm.weight"] = _vec(g, w, 0.1, 1.0)
    sd["embeddings.LayerNorm.bias"] = _vec(g, w)
    for i in range(cfg.layers):
        p = f"encoder.layer.{i}."
        for nm in ("q", "k", "v"):
            sd[p + f"attention.attn.{nm}.weight"] = _lin(g, w, w, 1.5)
            sd[p + f"attention.attn.{nm}.bias"] = _vec(g, w)
        sd[p + "attention.attn.o.weight"] = _lin(g, w, w)
        sd[p + "attention.attn.o.bias"] = _vec(g, w)
        sd[p + "attention.LayerNorm.weight"] = _vec(g, w, 0.1, 1.0)
        sd[p + "attention.LayerNorm.bias"] = _vec(g, w)
        sd[p + "intermediate.dense.weight"] = _lin(g, cfg.mlp, w)
        sd[p + "intermediate.dense.bias"] = _vec(g, cfg.mlp)
        sd[p + "output.dense.weight"] = _lin(g, w, cfg.mlp)
        sd[p + "output.dense.bias"] = _vec(g, w)
        sd[p + "output.LayerNorm.weight"] = _vec(g, w, 0.1, 1.0)
        sd[p + "output.LayerNorm.bias"] = _vec(g, w)
    sd["encoder.relative_attention_bias.weight"] = bias_std * torch.randn(cfg.buckets, cfg.heads, generator=g)
    return sd


def relative_position_bucket(relative_position: torch.Tensor, num_buckets: int = 32,
                             max_distance: int = 128) -> torch.Tensor:
    """MPNetEncoder.relative_position_bucket: relative_position = key - query; fp32 log as upstream."""
    n = -relative_position
    num_buckets //= 2
    ret = (n < 0).to(torch.long) * num_buckets
    n = torch.abs(n)
    max_exact = num_buckets // 2
    is_small = n < max_exact
    val_if_large = max_exact + (torch.log(n.float() / max_exact) / math.log(max_distance / max_exact)
                                * (num_buckets - max_exact)).to(torch.long)
    val_if_large = torch.min(val_if_large, torch.full_like(val_if_large, num_buckets - 1))
    return ret + torch.where(is_small, n, val_if_large)


def position_bias(rel_bias: torch.Tensor, S: int) -> torch.Tensor:
    """[H, S, S] bias of (query i, key j) = rel_bias[bucket(j - i), h] (MPNetEncoder.compute_position_bias; it always
    uses 32 buckets)."""
    pos = torch.arange(S, dtype=torch.long)
    bucket = relative_position_bucket(pos[None, :] - pos[:, None], num_buckets=32).to(rel_bias.device)
    return rel_bias[bucket].permute(2, 0, 1)


@torch.no_grad()
def mpnet_encode(sd, cfg: MpnetCfg, ids: torch.Tensor, attn_mask: Optional[torch.Tensor] = None,
                 normalize: bool = True, dtype: torch.dtype = torch.float32) -> torch.Tensor:
    """HF MPNetModel forward (eval) + Marqo's mean / CLS pooling and F.normalize.  ids: int [B, S], right padded with
    the padding id 1 where attn_mask is 0.  dtype: the compute type, on the ids' device."""
    ids = ids.long()
    B, S = ids.shape
    sd = _cast(sd, dtype, ids.device)
    if attn_mask is None:
        attn_mask = torch.ones(B, S, dtype=torch.long, device=ids.device)
    attn_mask = attn_mask.to(ids.device).long()
    w, hd = cfg.width, cfg.width // cfg.heads
    # create_position_ids_from_input_ids: non-pad tokens count up from padding_idx + 1
    not_pad = ids.ne(PADDING_IDX).long()
    position_ids = torch.cumsum(not_pad, dim=1) * not_pad + PADDING_IDX
    x = sd["embeddings.word_embeddings.weight"][ids] + sd["embeddings.position_embeddings.weight"][position_ids]
    x = F.layer_norm(x, (w,), sd["embeddings.LayerNorm.weight"], sd["embeddings.LayerNorm.bias"], cfg.ln_eps)
    bias = position_bias(sd["encoder.relative_attention_bias.weight"], S)[None]          # [1, H, S, S]
    add_mask = (1.0 - attn_mask[:, None, None, :].to(dtype)) * torch.finfo(dtype).min
    for i in range(cfg.layers):
        p = f"encoder.layer.{i}."
        q = F.linear(x, sd[p + "attention.attn.q.weight"], sd[p + "attention.attn.q.bias"])
        k = F.linear(x, sd[p + "attention.attn.k.weight"], sd[p + "attention.attn.k.bias"])
        v = F.linear(x, sd[p + "attention.attn.v.weight"], sd[p + "attention.attn.v.bias"])
        q = q.view(B, S, cfg.heads, hd).transpose(1, 2)
        k = k.view(B, S, cfg.heads, hd).transpose(1, 2)
        v = v.view(B, S, cfg.heads, hd).transpose(1, 2)
        att = (q @ k.transpose(-1, -2)) / math.sqrt(hd) + bias + add_mask
        att = att.softmax(dim=-1)
        o = (att @ v).transpose(1, 2).reshape(B, S, w)
        o = F.linear(o, sd[p + "attention.attn.o.weight"], sd[p + "attention.attn.o.bias"])
        x = F.layer_norm(o + x, (w,), sd[p + "attention.LayerNorm.weight"], sd[p + "attention.LayerNorm.bias"],
                         cfg.ln_eps)
        h = F.gelu(F.linear(x, sd[p + "intermediate.dense.weight"], sd[p + "intermediate.dense.bias"]))
        h = F.linear(h, sd[p + "output.dense.weight"], sd[p + "output.dense.bias"])
        x = F.layer_norm(h + x, (w,), sd[p + "output.LayerNorm.weight"], sd[p + "output.LayerNorm.bias"], cfg.ln_eps)
    if cfg.pool == "cls":
        emb = x[:, 0]
    else:
        last = x.masked_fill(~attn_mask[..., None].bool(), 0.0)
        emb = last.sum(dim=1) / attn_mask.sum(dim=1)[..., None]
    if normalize:
        emb = F.normalize(emb, p=2, dim=1)
    return emb


def ragged_ids(B: int, S: int, vocab: int, lengths, seed: int = 0):
    """Right-padded token ids [B, S] (real tokens never the padding id) and their attention mask."""
    g = torch.Generator().manual_seed(seed)
    ids = torch.randint(PADDING_IDX + 1, vocab, (B, S), generator=g)
    mask = torch.zeros(B, S, dtype=torch.long)
    for b, n in enumerate(lengths):
        mask[b, :n] = 1
    ids = ids.masked_fill(mask == 0, PADDING_IDX)
    return ids, mask
