"""Model name -> properties + architecture for the models the engine serves.

Property dicts (`name`, `dimensions`, `type`, `tokens`, prefixes) are the reference's registry entries
(src/marqo/s2_inference/model_registry.py:142-231 for open_clip/*, :771-788 for hf/e5-*, :630-641 and :668-679 for the
MPNet sentence encoders); `type` is rewritten to the
engine's loader types ("b200_open_clip" / "b200_hf") so that both engines can be registered side by side in
MODEL_PROPERTIES['loaders'] (model_registry.py:2133-2145).  The `arch` blocks are the shapes that live in
open_clip 2.24.0 `model_configs/*.json` and the HF `config.json` files (SURVEY.md §8)."""
from __future__ import annotations

import copy
from typing import Dict

OPENAI_MEAN = (0.48145466, 0.4578275, 0.40821073)   # src/marqo/s2_inference/clip_utils.py:32-33
OPENAI_STD = (0.26862954, 0.26130258, 0.27577711)

TYPE_OPEN_CLIP = "b200_open_clip"
TYPE_HF = "b200_hf"


def _clip_arch(embed, vw, vl, vh, patch, tw, tl, th, act="gelu"):
    return {
        "embed_dim": embed, "act": act, "mean": OPENAI_MEAN, "std": OPENAI_STD,
        "vision": {"width": vw, "layers": vl, "heads": vh, "mlp": 4 * vw, "patch": patch, "image_size": 224},
        "text": {"width": tw, "layers": tl, "heads": th, "mlp": 4 * tw, "ctx": 77, "vocab": 49408},
    }


def _bert_arch(w, layers, heads, pool="mean"):
    return {"width": w, "layers": layers, "heads": heads, "mlp": 4 * w, "vocab": 30522, "max_pos": 512,
            "type_vocab": 2, "pool": pool}


def _mpnet_arch(pool="mean"):
    # HF MPNetModel config.json of the all-mpnet-base / all_datasets_*_mpnet-base checkpoints
    return {"family": "mpnet", "width": 768, "layers": 12, "heads": 12, "mlp": 3072, "vocab": 30527, "max_pos": 514,
            "buckets": 32, "ln_eps": 1e-5, "pool": pool}


_VIT_B_32 = dict(embed=512, vw=768, vl=12, vh=12, patch=32, tw=512, tl=12, th=8)
_VIT_B_16 = dict(embed=512, vw=768, vl=12, vh=12, patch=16, tw=512, tl=12, th=8)
_VIT_L_14 = dict(embed=768, vw=1024, vl=24, vh=16, patch=14, tw=768, tl=12, th=12)


def _open_clip(name: str, dims: int, pretrained: str, shape: dict, act: str) -> dict:
    return {"name": name, "dimensions": dims, "note": "open_clip models", "type": TYPE_OPEN_CLIP,
            "pretrained": pretrained, "arch": _clip_arch(**shape, act=act)}


def _models() -> Dict[str, dict]:
    m: Dict[str, dict] = {}
    for tag in ("laion400m_e31", "laion400m_e32", "laion2b_e16", "laion2b_s34b_b79k"):
        m[f"open_clip/ViT-B-32/{tag}"] = _open_clip(f"open_clip/ViT-B-32/{tag}", 512, tag, _VIT_B_32, "gelu")
    m["open_clip/ViT-B-32/openai"] = _open_clip("open_clip/ViT-B-32/openai", 512, "openai", _VIT_B_32, "quickgelu")
    m["open_clip/ViT-B-32-quickgelu/openai"] = _open_clip("open_clip/ViT-B-32-quickgelu/openai", 512, "openai",
                                                          _VIT_B_32, "quickgelu")
    m["open_clip/ViT-B-16/openai"] = _open_clip("open_clip/ViT-B-16/openai", 512, "openai", _VIT_B_16, "quickgelu")
    m["open_clip/ViT-B-16/laion2b_s34b_b88k"] = _open_clip("open_clip/ViT-B-16/laion2b_s34b_b88k", 512,
                                                           "laion2b_s34b_b88k", _VIT_B_16, "gelu")
    for tag in ("laion400m_e31", "laion400m_e32", "laion2b_s32b_b82k"):
        m[f"open_clip/ViT-L-14/{tag}"] = _open_clip(f"open_clip/ViT-L-14/{tag}", 768, tag, _VIT_L_14, "gelu")
    m["open_clip/ViT-L-14/openai"] = _open_clip("open_clip/ViT-L-14/openai", 768, "openai", _VIT_L_14, "quickgelu")
    # (verify) upstream uses 0.5/0.5 image statistics for this tag (SURVEY.md Appendix B)
    m["open_clip/ViT-L-14/laion2b_s32b_b82k"]["arch"]["mean"] = (0.5, 0.5, 0.5)
    m["open_clip/ViT-L-14/laion2b_s32b_b82k"]["arch"]["std"] = (0.5, 0.5, 0.5)
    for short, repo, w, layers, heads, size in (("e5-small-v2", "intfloat/e5-small-v2", 384, 12, 6, 0.134),
                                                ("e5-base-v2", "intfloat/e5-base-v2", 768, 12, 12, 0.438),
                                                ("e5-large-v2", "intfloat/e5-large-v2", 1024, 24, 16, 1.34),
                                                ("e5-base", "intfloat/e5-base", 768, 12, 12, 0.438),
                                                ("e5-large", "intfloat/e5-large", 1024, 24, 16, 1.34)):
        m[f"hf/{short}"] = {"name": repo, "dimensions": w, "tokens": 512, "type": TYPE_HF, "model_size": size,
                            "text_query_prefix": "query: ", "text_chunk_prefix": "passage: ", "notes": "",
                            "arch": _bert_arch(w, layers, heads)}
    for short, repo in (("all-mpnet-base-v1", "sentence-transformers/all-mpnet-base-v1"),
                        ("all-mpnet-base-v2", "sentence-transformers/all-mpnet-base-v2"),
                        ("all_datasets_v3_mpnet-base", "flax-sentence-embeddings/all_datasets_v3_mpnet-base"),
                        ("all_datasets_v4_mpnet-base", "flax-sentence-embeddings/all_datasets_v4_mpnet-base")):
        m[f"hf/{short}"] = {"name": repo, "dimensions": 768, "tokens": 128, "type": TYPE_HF, "notes": "",
                            "arch": _mpnet_arch()}
    return m


MODELS: Dict[str, dict] = _models()


def get_model_properties(model_name: str) -> dict:
    from .errors import UnknownModelError
    if model_name not in MODELS:
        raise UnknownModelError(f"Could not find model properties in model registry for model={model_name}. "
                                f"Model is not supported by default.")
    return copy.deepcopy(MODELS[model_name])
