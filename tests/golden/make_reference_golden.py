"""Generate tests/golden/reference_golden.npz by RUNNING THE REFERENCE'S OWN CODE in the build container
(/root/reference is mounted there and nowhere else; the GPU box only sees the committed fixture).

What is executed from /root/reference (via the import shim in _reference_import.py):
  * marqo.s2_inference.s2_inference.vectorise / _encode_without_cache / _convert_vectorized_output with a
    deterministic fake model injected into `_available_models` exactly as the reference's own unit tests do
    (tests/s2_inference/test_vectorise.py:15-49)                                                        -> (a1)
  * marqo.core.inference.embedding_models.hugging_face_model.HuggingFaceModel.encode on a config-instantiated
    transformers BertModel with the oracle's seeded weights and a synthetic WordPiece vocabulary      -> (a5)
  * marqo.core.inference.embedding_models.open_clip_model.OPEN_CLIP.encode_image / encode_text with `self.model`
    = transformers' CLIP towers carrying the oracle's weights (open_clip itself is not installed)      -> (a3, a4)
  * marqo.s2_inference.clip_utils._get_transform on seeded random images                               -> (a2)
  * marqo.core.inference.tensor_fields_container.MultiModalTensorFieldContent.tensor_field_embeddings  -> (a7)
  * marqo.core.inference.image_download._is_image on typed inputs                                      -> (a6)

Caveat recorded in the fixture: transformers here is 5.5.0 (reference pins 4.41.2), torch 2.11 (pins 1.12.1).

Run:  python tests/golden/make_reference_golden.py
"""
import hashlib
import json
import os
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, HERE)
sys.path.insert(0, ROOT)

import _reference_import as RI  # noqa: E402

stubbed = RI.install()
import torchaudio  # noqa: E402

if not hasattr(torchaudio, "set_audio_backend"):
    torchaudio.set_audio_backend = lambda *a, **k: None

import torch  # noqa: E402

from oracle import encoders as E  # noqa: E402

out = {}
meta = {}

# ------------------------------------------------------------------------------------------------ (a1) vectorise shell
import marqo.s2_inference.s2_inference as s2  # noqa: E402
from marqo.s2_inference.multimodal_model_load import Modality  # noqa: E402


class FakeModel:
    """Deterministic stand-in: row i of the output encodes the batch it arrived in, its position and its length."""

    def __init__(self):
        self.calls = []

    def encode(self, content, normalize=True, **kwargs):
        items = [content] if isinstance(content, str) else list(content)
        self.calls.append(len(items))
        rows = [[float(len(self.calls)), float(j), float(len(str(it))), 1.0 if normalize else 0.0]
                for j, it in enumerate(items)]
        return np.asarray(rows, dtype=np.float32)


props = {"name": "fake", "dimensions": 4, "type": "hf", "tokens": 128}
key = s2._create_model_cache_key("fake", "cpu", props)
meta["cache_key_example"] = key
fake = FakeModel()
s2._available_models[key] = {"model": fake, "most_recently_used_time": 0, "model_size": 1}
content = [f"item number {i} " + "x" * (i % 7) for i in range(37)]
os.environ["MARQO_MAX_VECTORISE_BATCH_SIZE"] = "16"
res16 = s2._encode_without_cache(key, content, True, Modality.TEXT)
calls16 = list(fake.calls)
fake.calls.clear()
os.environ["MARQO_MAX_VECTORISE_BATCH_SIZE"] = "5"
res5 = s2._encode_without_cache(key, content, False, Modality.TEXT)
calls5 = list(fake.calls)
fake.calls.clear()
res_str = s2._encode_without_cache(key, "a single string", True, Modality.TEXT)
assert isinstance(res16, list) and isinstance(res16[0], list) and isinstance(res16[0][0], float)
out["a1_content_lengths"] = np.asarray([len(c) for c in content], dtype=np.int32)
out["a1_res16"] = np.asarray(res16, dtype=np.float64)
out["a1_res5"] = np.asarray(res5, dtype=np.float64)
out["a1_res_str"] = np.asarray(res_str, dtype=np.float64)
meta["a1_calls16"] = calls16
meta["a1_calls5"] = calls5
try:
    s2._encode_without_cache(key, [], True, Modality.TEXT)
    meta["a1_empty_error"] = None
except Exception as e:  # RuntimeError('Vectorise created an empty list of batches! ...')
    meta["a1_empty_error"] = [type(e).__name__, str(e)[:60]]
try:
    s2.vectorise("fake", ["x"], model_properties=props, device=None)
    meta["a1_no_device_error"] = None
except Exception as e:
    meta["a1_no_device_error"] = type(e).__name__
os.environ.pop("MARQO_MAX_VECTORISE_BATCH_SIZE")

# ------------------------------------------------------------------------------------------------ (a5) HuggingFaceModel.encode
from marqo.core.inference.embedding_models.hugging_face_model import HuggingFaceModel  # noqa: E402
from transformers import BertConfig, BertModel, BertTokenizer  # noqa: E402

for pool in ("mean", "cls"):
    cfg = E.tiny_bert(pool)
    sd = E.make_bert_weights(cfg, seed=2024)
    hc = BertConfig(vocab_size=cfg.vocab, hidden_size=cfg.width, num_hidden_layers=cfg.layers,
                    num_attention_heads=cfg.heads, intermediate_size=cfg.mlp, max_position_embeddings=cfg.max_pos,
                    type_vocab_size=cfg.type_vocab, hidden_act="gelu", layer_norm_eps=cfg.ln_eps,
                    hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0, attn_implementation="eager")
    bert = BertModel(hc, add_pooling_layer=False).eval()
    bert.load_state_dict(sd, strict=False)
    words = ["[PAD]", "[UNK]", "[CLS]", "[SEP]", "[MASK]"] + [f"w{i}" for i in range(cfg.vocab - 5)]
    with tempfile.TemporaryDirectory() as td:
        vf = os.path.join(td, "vocab.txt")
        with open(vf, "w") as f:
            f.write("\n".join(words))
        tok = BertTokenizer(vf, do_lower_case=True)
    ref_model = HuggingFaceModel.__new__(HuggingFaceModel)   # bypass load(): no network, no checkpoint
    ref_model.device = "cpu"
    ref_model._model = bert
    ref_model._tokenizer = tok
    ref_model.model_properties = type("P", (), {"tokens": 32, "pooling_method": pool})()
    ref_model._pooling_func = HuggingFaceModel._average_pool_func if pool == "mean" else HuggingFaceModel._cls_pool_func
    rng = np.random.default_rng(7)
    sentences = [" ".join(f"w{int(x)}" for x in rng.integers(0, cfg.vocab - 5, size=n)) for n in (3, 30, 11, 1, 50, 17)]
    vec = ref_model.encode(sentences, normalize=True)
    vec_un = ref_model.encode(sentences, normalize=False)
    enc = tok(sentences, padding=True, truncation=True, max_length=32, return_tensors="np")
    out[f"a5_{pool}_ids"] = enc["input_ids"].astype(np.int32)
    out[f"a5_{pool}_mask"] = enc["attention_mask"].astype(np.int32)
    out[f"a5_{pool}_vec"] = np.asarray(vec, dtype=np.float32)
    out[f"a5_{pool}_vec_unnormalized"] = np.asarray(vec_un, dtype=np.float32)
meta["a5_weights"] = "oracle.encoders.make_bert_weights(tiny_bert(pool), seed=2024)"

# ------------------------------------------------------------------------------------------------ (a3, a4) OPEN_CLIP wrapper
from marqo.core.inference.embedding_models.open_clip_model import OPEN_CLIP  # noqa: E402
from marqo.s2_inference.clip_utils import _get_transform  # noqa: E402
from transformers import (CLIPTextConfig, CLIPTextModelWithProjection, CLIPVisionConfig,  # noqa: E402
                          CLIPVisionModelWithProjection)

sys.path.insert(0, os.path.join(ROOT, "tests"))
from test_oracle_encoders import _copy_clip_block  # noqa: E402

cfg = E.tiny_clip("gelu")
sd = E.make_clip_weights(cfg, seed=2025)
v, t = cfg.vision, cfg.text
vm = CLIPVisionModelWithProjection(CLIPVisionConfig(
    hidden_size=v.width, intermediate_size=v.mlp, num_hidden_layers=v.layers, num_attention_heads=v.heads,
    image_size=v.image_size, patch_size=v.patch, projection_dim=cfg.embed_dim, hidden_act="gelu", layer_norm_eps=1e-5,
    attn_implementation="eager")).eval()
m = vm.vision_model
m.embeddings.patch_embedding.weight.data.copy_(sd["visual.conv1.weight"])
m.embeddings.class_embedding.data.copy_(sd["visual.class_embedding"])
m.embeddings.position_embedding.weight.data.copy_(sd["visual.positional_embedding"])
pre = getattr(m, "pre_layrnorm", None) or getattr(m, "pre_layernorm")
pre.weight.data.copy_(sd["visual.ln_pre.weight"]); pre.bias.data.copy_(sd["visual.ln_pre.bias"])
m.post_layernorm.weight.data.copy_(sd["visual.ln_post.weight"]); m.post_layernorm.bias.data.copy_(sd["visual.ln_post.bias"])
for i, layer in enumerate(m.encoder.layers):
    _copy_clip_block(layer, sd, f"visual.transformer.resblocks.{i}.", v.width)
vm.visual_projection.weight.data.copy_(sd["visual.proj"].t())
tm_ = CLIPTextModelWithProjection(CLIPTextConfig(
    vocab_size=t.vocab, hidden_size=t.width, intermediate_size=t.mlp, num_hidden_layers=t.layers,
    num_attention_heads=t.heads, max_position_embeddings=t.ctx, projection_dim=cfg.embed_dim, hidden_act="gelu",
    layer_norm_eps=1e-5, eos_token_id=t.vocab - 1, bos_token_id=t.vocab - 2, pad_token_id=0,
    attn_implementation="eager")).eval()
tmm = tm_.text_model
tmm.embeddings.token_embedding.weight.data.copy_(sd["token_embedding.weight"])
tmm.embeddings.position_embedding.weight.data.copy_(sd["positional_embedding"])
tmm.final_layer_norm.weight.data.copy_(sd["ln_final.weight"]); tmm.final_layer_norm.bias.data.copy_(sd["ln_final.bias"])
for i, layer in enumerate(tmm.encoder.layers):
    _copy_clip_block(layer, sd, f"transformer.resblocks.{i}.", t.width)
tm_.text_projection.weight.data.copy_(sd["text_projection"].t())


class HFClipAsOpenClip:
    """Gives the reference's OPEN_CLIP wrapper the `encode_image` / `encode_text` methods it calls on `self.model`."""

    def encode_image(self, x):
        return vm(pixel_values=x).image_embeds

    def encode_text(self, ids):
        return tm_(input_ids=ids).text_embeds


rng = np.random.default_rng(11)
clip_ids = np.zeros((5, t.ctx), dtype=np.int64)
for b, L in enumerate([4, 77, 20, 9, 50]):
    clip_ids[b, 0] = t.vocab - 2
    clip_ids[b, 1:L - 1] = rng.integers(1, t.vocab - 2, size=L - 2)
    clip_ids[b, L - 1] = t.vocab - 1
oc = OPEN_CLIP.__new__(OPEN_CLIP)
oc.device = "cpu"
oc.model = HFClipAsOpenClip()
oc.preprocess = _get_transform(224)          # the in-tree statement of the CLIP transform, clip_utils.py:48-67
oc.tokenizer = lambda s: torch.from_numpy(clip_ids[: len(s)])
from PIL import Image  # noqa: E402

imgs_sq = rng.integers(0, 256, size=(3, 224, 224, 3), dtype=np.uint8)
imgs_big = rng.integers(0, 256, size=(2, 300, 400, 3), dtype=np.uint8)
# the test regenerates the pixels from this seeded stream (1.2 MB that does not compress); it checks these digests
meta["a3_images_sha256"] = {"224": hashlib.sha256(imgs_sq.tobytes()).hexdigest(),
                            "300x400": hashlib.sha256(imgs_big.tobytes()).hexdigest()}
out["a3_vec_224"] = np.asarray(oc.encode_image([Image.fromarray(a) for a in imgs_sq], normalize=True), np.float32)
out["a3_vec_300x400"] = np.asarray(oc.encode_image([Image.fromarray(a) for a in imgs_big], normalize=True), np.float32)
out["a3_vec_224_unnormalized"] = np.asarray(oc.encode_image([Image.fromarray(a) for a in imgs_sq], normalize=False),
                                            np.float32)
out["a4_ids"] = clip_ids.astype(np.int32)
out["a4_vec"] = np.asarray(oc.encode_text(["s"] * 5, normalize=True), np.float32)
meta["a3_weights"] = "oracle.encoders.make_clip_weights(tiny_clip('gelu'), seed=2025)"

# ------------------------------------------------------------------------------------------------ (a2) transform
tfm = _get_transform(224)
pre_big = torch.stack([tfm(Image.fromarray(a)) for a in imgs_big]).numpy()
out["a2_pre_300x400_sample"] = pre_big[:, :, ::16, ::16].copy()        # subsample: full tensor is 1.2 MB
out["a2_pre_300x400_sum"] = np.asarray([float(pre_big.astype(np.float64).sum())])

# ------------------------------------------------------------------------------------------------ (a7) fusion
from marqo.core.inference.tensor_fields_container import MultiModalTensorFieldContent, TensorFieldContent  # noqa: E402
from marqo.core.models.marqo_index import FieldType  # noqa: E402

rng = np.random.default_rng(13)
e1, e2, e3 = rng.standard_normal((3, 16))
for norm in (False, True):
    subs = {}
    for name, e in (("f1", e1), ("f2", e2), ("f3", e3)):
        sf = TensorFieldContent(field_type=FieldType.Text, field_content="x", is_tensor_field=False,
                                is_multimodal_subfield=True)
        sf.chunks = ["c"]
        sf.embeddings = [e.tolist()]
        subs[name] = sf
    mm = MultiModalTensorFieldContent(weights={"f1": 0.3, "f2": -1.2, "f3": 2.0}, field_content="",
                                      field_type=FieldType.MultimodalCombination, subfields=subs,
                                      is_tensor_field=True, normalize_embeddings=norm)
    out[f"a7_fused_norm{int(norm)}"] = np.asarray(mm.tensor_field_embeddings[0], dtype=np.float64)
out["a7_inputs"] = np.stack([e1, e2, e3])
out["a7_weights"] = np.asarray([0.3, -1.2, 2.0])

# ------------------------------------------------------------------------------------------------ (a6) routing
from marqo.core.inference.image_download import _is_image  # noqa: E402

meta["a6_is_image"] = {
    "pil": bool(_is_image([Image.fromarray(imgs_sq[0])])),
    "ndarray": bool(_is_image([imgs_sq[0]])),
    "tensor": bool(_is_image([torch.zeros(3, 224, 224)])),
    "ext_jpg": bool(_is_image(["some/where/cat.JPG"])),
    "ext_png_str": bool(_is_image("dog.png")),
}

meta["stubbed_modules"] = sorted(set(stubbed))
meta["versions"] = {"torch": torch.__version__, "transformers": __import__("transformers").__version__,
                    "numpy": np.__version__, "PIL": __import__("PIL").__version__,
                    "torchvision": __import__("torchvision").__version__}
out["meta_json"] = np.frombuffer(json.dumps(meta, sort_keys=True).encode(), dtype=np.uint8)
path = os.path.join(HERE, "reference_golden.npz")
np.savez_compressed(path, **out)
print("wrote", path, os.path.getsize(path), "bytes")
print(json.dumps(meta, indent=1))
