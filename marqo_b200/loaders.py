"""Loader classes behind the reference's loader-registry seam (boundary B1, SURVEY §8b).

`MODEL_PROPERTIES['loaders'][type]` (src/marqo/s2_inference/model_registry.py:2133-2145) maps a model `type` to a class
that is constructed as `loader(device=, model_properties=, model_auth=)`, `.load()`-ed once and then driven only
through `.encode(...)` (+ `.preprocess`, `.encode_image`, `.encode_text` on CLIP-type models)
(src/marqo/s2_inference/s2_inference.py:520-568, :129-146, :228-233).  These two classes provide exactly that
surface on top of the C ABI:

  B200OpenCLIP    <-> OPEN_CLIP        (src/marqo/core/inference/embedding_models/open_clip_model.py:249-286,
                                        abstract_clip_model.py:56-112)
  B200HuggingFace <-> HuggingFaceModel (src/marqo/core/inference/embedding_models/hugging_face_model.py:172-214)

Weights: `model_properties["weights"]` is a state dict (checkpoint names) or a path to one; `"random_init": seed`
builds seeded random weights (benchmarks / self-test).  Tokenisers, in order of preference:
`model_properties["tokenizer"]` (a callable); `model_properties["vocab_file"]` (HF: vocab.txt) /
`model_properties["merges_file"]` (CLIP: bpe_simple_vocab_16e6.txt[.gz]) -> the C++ tokenizers behind the C ABI
(marqo_b200/tokenizers.py, §8 f2); else the HF loader tries `transformers.AutoTokenizer.from_pretrained(name)` and the
CLIP loader `open_clip.get_tokenizer` — both need files that only exist where Marqo's own model cache does.
"""
from __future__ import annotations

from typing import Callable, Dict, List, Optional, Union

import numpy as np

from . import model_registry, weights as weights_mod
from .errors import InvalidModelPropertiesError, ModelLoadError, VectoriseError
from .s2_inference import Modality, UnidentifiedImageError, _is_image, _is_tensor, _validate_device


def _resolve_weights(props: dict, arch: dict, kind: str) -> Dict[str, np.ndarray]:
    w = props.get("weights")
    if w is None and props.get("random_init") is not None:
        seed = int(props["random_init"])
        random = {"clip": weights_mod.random_clip_weights, "bert": weights_mod.random_bert_weights,
                  "mpnet": weights_mod.random_mpnet_weights}[kind]
        return random(arch, seed)
    if w is None:
        raise ModelLoadError("model_properties needs `weights` (state dict or checkpoint path) or `random_init`; "
                             "checkpoint download is Marqo's job (open_clip_model.py:107-131) and out of scope here")
    if isinstance(w, (str, bytes)) or hasattr(w, "__fspath__"):
        w = weights_mod.load_state_dict(w)
    if kind == "bert":
        w = weights_mod.strip_hf_prefix(w)
    elif kind == "mpnet":
        w = weights_mod.strip_hf_prefix(w, "mpnet.")
    return w


class _PreprocessToU8:
    """`model.preprocess` replacement (read at s2_inference.py:228-233, applied in the download threads at
    src/marqo/tensor_search/add_docs.py:129-134).  The reference runs Resize+CenterCrop+ToTensor+Normalize on the CPU
    thread; here the thread only hands the decoded pixels over as a uint8 HWC tensor and the whole transform runs on
    the GPU fused into the patch-embed load."""

    def __init__(self, gpu_decode: bool = True):
        self.gpu_decode = gpu_decode

    def __call__(self, pil_image):
        import torch
        if self.gpu_decode:
            # Image.open() is lazy: a JPEG that has not been decoded yet is handed over still encoded and decoded on
            # the GPU with the rest of its batch (image_decode.py, b200_jpeg_decode_batch — bit-exact with Pillow)
            from .image_decode import EncodedImage, encoded_bytes_of
            data = encoded_bytes_of(pil_image)
            if data is not None:
                return EncodedImage(data, "JPEG")
        return torch.from_numpy(np.asarray(pil_image.convert("RGB"), dtype=np.uint8).copy())


class B200OpenCLIP:
    def __init__(self, device: Optional[str] = None, model_properties: Optional[dict] = None, model_auth=None):
        if device is None:
            raise ModelLoadError("`device` is required for loading CLIP models!")  # open_clip_model.py:__init__
        self.device = device
        self.model_properties = dict(model_properties or {})
        self.model_auth = model_auth
        self.model = None
        self.tokenizer: Optional[Callable] = None
        self.preprocess = _PreprocessToU8()
        self.preprocess_config = None

    def load(self) -> None:
        from .engine import Encoder
        props = self.model_properties
        arch = props.get("arch")
        if arch is None:
            raise InvalidModelPropertiesError("model_properties has no `arch` block")
        if props.get("mean") is not None:  # open_clip_model_properties.py:24-61 overrides
            arch = dict(arch, mean=tuple(props["mean"]))
        if props.get("std") is not None:
            arch = dict(arch, std=tuple(props["std"]))
        self.arch = arch
        self.model = Encoder("clip", arch, _resolve_weights(props, arch, "clip"), device=_validate_device(self.device),
                             max_batch=int(props.get("max_batch", 256)))
        self.tokenizer = props.get("tokenizer") or self._default_tokenizer()

    def _default_tokenizer(self):
        if self.model_properties.get("merges_file"):
            from .tokenizers import ClipBpeTokenizer
            return ClipBpeTokenizer(self.model_properties["merges_file"], context_length=int(self.arch["text"]["ctx"]))
        try:
            import open_clip  # type: ignore
            return open_clip.get_tokenizer(self.model_properties.get("name", "").split("/")[1])
        except Exception:
            return None  # encode_text raises a clear error if text arrives without a tokenizer

    def close(self) -> None:
        if self.model is not None:
            self.model.close()
            self.model = None

    # -- reference surface -------------------------------------------------------------------------------------
    def encode(self, inputs, default: str = 'text', normalize=True, **kwargs) -> np.ndarray:
        """abstract_clip_model.py:56-75"""
        infer = kwargs.pop('infer', True)
        if infer and _is_image(inputs):
            is_image = True
        else:
            if default == 'text':
                is_image = False
            elif default == 'image':
                is_image = True
            else:
                raise UnidentifiedImageError(f"expected default='image' or default='text' but received {default}")
        if is_image:
            return self.encode_image(inputs, normalize=normalize,
                                     image_download_headers=kwargs.get("image_download_headers", dict()))
        return self.encode_text(inputs, normalize=normalize)

    def encode_image(self, images, image_download_headers: Optional[Dict] = None, normalize=True) -> np.ndarray:
        """open_clip_model.py:249-266.  List elements may be PIL images, uint8 HWC tensors/arrays (what
        `self.preprocess` returns) or already-preprocessed float CHW tensors (passed through unchanged by the
        reference, abstract_clip_model.py:108-111)."""
        if self.model is None:
            self.load()
        items = images if isinstance(images, list) else [images]
        if len(items) == 0:
            raise UnidentifiedImageError("received empty list, expected at least one element.")
        S = self.model.image_size
        from .image_decode import EncodedImage, decode_images_to_device
        if any(isinstance(it, (EncodedImage, bytes, bytearray)) for it in items):
            # still-encoded files (what the preprocessor hands over for JPEGs): decode the batch on the GPU; the pixels
            # stay in HBM for the resize + patch-embed kernels
            enc_idx = [i for i, it in enumerate(items) if isinstance(it, (EncodedImage, bytes, bytearray))]
            try:
                decoded = decode_images_to_device([items[i] for i in enc_idx], device=self.model.device)
            except OSError as e:              # Pillow's error for broken files, wrapped like the reference does
                raise UnidentifiedImageError(str(e)) from e
            items = list(items)
            for i, t in zip(enc_idx, decoded):
                items[i] = t
        if all(self._on_model_device(it) for it in items):
            return self._encode_device_images(items, bool(normalize))
        u8, f32 = [], []
        for it in items:
            if isinstance(it, str):
                raise VectoriseError("image download is Marqo's job (image_download.py:130-215); pass decoded images")
            if type(it).__module__.startswith("PIL."):
                it = np.asarray(it.convert("RGB"), dtype=np.uint8)
            if _is_tensor(it):
                it = it.detach().to("cpu").numpy()
            a = np.asarray(it)
            if a.dtype == np.uint8 and a.ndim == 3 and a.shape[2] == 3:
                u8.append(a)
            elif a.dtype.kind == "f" and a.shape == (3, S, S):
                f32.append(a.astype(np.float32, copy=False))
            else:
                raise UnidentifiedImageError(f"unsupported image element: dtype {a.dtype}, shape {a.shape}")
        if u8 and f32:
            raise UnidentifiedImageError("a batch must not mix raw uint8 images and preprocessed tensors")
        if f32:
            return self.model.encode_images_f32(np.stack(f32), normalize=bool(normalize))
        out = np.empty((len(u8), self.model.embed_dim), np.float32)
        # group by (h, w): the C ABI takes one rectangular uint8 block per call
        groups: Dict[tuple, List[int]] = {}
        for i, a in enumerate(u8):
            groups.setdefault(a.shape[:2], []).append(i)
        for (h, w), idx in groups.items():
            out[idx] = self.model.encode_images_u8_list([u8[i] for i in idx], normalize=bool(normalize))
        return out

    def _on_model_device(self, it) -> bool:
        """A uint8 HWC torch tensor already resident on this model's GPU — what Marqo's download threads produce:
        `preprocessors['image'](image).to(device)` (add_docs.py:129-134)."""
        return (_is_tensor(it) and getattr(it, "is_cuda", False) and it.device.index == self.model.device
                and str(it.dtype) == "torch.uint8" and it.ndim == 3 and it.shape[2] == 3)

    def _encode_device_images(self, items, normalize: bool) -> np.ndarray:
        """Images that are already in HBM stay there: one device-side stack per image size, the device entry point,
        one D2H copy of the [n, dim] result — no per-image round trip through the host."""
        import torch
        out = torch.empty((len(items), self.model.embed_dim), dtype=torch.float32, device=items[0].device)
        groups: Dict[tuple, List[int]] = {}
        for i, t in enumerate(items):
            groups.setdefault((int(t.shape[0]), int(t.shape[1])), []).append(i)
        for (h, w), idx in groups.items():
            batch = torch.stack([items[i] for i in idx]).contiguous()
            res = out if len(groups) == 1 else torch.empty((len(idx), self.model.embed_dim), dtype=torch.float32,
                                                          device=batch.device)
            self._sync_device(batch.device)      # the engine runs on its own stream: the stack must have landed
            self.model.encode_images_u8_device(batch.data_ptr(), len(idx), h, w, res.data_ptr(), normalize=normalize,
                                               sync=True)
            if res is not out:
                out[torch.as_tensor(idx, device=out.device)] = res
        return out.cpu().numpy()

    @staticmethod
    def _sync_device(device) -> None:
        import torch
        torch.cuda.synchronize(device)

    def _tokenize(self, sentence) -> np.ndarray:
        if self.tokenizer is None:
            raise ModelLoadError("no CLIP tokenizer available: supply model_properties['tokenizer'] "
                                 "(open_clip's BPE vocabulary is not bundled)")
        text = self.tokenizer(sentence if isinstance(sentence, list) else [sentence])
        if _is_tensor(text):
            text = text.detach().to("cpu").numpy()
        return np.ascontiguousarray(text, dtype=np.int32)

    def encode_text(self, sentence: Union[str, List[str]], normalize=True) -> np.ndarray:
        """open_clip_model.py:268-286"""
        if self.model is None:
            self.load()
        return self.model.encode_tokens(self._tokenize(sentence), None, normalize=bool(normalize))

    # -- add_documents fast path: embeddings stay in HBM (consumed by GpuTensorIndex.feed_batch as DeviceChunks) ----
    def encode_to_device(self, inputs, default: str = 'text', normalize=True, sub_batch: int = 256, **kwargs):
        """encode() whose result is a CUDA fp32 tensor [n, dim] on the model's device instead of a host ndarray: the
        vectors go from the projection + L2 epilogue straight into the row store (b200_index_add_device_docs), never
        through `List[List[float]]`.  Same routing rules as encode() (abstract_clip_model.py:56-75).  Images: uint8 HWC
        arrays / tensors of ONE size per call; texts: strings, or an int32 [n, ctx] array of token ids."""
        import torch
        if self.model is None:
            self.load()
        infer = kwargs.pop('infer', True)
        items = inputs if isinstance(inputs, list) else [inputs]
        is_ids = isinstance(inputs, np.ndarray) and inputs.dtype.kind in "iu" and inputs.ndim == 2
        is_image = not is_ids and ((infer and _is_image(inputs)) or default == 'image')
        dev = torch.device("cuda", self.model.device)
        n = inputs.shape[0] if is_ids else len(items)
        out = torch.empty((n, self.model.embed_dim), dtype=torch.float32, device=dev)
        step = max(1, min(int(sub_batch), int(self.model_properties.get("max_batch", 256))))
        if is_image:
            for lo in range(0, n, step):
                part = items[lo:lo + step]
                if all(self._on_model_device(it) for it in part):
                    batch = torch.stack(part).contiguous()
                else:
                    host = np.stack([np.asarray(it.cpu() if _is_tensor(it) else
                                                (it.convert("RGB") if type(it).__module__.startswith("PIL.") else it),
                                                dtype=np.uint8) for it in part])
                    batch = torch.from_numpy(host).to(dev, non_blocking=False)
                if batch.ndim != 4 or batch.shape[3] != 3:
                    raise UnidentifiedImageError(f"expected uint8 [n, H, W, 3] images, got {tuple(batch.shape)}")
                self._sync_device(dev)
                self.model.encode_images_u8_device(batch.data_ptr(), len(part), int(batch.shape[1]), int(batch.shape[2]),
                                                   out[lo:].data_ptr(), normalize=bool(normalize), sync=True)
        else:
            ids = np.ascontiguousarray(inputs, dtype=np.int32) if is_ids else self._tokenize(items)
            d_ids = torch.from_numpy(ids).to(dev)
            self._sync_device(dev)
            for lo in range(0, n, step):
                m = min(step, n - lo)
                self.model.encode_tokens_device(d_ids[lo:].data_ptr(), None, m, int(ids.shape[1]), out[lo:].data_ptr(),
                                                normalize=bool(normalize), sync=True)
        return out


class B200HuggingFace:
    def __init__(self, device: Optional[str] = None, model_properties: Optional[dict] = None, model_auth=None):
        if device is None:
            raise ModelLoadError("`device` is required for loading HF models!")
        self.device = device
        self.model_properties = dict(model_properties or {})
        self.model_auth = model_auth
        self._model = None
        self._tokenizer = None
        self.max_seq_length = int(self.model_properties.get("tokens", 128))

    def load(self) -> None:
        from .engine import Encoder
        props = self.model_properties
        arch = props.get("arch")
        if arch is None:
            raise InvalidModelPropertiesError("model_properties has no `arch` block")
        if props.get("poolingMethod") or props.get("pooling_method"):  # hugging_face_model_properties.py
            arch = dict(arch, pool=(props.get("poolingMethod") or props.get("pooling_method")))
        self.arch = arch
        kind = arch.get("family", "bert")   # "bert" (e5 & co.) or "mpnet" (all-mpnet-base & co.)
        self._model = Encoder(kind, arch, _resolve_weights(props, arch, kind), device=_validate_device(self.device),
                              max_batch=int(props.get("max_batch", 256)))
        self._tokenizer = props.get("tokenizer") or self._default_tokenizer()

    def _default_tokenizer(self):
        if self.model_properties.get("vocab_file"):
            from .tokenizers import WordPieceTokenizer
            specials = {}
            if self.arch.get("family") == "mpnet":   # MPNetTokenizer: WordPiece framed by <s> ... </s>, <pad> id 1
                specials = dict(cls_token="<s>", sep_token="</s>", pad_token="<pad>", unk_token="[UNK]")
            return WordPieceTokenizer(self.model_properties["vocab_file"],
                                      do_lower_case=bool(self.model_properties.get("do_lower_case", True)), **specials)
        try:
            from transformers import AutoTokenizer
            return AutoTokenizer.from_pretrained(self.model_properties["name"])
        except Exception:
            return None

    def close(self) -> None:
        if self._model is not None:
            self._model.close()
            self._model = None

    def encode(self, sentence: Union[str, List[str]], normalize=True, **kwargs) -> np.ndarray:
        """hugging_face_model.py:172-197: tokenizer(padding=True, truncation=True, max_length=tokens) -> forward ->
        pooling -> F.normalize."""
        if isinstance(sentence, str):
            sentence = [sentence]
        if self._model is None:
            self.load()
        if self._tokenizer is None:
            raise ModelLoadError("no tokenizer available: supply model_properties['tokenizer'] or make "
                                 f"{self.model_properties.get('name')!r} loadable by transformers.AutoTokenizer")
        tok = self._tokenizer(sentence, padding=True, truncation=True, max_length=self.max_seq_length,
                              return_tensors="np")
        ids = np.asarray(tok["input_ids"], dtype=np.int32)
        mask = np.asarray(tok["attention_mask"], dtype=np.int32)
        return self._model.encode_tokens(ids, mask, normalize=bool(normalize))

    def encode_to_device(self, sentence, normalize=True, sub_batch: int = 64, attention_mask=None, **kwargs):
        """encode() whose result stays on the GPU (CUDA fp32 tensor [n, dim]) for the add_documents fast path.
        `sentence`: strings (tokenised per sub-batch with padding=True, like the reference's own sub-batching,
        s2_inference.py:137-146), or an int32 [n, seq] array of token ids (+ optional attention_mask)."""
        import torch
        if self._model is None:
            self.load()
        dev = torch.device("cuda", self._model.device)
        is_ids = isinstance(sentence, np.ndarray) and sentence.dtype.kind in "iu" and sentence.ndim == 2
        items = sentence if is_ids else ([sentence] if isinstance(sentence, str) else list(sentence))
        n = len(items)
        out = torch.empty((n, self._model.embed_dim), dtype=torch.float32, device=dev)
        step = max(1, min(int(sub_batch), int(self.model_properties.get("max_batch", 256))))
        for lo in range(0, n, step):
            if is_ids:
                ids = np.ascontiguousarray(items[lo:lo + step], dtype=np.int32)
                mask = None if attention_mask is None else np.ascontiguousarray(attention_mask[lo:lo + step], dtype=np.int32)
            else:
                if self._tokenizer is None:
                    raise ModelLoadError("no tokenizer available: supply model_properties['tokenizer'] or 'vocab_file'")
                tok = self._tokenizer(items[lo:lo + step], padding=True, truncation=True, max_length=self.max_seq_length,
                                      return_tensors="np")
                ids = np.asarray(tok["input_ids"], dtype=np.int32)
                mask = np.asarray(tok["attention_mask"], dtype=np.int32)
            d_ids = torch.from_numpy(ids).to(dev)
            d_mask = None if mask is None else torch.from_numpy(mask).to(dev)
            torch.cuda.synchronize(dev)
            self._model.encode_tokens_device(d_ids.data_ptr(), None if d_mask is None else d_mask.data_ptr(), ids.shape[0],
                                             ids.shape[1], out[lo:].data_ptr(), normalize=bool(normalize), sync=True)
        return out


LOADERS = {
    model_registry.TYPE_OPEN_CLIP: B200OpenCLIP,
    model_registry.TYPE_HF: B200HuggingFace,
}


def get_model_loader(model_name: Optional[str], model_properties: dict):
    """s2_inference.py:752-771"""
    model_type = model_properties['type']
    if model_type not in LOADERS:
        raise KeyError(f"model_name={model_name} for model_type={model_type} not in allowed model types")
    return LOADERS[model_type]


def register_with_marqo() -> None:
    """Install the two loader types into a live Marqo process (see INTEGRATION.md)."""
    from marqo.s2_inference import s2_inference as marqo_s2  # type: ignore
    marqo_s2.MODEL_PROPERTIES['loaders'].update(LOADERS)
    marqo_s2.MODEL_PROPERTIES['models'].update(model_registry.MODELS)
