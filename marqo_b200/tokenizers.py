"""Host mirror of the two tokenizers on the reference's vectorise path, backed by the C ABI (b200_tokenizer_*, §8 f2).

* `WordPieceTokenizer` is called the way hugging_face_model.py:179-185 calls its AutoTokenizer:
  `tok(sentences, padding=True, truncation=True, max_length=N, return_tensors="np")` -> {input_ids, attention_mask,
  token_type_ids}.
* `ClipBpeTokenizer` is called the way open_clip_model.py:277-279 calls open_clip's tokenizer:
  `tok(texts) -> int64 [n, context_length]`.

Both take the vocabulary FILE Marqo's model cache already holds (vocab.txt / bpe_simple_vocab_16e6.txt[.gz])."""
from __future__ import annotations

import ctypes as C
import gzip
from pathlib import Path
from typing import Dict, List, Sequence, Union

import numpy as np

from . import _native as N


class _Tokenizer:
    def __init__(self, handle):
        self._lib = N.load()
        self._h = handle

    def close(self) -> None:
        h, self._h = getattr(self, "_h", None), None
        if h:
            self._lib.b200_tokenizer_destroy(h)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def vocab_size(self) -> int:
        n = C.c_int(0)
        N.check(self._lib.b200_tokenizer_vocab_size(self._h, C.byref(n)))
        return n.value

    def _encode(self, texts: Sequence[str], max_length: int):
        raw = [t.encode("utf-8", "replace") for t in texts]
        n = len(raw)
        ptrs = (C.c_char_p * n)(*raw)
        lens = np.asarray([len(b) for b in raw], dtype=np.int64)
        ids = np.empty((n, max_length), dtype=np.int32)
        mask = np.empty((n, max_length), dtype=np.int32)
        L = C.c_int(0)
        N.check(self._lib.b200_tokenizer_encode(self._h, C.cast(ptrs, C.c_void_p), lens.ctypes.data_as(C.c_void_p), n,
                                                int(max_length), ids.ctypes.data_as(C.c_void_p),
                                                mask.ctypes.data_as(C.c_void_p), C.byref(L)))
        L = L.value
        return ids.reshape(-1)[: n * L].reshape(n, L), mask.reshape(-1)[: n * L].reshape(n, L)


def _read(path_or_bytes: Union[str, Path, bytes]) -> bytes:
    if isinstance(path_or_bytes, bytes):
        return path_or_bytes
    data = Path(path_or_bytes).read_bytes()
    return gzip.decompress(data) if data[:2] == b"\x1f\x8b" else data


class WordPieceTokenizer(_Tokenizer):
    """BERT's special tokens by default; MPNet's tokenizer is cls_token="<s>", sep_token="</s>", pad_token="<pad>",
    unk_token="[UNK]"."""

    def __init__(self, vocab: Union[str, Path, bytes], do_lower_case: bool = True, model_max_length: int = 512,
                 cls_token: str = "[CLS]", sep_token: str = "[SEP]", pad_token: str = "[PAD]", unk_token: str = "[UNK]"):
        data = _read(vocab)
        h = C.c_void_p()
        N.check(N.load().b200_tokenizer_create_wordpiece_special(
            data, len(data), 1 if do_lower_case else 0, cls_token.encode(), sep_token.encode(), pad_token.encode(),
            unk_token.encode(), C.byref(h)))
        super().__init__(h)
        self.model_max_length = model_max_length

    def __call__(self, sentences: Union[str, List[str]], padding=True, truncation=True, max_length: int = None,
                 return_tensors: str = "np") -> Dict[str, np.ndarray]:
        if padding is not True or truncation is not True:
            raise ValueError("WordPieceTokenizer implements the reference's call only: padding=True, truncation=True")
        single = isinstance(sentences, str)
        ids, mask = self._encode([sentences] if single else list(sentences), max_length or self.model_max_length)
        out = {"input_ids": ids.astype(np.int64), "token_type_ids": np.zeros_like(ids, dtype=np.int64),
               "attention_mask": mask.astype(np.int64)}
        if return_tensors == "pt":
            import torch
            return {k: torch.from_numpy(v) for k, v in out.items()}
        return out


class ClipBpeTokenizer(_Tokenizer):
    def __init__(self, merges: Union[str, Path, bytes], context_length: int = 77):
        data = _read(merges)
        h = C.c_void_p()
        N.check(N.load().b200_tokenizer_create_clip_bpe(data, len(data), C.byref(h)))
        super().__init__(h)
        self.context_length = context_length

    def __call__(self, texts: Union[str, List[str]], context_length: int = None) -> np.ndarray:
        if isinstance(texts, str):
            texts = [texts]
        ids, _ = self._encode(list(texts), context_length or self.context_length)
        return ids.astype(np.int64)
