"""Thin Python objects over the C ABI handles (include/marqo_b200.h).  No arithmetic happens here."""
from __future__ import annotations

import ctypes as C
import threading
from typing import Optional, Sequence, Tuple

import numpy as np

from . import _native as N

_METRICS = {
    # names: src/marqo/core/models/marqo_index.py:63-69 (DistanceMetric)
    "prenormalized-angular": N.METRIC_PRENORMALIZED_ANGULAR,
    "angular": N.METRIC_ANGULAR,
    "dotproduct": N.METRIC_DOTPRODUCT,
    "euclidean": N.METRIC_EUCLIDEAN,
}


def _ptr(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _as(a, dtype) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=dtype)


class RowStore:
    """GPU-resident fp16 embedding matrix with exact top-k search (b200_index_*)."""

    def __init__(self, dim: int, metric: str = "prenormalized-angular", device: int = 0, capacity: int = 0,
                 _handle=None):
        self._lib = N.load()
        self.dim = int(dim)
        self.metric = metric
        self.device = int(device)
        if _handle is not None:
            self._h = _handle
            return
        if metric not in _METRICS:
            raise ValueError(f"unknown distance metric {metric!r}; expected one of {sorted(_METRICS)}")
        h = C.c_void_p()
        N.check(self._lib.b200_index_create(self.device, self.dim, _METRICS[metric], int(capacity), C.byref(h)))
        self._h = h

    # -- lifetime -------------------------------------------------------------------------------
    def close(self) -> None:
        h, self._h = getattr(self, "_h", None), None
        if h:
            self._lib.b200_index_destroy(h)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _handle(self):
        if not self._h:
            raise RuntimeError("RowStore is closed")
        return self._h

    # -- mutation -------------------------------------------------------------------------------
    def add(self, vecs, doc_ids: Optional[Sequence[int]] = None) -> None:
        v = _as(vecs, np.float32)
        if v.ndim != 2 or v.shape[1] != self.dim:
            raise ValueError(f"expected [m, {self.dim}] embeddings, got {v.shape}")
        d = None
        if doc_ids is not None:
            d = _as(doc_ids, np.int32)
            if d.shape != (v.shape[0],):
                raise ValueError("doc_ids must have one entry per row")
        N.check(self._lib.b200_index_add(self._handle(), _ptr(v), _ptr(d), v.shape[0]))

    def add_device(self, d_vecs_ptr: int, m: int, d_doc_ids_ptr: Optional[int] = None) -> None:
        N.check(self._lib.b200_index_add_device(self._handle(), C.c_void_p(d_vecs_ptr),
                                                C.c_void_p(d_doc_ids_ptr) if d_doc_ids_ptr else None, int(m)))

    def add_device_docs(self, d_vecs_ptr: int, doc_ids: Sequence[int]) -> None:
        """Embeddings already on the device (fp32 [m, dim]), document numbers on the host: the add_documents fast path."""
        d = _as(doc_ids, np.int32)
        N.check(self._lib.b200_index_add_device_docs(self._handle(), C.c_void_p(d_vecs_ptr), _ptr(d), d.shape[0]))

    def delete_doc(self, doc_id: int) -> None:
        N.check(self._lib.b200_index_delete_doc(self._handle(), int(doc_id)))

    def delete_rows(self, rows: Sequence[int]) -> None:
        r = _as(rows, np.int32)
        N.check(self._lib.b200_index_delete_rows(self._handle(), _ptr(r), r.shape[0]))

    def compact(self) -> np.ndarray:
        """Squeeze tombstoned rows out; -> new_of_old int32 [old rows] (-1 = removed)."""
        n = len(self)
        m = np.empty(n, np.int32)
        left = C.c_int64(0)
        N.check(self._lib.b200_index_compact(self._handle(), _ptr(m), C.byref(left)))
        return m

    # -- queries --------------------------------------------------------------------------------
    def __len__(self) -> int:
        n = C.c_int64(0)
        N.check(self._lib.b200_index_num_rows(self._handle(), C.byref(n)))
        return n.value

    def get_row(self, row: int) -> np.ndarray:
        out = np.empty(self.dim, dtype=np.float32)
        N.check(self._lib.b200_index_get_row(self._handle(), int(row), _ptr(out)))
        return out

    def get_rows(self, rows: Sequence[int]) -> np.ndarray:
        r = _as(rows, np.int64)
        out = np.empty((r.shape[0], self.dim), dtype=np.float32)
        N.check(self._lib.b200_index_get_rows(self._handle(), _ptr(r), r.shape[0], _ptr(out)))
        return out

    def search(self, queries, k: int, mult: Sequence[Tuple[int, float]] = (), add: Sequence[Tuple[int, float]] = (),
               filter_bits: Optional[np.ndarray] = None, filter_docs: int = 0,
               filter_tag: int = 0) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
        """-> (doc [nq,k] int32, row [nq,k] int32, score [nq,k] float64); unused slots are -1/-1/-inf.
        mult / add: score modifiers [(attribute column, weight), ...] (score = modified score then);
        filter_bits: uint32 bitset over document numbers (bit set = may match), covering filter_docs documents;
        filter_tag != 0 lets the device keep the bitset between calls."""
        q = _as(queries, np.float32)
        if q.ndim == 1:
            q = q[None, :]
        if q.ndim != 2 or q.shape[1] != self.dim:
            raise ValueError(f"expected [nq, {self.dim}] queries, got {q.shape}")
        nq = q.shape[0]
        doc = np.empty((nq, k), dtype=np.int32)
        row = np.empty((nq, k), dtype=np.int32)
        score = np.empty((nq, k), dtype=np.float64)
        opts = None
        keep = []
        if mult or add or filter_bits is not None:
            o = N.SearchOpts()
            mc = _as([c for c, _ in mult], np.int32)
            mw = _as([w for _, w in mult], np.float64)
            ac = _as([c for c, _ in add], np.int32)
            aw = _as([w for _, w in add], np.float64)
            keep = [mc, mw, ac, aw]
            o.mult_cols, o.mult_w, o.n_mult = mc.ctypes.data, mw.ctypes.data, len(mc)
            o.add_cols, o.add_w, o.n_add = ac.ctypes.data, aw.ctypes.data, len(ac)
            if filter_bits is not None:
                fb = _as(filter_bits, np.uint32)
                if fb.shape[0] * 32 < filter_docs:
                    raise ValueError("filter_bits does not cover filter_docs documents")
                keep.append(fb)
                o.filter_bits, o.filter_docs, o.filter_tag = fb.ctypes.data, int(filter_docs), int(filter_tag)
            opts = C.byref(o)
        N.check(self._lib.b200_index_search_ex(self._handle(), _ptr(q), nq, int(k), opts, _ptr(doc), _ptr(row),
                                               _ptr(score)))
        del keep
        return doc, row, score

    def search_stats(self) -> dict:
        a, b, c, d = C.c_int64(0), C.c_int64(0), C.c_int64(0), C.c_int64(0)
        N.check(self._lib.b200_index_search_stats(self._handle(), C.byref(a), C.byref(b), C.byref(c), C.byref(d)))
        return {"groups": a.value, "flagged": b.value, "collect_passes": c.value, "unresolved_async": d.value}

    # -- score modifiers -----------------------------------------------------------------------
    def set_attributes(self, column: int, doc_ids: Sequence[int], values: Optional[Sequence[float]]) -> None:
        """Set (values given) or remove (values None) the numeric attribute `column` of the listed documents;
        column == -1 with values None removes every attribute of those documents."""
        d = _as(doc_ids, np.int32)
        v = None
        if values is not None:
            v = _as(values, np.float64)
            if v.shape != d.shape:
                raise ValueError("values must have one entry per document")
        N.check(self._lib.b200_index_set_attributes(self._handle(), int(column), _ptr(d), _ptr(v), d.shape[0]))

    def set_attributes_multi(self, columns: Sequence[int], doc_ids: Sequence[int], values: Sequence[float]) -> None:
        """Many (column, document, value) cells in one call."""
        c, d, v = _as(columns, np.int32), _as(doc_ids, np.int32), _as(values, np.float64)
        if not (c.shape == d.shape == v.shape):
            raise ValueError("columns, doc_ids and values must have the same length")
        N.check(self._lib.b200_index_set_attributes_multi(self._handle(), _ptr(c), _ptr(d), _ptr(v), c.shape[0]))

    def search_modified(self, queries, k: int, mult: Sequence[Tuple[int, float]] = (),
                        add: Sequence[Tuple[int, float]] = ()) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
        """search() ranked by modify(closeness) = prod(w * attr) * closeness + sum(w * attr)
        (unstructured_vespa_schema.py:266-271).  mult / add: [(attribute column, weight), ...].
        -> (doc, row, modified score)."""
        return self.search(queries, k, mult=mult, add=add)

    def search_device(self, d_q_ptr: int, nq: int, k: int, d_doc_ptr: int, d_row_ptr: int, d_score_ptr: int,
                      sync: bool = True) -> None:
        N.check(self._lib.b200_index_search_device(self._handle(), C.c_void_p(d_q_ptr), int(nq), int(k),
                                                   C.c_void_p(d_doc_ptr), C.c_void_p(d_row_ptr),
                                                   C.c_void_p(d_score_ptr), 1 if sync else 0))

    def set_stream(self, cuda_stream: Optional[int]) -> None:
        """cuda_stream: a cudaStream_t handle (0 = legacy default stream); None restores the private stream."""
        N.check(self._lib.b200_index_set_stream(self._handle(), C.c_void_p(cuda_stream or 0),
                                                0 if cuda_stream is None else 1))

    def set_doc_offset(self, offset: int) -> None:
        N.check(self._lib.b200_index_set_doc_offset(self._handle(), int(offset)))

    def merge_shards_device(self, d_gathered_ptr: int, nshards: int, nq: int, k: int, d_doc_ptr: int, d_row_ptr: int,
                            d_score_ptr: int, sync: bool = True) -> None:
        N.check(self._lib.b200_topk_merge_device(self._handle(), C.c_void_p(d_gathered_ptr), nshards, nq, k,
                                                 C.c_void_p(d_doc_ptr), C.c_void_p(d_row_ptr), C.c_void_p(d_score_ptr),
                                                 1 if sync else 0))

    def search_exchange(self, exchange: "Exchange", d_q_ptr: int, nq: int, k: int, d_block_ptr: int, d_doc_ptr: int,
                        d_row_ptr: int, d_score_ptr: int, sync: bool = True) -> None:
        """Local search + fused peer-store exchange + merge (b200_index_search_exchange)."""
        N.check(self._lib.b200_index_search_exchange(self._handle(), exchange._handle(), C.c_void_p(d_q_ptr), int(nq),
                                                     int(k), C.c_void_p(d_block_ptr), C.c_void_p(d_doc_ptr),
                                                     C.c_void_p(d_row_ptr), C.c_void_p(d_score_ptr), 1 if sync else 0))

    def last_timing(self) -> Tuple[float, float]:
        a, b = C.c_float(0), C.c_float(0)
        N.check(self._lib.b200_index_last_timing(self._handle(), C.byref(a), C.byref(b)))
        return a.value, b.value

    # -- persistence ----------------------------------------------------------------------------
    def save(self, path: str) -> None:
        N.check(self._lib.b200_index_save(self._handle(), str(path).encode()))

    @classmethod
    def load(cls, path: str, device: int = 0) -> "RowStore":
        lib = N.load()
        h = C.c_void_p()
        N.check(lib.b200_index_load(int(device), str(path).encode(), C.byref(h)))
        d, m, dev = C.c_int(0), C.c_int(0), C.c_int(0)
        N.check(lib.b200_index_info(h, C.byref(d), C.byref(m), C.byref(dev)))
        names = {v: k for k, v in _METRICS.items()}
        return cls(dim=d.value, metric=names[m.value], device=dev.value, _handle=h)


class Exchange:
    """Symmetric NVLink exchange buffer of one rank (b200_exchange_*).  `handle` (64 bytes) is what the ranks swap;
    `open(all_handles)` maps the peers' buffers."""

    def __init__(self, device: int, rank: int, world: int, max_nq: int = 64, max_k: int = 16):
        self._lib = N.load()
        h = C.c_void_p()
        buf = (C.c_uint8 * N.EXCHANGE_HANDLE_BYTES)()
        N.check(self._lib.b200_exchange_create(int(device), int(rank), int(world), int(max_nq), int(max_k), C.byref(h),
                                               C.cast(buf, C.c_void_p)))
        self._h = h
        self.rank, self.world = int(rank), int(world)
        self.handle = bytes(buf)

    def open(self, handles: Sequence[bytes]) -> None:
        if len(handles) != self.world or any(len(h) != N.EXCHANGE_HANDLE_BYTES for h in handles):
            raise ValueError("expected one 64-byte handle per rank")
        blob = b"".join(handles)
        N.check(self._lib.b200_exchange_open(self._handle(), C.c_char_p(blob)))

    def _handle(self):
        if not self._h:
            raise RuntimeError("Exchange is closed")
        return self._h

    def close(self) -> None:
        h, self._h = getattr(self, "_h", None), None
        if h:
            self._lib.b200_exchange_destroy(h)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def topk_merge(doc: np.ndarray, row: np.ndarray, score: np.ndarray) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
    """Merge per-shard lists [nshards, nq, k] into [nq, k] under (score desc, doc asc)."""
    doc, row, score = _as(doc, np.int32), _as(row, np.int32), _as(score, np.float64)
    ns, nq, k = doc.shape
    od = np.empty((nq, k), np.int32)
    orow = np.empty((nq, k), np.int32)
    osc = np.empty((nq, k), np.float64)
    N.check(N.load().b200_topk_merge(ns, nq, k, _ptr(doc), _ptr(row), _ptr(score), _ptr(od), _ptr(orow), _ptr(osc)))
    return od, orow, osc


# ---------------------------------------------------------------------------------------------------------
# Encoders (b200_model_*)
# ---------------------------------------------------------------------------------------------------------
def _to_numpy_f32(t) -> np.ndarray:
    if hasattr(t, "detach"):
        t = t.detach().to("cpu").float().numpy()
    return np.ascontiguousarray(t, dtype=np.float32)


class Encoder:
    """A CLIP (vision + text towers), BERT or MPNet encoder resident on one GPU.

    `config` keys — CLIP: embed_dim, act ("gelu"|"quickgelu"), mean, std, vision{width,layers,heads,mlp,patch,
    image_size}, text{width,layers,heads,mlp,ctx,vocab};  BERT: width, layers, heads, mlp, vocab, max_pos, type_vocab,
    pool ("mean"|"cls");  MPNet: as BERT without type_vocab, max_pos = max_position_embeddings (514: sequences of up to
    512 tokens), optional buckets (32) and ln_eps (1e-5), the only values the library implements.  `weights` maps
    checkpoint parameter names (open_clip state_dict names / HF BertModel / MPNetModel names) to fp32 arrays or torch
    tensors.
    """

    def __init__(self, arch: str, config: dict, weights: dict, device: int = 0, max_batch: int = 256):
        self._lib = N.load()
        self.arch = arch
        self.device = int(device)
        d = N.ModelDesc()
        d.max_batch = int(max_batch)
        if arch == "clip":
            d.arch = N.ARCH_CLIP
            d.embed_dim = int(config["embed_dim"])
            d.act = N.ACT_QUICKGELU if config.get("act", "gelu") == "quickgelu" else N.ACT_GELU
            mean = config.get("mean", (0.48145466, 0.4578275, 0.40821073))
            std = config.get("std", (0.26862954, 0.26130258, 0.27577711))
            for i in range(3):
                d.image_mean[i] = float(np.float32(mean[i]))
                d.image_std[i] = float(np.float32(std[i]))
            v, t = config.get("vision"), config.get("text")
            if v:
                d.vision = N.TowerDesc(v["width"], v["layers"], v["heads"], v["mlp"], 0, 0, v.get("image_size", 224),
                                       v["patch"])
            if t:
                d.text = N.TowerDesc(t["width"], t["layers"], t["heads"], t["mlp"], t["ctx"], t["vocab"], 0, 0)
            self.image_size = v.get("image_size", 224) if v else 0
        elif arch == "bert":
            d.arch = N.ARCH_BERT
            d.embed_dim = int(config["width"])
            d.pool = N.POOL_CLS if config.get("pool", "mean") == "cls" else N.POOL_MEAN
            d.type_vocab = int(config.get("type_vocab", 2))
            d.text = N.TowerDesc(config["width"], config["layers"], config["heads"], config["mlp"],
                                 config.get("max_pos", 512), config["vocab"], 0, 0)
            self.image_size = 0
        elif arch == "mpnet":
            if int(config.get("buckets", 32)) != 32 or float(config.get("ln_eps", 1e-5)) != 1e-5:
                raise ValueError("MPNet: only 32 relative-position buckets and LayerNorm eps 1e-5 are implemented")
            d.arch = N.ARCH_MPNET
            d.embed_dim = int(config["width"])
            d.pool = N.POOL_CLS if config.get("pool", "mean") == "cls" else N.POOL_MEAN
            d.text = N.TowerDesc(config["width"], config["layers"], config["heads"], config["mlp"],
                                 config.get("max_pos", 514), config["vocab"], 0, 0)
            self.image_size = 0
        else:
            raise ValueError(f"unknown arch {arch!r}")
        self.embed_dim = int(d.embed_dim)
        self._stage_ptr, self._stage_bytes = None, 0
        self._stage_lock = threading.Lock()
        self._pool = None
        h = C.c_void_p()
        N.check(self._lib.b200_model_create(self.device, C.byref(d), C.byref(h)))
        self._h = h
        try:
            for name, t in weights.items():
                a = _to_numpy_f32(t)
                N.check(self._lib.b200_model_load_tensor(h, name.encode(), _ptr(a), a.size))
            N.check(self._lib.b200_model_finalize(h))
        except Exception:
            self.close()
            raise

    def close(self) -> None:
        h, self._h = getattr(self, "_h", None), None
        if h:
            self._lib.b200_model_destroy(h)
        pool, self._pool = getattr(self, "_pool", None), None
        if pool is not None:
            pool.shutdown(wait=False)
        st, self._stage_ptr = getattr(self, "_stage_ptr", None), None
        if st:
            self._lib.b200_host_free(st)
            self._stage_bytes = 0

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _handle(self):
        if not self._h:
            raise RuntimeError("Encoder is closed")
        return self._h

    def _staging(self, nbytes: int) -> np.ndarray:
        """A reusable page-locked uint8 buffer of at least nbytes (caller holds self._stage_lock)."""
        if getattr(self, "_stage_bytes", 0) < nbytes:
            if getattr(self, "_stage_ptr", None):
                self._lib.b200_host_free(self._stage_ptr)
                self._stage_ptr, self._stage_bytes = None, 0
            want = int(nbytes * 1.25) + 4096
            p = C.c_void_p()
            N.check(self._lib.b200_host_alloc(want, C.byref(p)))
            self._stage_ptr, self._stage_bytes = p, want
        return np.ctypeslib.as_array((C.c_uint8 * self._stage_bytes).from_address(self._stage_ptr.value))

    def encode_images_u8_list(self, images: Sequence[np.ndarray], normalize: bool = True) -> np.ndarray:
        """uint8 HWC images of ONE size, given one by one (what Marqo's download threads hand over): they are
        assembled in a reusable page-locked staging buffer — no fresh 38 MB allocation per batch, full-rate H2D."""
        n = len(images)
        if n == 0:
            raise ValueError("expected at least one image")
        h, w = images[0].shape[:2]
        out = np.empty((n, self.embed_dim), np.float32)
        with self._stage_lock:
            buf = self._staging(n * h * w * 3)[: n * h * w * 3].reshape(n, h, w, 3)
            for i, a in enumerate(images):
                if a.shape != (h, w, 3) or a.dtype != np.uint8:
                    raise ValueError(f"image {i}: expected uint8 [{h}, {w}, 3], got {a.dtype} {a.shape}")

            def fill(lo: int, hi: int) -> None:
                for i in range(lo, hi):
                    np.copyto(buf[i], images[i])   # releases the GIL for the memcpy

            if n * h * w * 3 >= (8 << 20):   # a 38 MB batch: ~4 ms on one core, < 1 ms on eight
                if self._pool is None:
                    from concurrent.futures import ThreadPoolExecutor
                    self._pool = ThreadPoolExecutor(8, thread_name_prefix="b200-stage")
                step = (n + 7) // 8
                list(self._pool.map(lambda lo: fill(lo, min(n, lo + step)), range(0, n, step)))
            else:
                fill(0, n)
            N.check(self._lib.b200_model_encode_images_u8(self._handle(), C.c_void_p(self._stage_ptr.value), n, h, w,
                                                          1 if normalize else 0, _ptr(out)))
        return out

    def encode_images_u8(self, hwc: np.ndarray, normalize: bool = True) -> np.ndarray:
        a = _as(hwc, np.uint8)
        if a.ndim != 4 or a.shape[3] != 3:
            raise ValueError(f"expected uint8 [n, H, W, 3], got {a.shape}")
        out = np.empty((a.shape[0], self.embed_dim), np.float32)
        N.check(self._lib.b200_model_encode_images_u8(self._handle(), _ptr(a), a.shape[0], a.shape[1], a.shape[2],
                                                      1 if normalize else 0, _ptr(out)))
        return out

    def encode_images_f32(self, chw, normalize: bool = True) -> np.ndarray:
        a = _to_numpy_f32(chw)
        if a.ndim != 4 or a.shape[1] != 3 or a.shape[2] != self.image_size or a.shape[3] != self.image_size:
            raise ValueError(f"expected fp32 [n, 3, {self.image_size}, {self.image_size}], got {a.shape}")
        out = np.empty((a.shape[0], self.embed_dim), np.float32)
        N.check(self._lib.b200_model_encode_images_f32(self._handle(), _ptr(a), a.shape[0], 1 if normalize else 0,
                                                       _ptr(out)))
        return out

    def encode_tokens(self, ids, attn_mask=None, normalize: bool = True) -> np.ndarray:
        i = _as(ids.cpu().numpy() if hasattr(ids, "cpu") else ids, np.int32)
        if i.ndim != 2:
            raise ValueError(f"expected int [n, seq] token ids, got {i.shape}")
        mk = None
        if attn_mask is not None:
            mk = _as(attn_mask.cpu().numpy() if hasattr(attn_mask, "cpu") else attn_mask, np.int32)
            if mk.shape != i.shape:
                raise ValueError("attention mask shape must match ids")
        out = np.empty((i.shape[0], self.embed_dim), np.float32)
        N.check(self._lib.b200_model_encode_tokens(self._handle(), _ptr(i), _ptr(mk), i.shape[0], i.shape[1],
                                                   1 if normalize else 0, _ptr(out)))
        return out

    def encode_images_u8_device(self, d_ptr: int, n: int, h: int, w: int, d_out_ptr: int, normalize: bool = True,
                                sync: bool = True) -> None:
        N.check(self._lib.b200_model_encode_images_u8_device(self._handle(), C.c_void_p(d_ptr), n, h, w,
                                                             1 if normalize else 0, C.c_void_p(d_out_ptr),
                                                             1 if sync else 0))

    def encode_tokens_device(self, d_ids_ptr: int, d_mask_ptr: Optional[int], n: int, seq: int, d_out_ptr: int,
                             normalize: bool = True, sync: bool = True) -> None:
        N.check(self._lib.b200_model_encode_tokens_device(self._handle(), C.c_void_p(d_ids_ptr),
                                                          C.c_void_p(d_mask_ptr) if d_mask_ptr else None, n, seq,
                                                          1 if normalize else 0, C.c_void_p(d_out_ptr),
                                                          1 if sync else 0))

    def set_stream(self, cuda_stream: Optional[int]) -> None:
        """cuda_stream: a cudaStream_t handle (0 = legacy default stream); None restores the private stream."""
        N.check(self._lib.b200_model_set_stream(self._handle(), C.c_void_p(cuda_stream or 0),
                                                0 if cuda_stream is None else 1))

    def set_profiling(self, on: bool) -> None:
        N.check(self._lib.b200_model_set_profiling(self._handle(), 1 if on else 0))

    def profile(self) -> dict:
        g, gn, a, an = C.c_float(0), C.c_int(0), C.c_float(0), C.c_int(0)
        N.check(self._lib.b200_model_profile(self._handle(), C.byref(g), C.byref(gn), C.byref(a), C.byref(an)))
        return {"gemm_ms": g.value, "gemm_launches": gn.value, "attention_ms": a.value, "attention_launches": an.value}

    def last_timing(self) -> Tuple[float, int]:
        ms, n = C.c_float(0), C.c_int(0)
        N.check(self._lib.b200_model_last_timing(self._handle(), C.byref(ms), C.byref(n)))
        return ms.value, n.value


# ---------------------------------------------------------------------------------------------------------
# Kernel-level diagnostics (b200_debug_*)
# ---------------------------------------------------------------------------------------------------------
def debug_gemm(A, W, bias=None, residual=None, act: int = 0, out_bf16: bool = False, in_place: bool = False,
               device: int = 0) -> np.ndarray:
    """act(A @ W^T + bias) (+ residual).  in_place: the kernel writes over the residual's device buffer, as out_proj
    and fc2 write over the residual stream (needs a residual and fp32 output)."""
    A, W = _as(A, np.float32), _as(W, np.float32)
    M, K = A.shape
    Nn = W.shape[0]
    b = None if bias is None else _as(bias, np.float32)
    r = None if residual is None else _as(residual, np.float32)
    out = np.empty((M, Nn), np.float32)
    N.check(N.load().b200_debug_gemm(device, _ptr(A), _ptr(W), _ptr(b), _ptr(r), M, Nn, K, act, 1 if out_bf16 else 0,
                                     1 if in_place else 0, _ptr(out)))
    return out


def debug_patch_embed(images_u8, patch: int, conv_w, mean, std, pos=None, use_gather: bool = True,
                      device: int = 0) -> np.ndarray:
    """ViT patch embedding of uint8 HWC images [n, S, S, 3] -> token rows fp32 [n * (G + 1), N] (class rows zero)."""
    img = _as(images_u8, np.uint8)
    n, S = img.shape[0], img.shape[1]
    w = _as(conv_w, np.float32).reshape(conv_w.shape[0], -1)
    Nn = w.shape[0]
    G = (S // patch) ** 2
    m3, s3 = _as(mean, np.float32), _as(std, np.float32)
    ps = None if pos is None else _as(pos, np.float32)
    out = np.empty((n * (G + 1), Nn), np.float32)
    N.check(N.load().b200_debug_patch_embed(device, _ptr(img), n, S, patch, _ptr(w), Nn, _ptr(m3), _ptr(s3), _ptr(ps),
                                            1 if use_gather else 0, _ptr(out)))
    return out


def debug_attention(qkv, B: int, S: int, W: int, H: int, mask: int = 0, kv_len=None, device: int = 0) -> np.ndarray:
    q = _as(qkv, np.float32)
    kl = None if kv_len is None else _as(kv_len, np.int32)
    out = np.empty((B * S, W), np.float32)
    N.check(N.load().b200_debug_attention(device, _ptr(q), B, S, W, H, mask, _ptr(kl), _ptr(out)))
    return out


def debug_attention_relbias(qkv, B: int, S: int, W: int, H: int, rel_bias, mask: int = 0, kv_len=None,
                            device: int = 0) -> np.ndarray:
    """debug_attention with MPNet's relative-position bias rel_bias [32, H] (checkpoint layout) added to the scores."""
    q = _as(qkv, np.float32)
    rb = _as(rel_bias, np.float32)
    if rb.shape != (32, H):
        raise ValueError(f"expected rel_bias [32, {H}], got {rb.shape}")
    kl = None if kv_len is None else _as(kv_len, np.int32)
    out = np.empty((B * S, W), np.float32)
    N.check(N.load().b200_debug_attention_relbias(device, _ptr(q), B, S, W, H, mask, _ptr(kl), _ptr(rb), _ptr(out)))
    return out


def relative_position_buckets(max_distance: int) -> np.ndarray:
    """The library's relative-position bucket of every d = key - query in [-max_distance, max_distance] (host only)."""
    out = np.empty(2 * max_distance + 1, np.int32)
    N.check(N.load().b200_debug_relative_position_buckets(int(max_distance), _ptr(out)))
    return out


def debug_layernorm(x, gamma, beta, eps: float, device: int = 0) -> np.ndarray:
    x, g, b = _as(x, np.float32), _as(gamma, np.float32), _as(beta, np.float32)
    out = np.empty_like(x)
    N.check(N.load().b200_debug_layernorm(device, _ptr(x), _ptr(g), _ptr(b), eps, x.shape[0], x.shape[1], _ptr(out)))
    return out


def debug_resize(hwc, S: int, device: int = 0) -> np.ndarray:
    a = _as(hwc, np.uint8)
    out = np.empty((a.shape[0], S, S, 3), np.uint8)
    N.check(N.load().b200_debug_resize(device, _ptr(a), a.shape[0], a.shape[1], a.shape[2], S, _ptr(out)))
    return out
