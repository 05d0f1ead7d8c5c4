"""GPU tests of the MPNet sentence encoders (hf/all-mpnet-base-v2 family).

* Kernel level: the tcgen05 attention with the relative-position bias (b200_debug_attention_relbias) against a float64
  torch reference that applies transformers' bucket function, with the bars of test_kernels_gpu.py's attention tests:
  one 128-key block (the MPNet serving shape), packed short sequences, the block kernel through the one-shot kernel's
  range, long sequences, more items than the persistent grid, and bias values large enough to decide the row maximum.
* Model level: every item of seeded tiny and all-mpnet-base-v2-shaped encoders against the float64 restatement
  (tests/_mpnet_oracle.py), as test_encoders_full_batch_gpu.py does for the other encoders.
* Through the seams: vectorise() and encode_to_device() with the offline tokenizer against direct Encoder calls."""
import numpy as np
import pytest
import torch

from _mpnet_oracle import (ALL_MPNET_BASE, MpnetCfg, arch_of, make_mpnet_weights, mpnet_encode, position_bias,
                           ragged_ids, tiny_mpnet)

pytestmark = pytest.mark.gpu

COS_CONTRACT = 1e-3
NORM_CONTRACT = 1e-5


def _bf16(x: torch.Tensor) -> torch.Tensor:
    return x.to(torch.bfloat16).to(torch.float32)


def _dev64(x: torch.Tensor) -> torch.Tensor:
    return x.to("cuda", torch.float64)


def _rel_rms(got: torch.Tensor, ref: torch.Tensor, dim=None) -> torch.Tensor:
    d = _dev64(got) - ref
    if dim is None:
        return d.norm() / ref.norm()
    return d.pow(2).sum(dim).sqrt() / ref.pow(2).sum(dim).sqrt()


def _rel_bias(got: torch.Tensor, ref: torch.Tensor) -> float:
    return float(((_dev64(got) - ref) * ref.sign()).sum() / ref.abs().sum())


def _attention_case(B, S, H, mask, seed, bias_scale=1.0, peaked=False):
    """(qkv bf16-rounded fp32 [B*S, 3W], kv_len or None, rel_bias [32, H], float64 reference output [B*S, W])."""
    g = torch.Generator().manual_seed(seed)
    W = H * 64
    qkv = _bf16(torch.randn(B * S, 3 * W, generator=g))
    if peaked:   # +-30: the bias alone decides which keys hold the row maximum
        rel_bias = 30.0 * (2.0 * torch.randint(0, 2, (32, H), generator=g).float() - 1.0)
    else:
        rel_bias = bias_scale * torch.randn(32, H, generator=g)
    kv_len = None
    if mask == 2:
        kv_len = torch.randint(1, S + 1, (B,), generator=g).to(torch.int32)
        kv_len[0] = S
    q, k, v = _dev64(qkv).view(B, S, 3, H, 64).permute(2, 0, 3, 1, 4)
    att = (q @ k.transpose(-1, -2)) / 8.0 + position_bias(_dev64(rel_bias), S)[None]
    if mask == 2:
        keep = torch.arange(S, device=att.device)[None, :] < kv_len.to(att.device)[:, None]
        att = att.masked_fill(~keep[:, None, None, :], float("-inf"))
    ref = (att.softmax(-1) @ v).permute(0, 2, 1, 3).reshape(B * S, W)
    return qkv, kv_len, rel_bias, ref


def _check_attention(B, S, H, mask, got, ref, rtol=2e-2):
    g64 = _dev64(got)
    assert torch.isfinite(g64).all()
    torch.testing.assert_close(g64, ref, rtol=rtol, atol=rtol)     # P and the output are rounded to bf16
    # the bars of test_attention_matches_torch: worst (item, head) relative RMS and the signed error
    per_head = _rel_rms(g64.view(B, S, H, 64), ref.view(B, S, H, 64), dim=(1, 3))
    rr, rb = float(per_head.max()), _rel_bias(g64, ref)
    print(f"ERRSTAT relbias-attn B={B} S={S} H={H} mask={mask} worst_head_rel_rms={rr:.3e} rel_bias={rb:.3e}")
    assert rr < 4e-3, f"worst (item, head) relative RMS error {rr:.3e}"
    assert abs(rb) < 6e-4, f"relative signed error {rb:.3e}"


@pytest.mark.parametrize("B,S,H,mask", [
    # MPNet serving shapes: one 128-key block
    (256, 128, 12, 2), (8, 128, 12, 2), (8, 128, 12, 0),
    # packed short sequences (128 // S per tile)
    (9, 1, 2, 2), (11, 17, 2, 2), (10, 50, 2, 2), (7, 64, 2, 2), (9, 77, 12, 2), (5, 100, 2, 2), (6, 50, 2, 0),
    # the block kernel through the one-shot kernel's range (S = 129 / 257: one more masked block, no remainder path)
    (4, 129, 2, 2), (4, 200, 2, 2), (3, 257, 2, 0), (3, 257, 12, 2),
    # long sequences
    (3, 385, 2, 2), (4, 512, 12, 2),
    # more items than the persistent grid (2 CTAs x 148 SMs)
    (160, 129, 4, 2), (40, 512, 12, 2),
])
def test_relbias_attention_matches_torch(gpu_required, B, S, H, mask):
    from marqo_b200.engine import debug_attention_relbias
    qkv, kv_len, rel_bias, ref = _attention_case(B, S, H, mask, seed=B * 1000 + S + H)
    got = torch.from_numpy(debug_attention_relbias(qkv.numpy(), B, S, H * 64, H, rel_bias.numpy(), mask,
                                                   None if kv_len is None else kv_len.numpy()))
    _check_attention(B, S, H, mask, got, ref)


@pytest.mark.parametrize("B,S,H,mask", [(8, 128, 4, 2), (10, 50, 2, 2), (3, 257, 2, 0), (3, 512, 2, 2)])
def test_relbias_attention_peaked(gpu_required, B, S, H, mask):
    """Bias values of +-30: the row maximum is set by the bias, so the running reference and the lazy rescale must
    track biased scores."""
    from marqo_b200.engine import debug_attention_relbias
    qkv, kv_len, rel_bias, ref = _attention_case(B, S, H, mask, seed=S + 7, peaked=True)
    got = torch.from_numpy(debug_attention_relbias(qkv.numpy(), B, S, H * 64, H, rel_bias.numpy(), mask,
                                                   None if kv_len is None else kv_len.numpy()))
    _check_attention(B, S, H, mask, got, ref, rtol=3e-2)


def test_relbias_attention_zero_bias_equals_plain(gpu_required):
    """A zero bias gives the plain kernel's output (same scores, same softmax schedule)."""
    from marqo_b200.engine import debug_attention, debug_attention_relbias
    B, S, H = 8, 128, 4
    qkv, kv_len, _, _ = _attention_case(B, S, H, 2, seed=3)
    plain = debug_attention(qkv.numpy(), B, S, H * 64, H, 2, kv_len.numpy())
    zero = debug_attention_relbias(qkv.numpy(), B, S, H * 64, H, np.zeros((32, H), np.float32), 2, kv_len.numpy())
    assert float(np.abs(plain - zero).max()) < 1e-2
    assert float(np.abs(plain - zero).mean()) < 1e-4


# ------------------------------------------------------------------------------------------------ model level
def _encoder(cfg: MpnetCfg, seed, max_batch):
    from marqo_b200.engine import Encoder
    sd = make_mpnet_weights(cfg, seed=seed)
    enc = Encoder("mpnet", arch_of(cfg), sd, max_batch=max_batch)
    return enc, {k: v.to("cuda", torch.float64) for k, v in sd.items()}


def _compare(got, ref, name, cos_bar=COS_CONTRACT):
    got64 = _dev64(torch.as_tensor(np.asarray(got)))
    cos = torch.nn.functional.cosine_similarity(got64, ref)
    worst = float((1 - cos).max())
    diff = (got64 - ref).norm(dim=1)
    print(f"ERRSTAT {name}: worst 1-cos {worst:.2e} worst |d| {float(diff.max()):.2e} mean |d| {float(diff.mean()):.2e}")
    assert worst < cos_bar, f"{name}: worst 1 - cos {worst:.3e}"
    assert float((got64.norm(dim=1) - 1).abs().max()) < NORM_CONTRACT


@pytest.mark.parametrize("pool", ["mean", "cls"])
def test_tiny_mpnet_matches_oracle(gpu_required, pool):
    cfg = tiny_mpnet(pool)
    enc, sd64 = _encoder(cfg, 21, max_batch=16)
    lengths = [128, 1, 2, 57, 128, 100, 3, 64, 127, 9, 33, 128]
    ids, mask = ragged_ids(len(lengths), 128, cfg.vocab, lengths, seed=5)
    got = enc.encode_tokens(ids.numpy(), mask.numpy())
    _compare(got, mpnet_encode(sd64, cfg, ids.cuda(), mask.cuda(), dtype=torch.float64), f"tiny-mpnet {pool}")
    # short rows through the packed tiles (S = 20: six sequences per tile)
    ids, mask = ragged_ids(13, 20, cfg.vocab, [20, 1, 7, 20, 13, 2, 19, 20, 5, 11, 20, 3, 8], seed=6)
    got = enc.encode_tokens(ids.numpy(), mask.numpy())
    _compare(got, mpnet_encode(sd64, cfg, ids.cuda(), mask.cuda(), dtype=torch.float64), f"tiny-mpnet {pool} S=20")
    enc.close()


@pytest.fixture(scope="module")
def mpnet_base():
    enc, sd64 = _encoder(ALL_MPNET_BASE, 1234, max_batch=256)
    yield enc, sd64
    enc.close()


def test_all_mpnet_base_b256_ragged(gpu_required, mpnet_base):
    enc, sd64 = mpnet_base
    g = torch.Generator().manual_seed(9)
    lengths = torch.randint(1, 129, (256,), generator=g).tolist()
    lengths[0] = 128
    ids, mask = ragged_ids(256, 128, ALL_MPNET_BASE.vocab, lengths, seed=10)
    got = enc.encode_tokens(ids.numpy(), mask.numpy())
    ref = torch.cat([mpnet_encode(sd64, ALL_MPNET_BASE, ids[lo:lo + 64].cuda(), mask[lo:lo + 64].cuda(),
                                  dtype=torch.float64) for lo in range(0, 256, 64)])
    _compare(got, ref, "all-mpnet-base b256x128 ragged")
    # the device entry point gives the same bits
    d_ids, d_mask = ids.to(torch.int32).cuda(), mask.to(torch.int32).cuda()
    out = torch.empty(256, 768, device="cuda")
    torch.cuda.synchronize()
    enc.encode_tokens_device(d_ids.data_ptr(), d_mask.data_ptr(), 256, 128, out.data_ptr(), sync=True)
    assert np.array_equal(out.cpu().numpy(), got)


def test_all_mpnet_base_b8_full_and_graph_replay(gpu_required, mpnet_base):
    enc, sd64 = mpnet_base
    ids, mask = ragged_ids(8, 128, ALL_MPNET_BASE.vocab, [128] * 8, seed=11)
    ref = mpnet_encode(sd64, ALL_MPNET_BASE, ids.cuda(), mask.cuda(), dtype=torch.float64)
    runs = [enc.encode_tokens(ids.numpy(), mask.numpy()) for _ in range(3)]   # eager, captured, replayed
    _compare(runs[0], ref, "all-mpnet-base b8x128")
    assert np.array_equal(runs[0], runs[1]) and np.array_equal(runs[0], runs[2])
    raw = enc.encode_tokens(ids.numpy(), mask.numpy(), normalize=False)
    ref_raw = mpnet_encode(sd64, ALL_MPNET_BASE, ids.cuda(), mask.cuda(), normalize=False, dtype=torch.float64)
    rel = (_dev64(torch.from_numpy(raw)) - ref_raw).norm(dim=1) / ref_raw.norm(dim=1)
    assert float(rel.max()) < 4.5e-2


def test_all_mpnet_base_512_tokens(gpu_required, mpnet_base):
    enc, sd64 = mpnet_base
    ids, mask = ragged_ids(8, 512, ALL_MPNET_BASE.vocab, [512, 1, 511, 256, 255, 257, 129, 384], seed=12)
    got = enc.encode_tokens(ids.numpy(), mask.numpy())
    _compare(got, mpnet_encode(sd64, ALL_MPNET_BASE, ids.cuda(), mask.cuda(), dtype=torch.float64),
             "all-mpnet-base b8x512 ragged")
    with pytest.raises(Exception):   # position ids 2 .. S + 1 must exist: 513 tokens is one too many
        enc.encode_tokens(np.full((1, 513), 5, np.int32), None)


# ------------------------------------------------------------------------------------------------ through the seams
def _vocab(tmp_path):
    words = [f"w{i}" for i in range(3000)] + ["##s", ".", ",", "the", "a"]
    lines = ["<s>", "<pad>", "</s>", "<unk>", "[UNK]"] + words + ["<mask>"]
    path = tmp_path / "vocab.txt"
    path.write_text("\n".join(lines) + "\n", encoding="utf-8")
    return path


def test_vectorise_all_mpnet_base_v2(gpu_required, tmp_path, monkeypatch):
    from marqo_b200 import s2_inference as s2, weights as Wt
    from marqo_b200.engine import Encoder
    from marqo_b200.loaders import B200HuggingFace
    from marqo_b200.tokenizers import WordPieceTokenizer
    s2.clear_loaded_models()
    monkeypatch.setenv("MARQO_MAX_VECTORISE_BATCH_SIZE", "64")
    vocab = _vocab(tmp_path)
    props = {"name": "sentence-transformers/all-mpnet-base-v2", "dimensions": 768, "type": "hf", "tokens": 128,
             "random_init": 4321, "vocab_file": str(vocab), "max_batch": 64}
    rng = np.random.default_rng(3)
    sentences = [" ".join(f"W{int(x)}s," for x in rng.integers(0, 3000, size=n)) for n in rng.integers(1, 90, size=23)]
    out = np.asarray(s2.vectorise("hf/all-mpnet-base-v2", sentences, model_properties=props, device="cuda:0",
                                  normalize_embeddings=True))
    assert out.shape == (23, 768)
    assert np.allclose(np.linalg.norm(out, axis=1), 1.0, atol=NORM_CONTRACT)
    # the direct Encoder call on the same tokens gives the same vectors
    arch = s2.validate_model_properties("hf/all-mpnet-base-v2", props)["arch"]
    tok = WordPieceTokenizer(str(vocab), cls_token="<s>", sep_token="</s>", pad_token="<pad>", unk_token="[UNK]")
    t = tok(sentences, max_length=128)
    assert t["input_ids"][0, 0] == 0 and (t["input_ids"][t["attention_mask"] == 0] == 1).all()
    enc = Encoder("mpnet", arch, Wt.random_mpnet_weights(arch, 4321), max_batch=64)
    direct = enc.encode_tokens(t["input_ids"], t["attention_mask"])
    assert np.array_equal(out.astype(np.float32), direct)
    enc.close()
    # batch order is kept
    rev = np.asarray(s2.vectorise("hf/all-mpnet-base-v2", sentences[::-1], model_properties=props, device="cuda:0"))
    assert np.allclose(rev[::-1], out, atol=1e-6)
    # encode_to_device: the same vectors, resident on the GPU
    loader = B200HuggingFace(device="cuda:0", model_properties=s2.validate_model_properties("hf/all-mpnet-base-v2", props))
    loader.load()
    dev = loader.encode_to_device(sentences)
    assert dev.is_cuda and tuple(dev.shape) == (23, 768)
    assert np.allclose(dev.cpu().numpy(), out, atol=1e-6)
    loader.close()
    s2.clear_loaded_models()
