"""CPU checks of the MPNet sentence-encoder support: the torch restatement (tests/_mpnet_oracle.py) against
transformers.MPNetModel, the library's relative-position buckets against transformers' bucket function, and the
special-token WordPiece tokenizer against transformers' MPNetTokenizerFast."""
import numpy as np
import pytest
import torch

from _mpnet_oracle import MpnetCfg, make_mpnet_weights, mpnet_encode, ragged_ids, tiny_mpnet


def _hf_model(cfg: MpnetCfg, sd):
    from transformers import MPNetConfig, MPNetModel
    hf_cfg = MPNetConfig(vocab_size=cfg.vocab, hidden_size=cfg.width, num_hidden_layers=cfg.layers,
                         num_attention_heads=cfg.heads, intermediate_size=cfg.mlp, hidden_act="gelu",
                         max_position_embeddings=cfg.max_pos, relative_attention_num_buckets=cfg.buckets,
                         layer_norm_eps=cfg.ln_eps, hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0)
    model = MPNetModel(hf_cfg, add_pooling_layer=False).eval()
    missing, unexpected = model.load_state_dict(sd, strict=False)
    assert not unexpected and not [k for k in missing if "position_ids" not in k], (missing, unexpected)
    return model


@pytest.mark.parametrize("pool", ["mean", "cls"])
def test_mpnet_encode_matches_transformers(pool):
    cfg = tiny_mpnet(pool)
    sd = make_mpnet_weights(cfg, seed=11)
    model = _hf_model(cfg, sd)
    lengths = [40, 1, 17, 40, 33, 2]
    ids, mask = ragged_ids(len(lengths), 40, cfg.vocab, lengths, seed=1)
    with torch.no_grad():
        last = model(input_ids=ids, attention_mask=mask).last_hidden_state
    if pool == "cls":
        ref = last[:, 0]
    else:
        ref = (last * mask[..., None]).sum(1) / mask.sum(1, keepdim=True)
    ref = torch.nn.functional.normalize(ref, p=2, dim=1)
    got = mpnet_encode(sd, cfg, ids, mask)
    assert float((got - ref).abs().max()) < 1e-4
    # unnormalised too: the pooled vectors themselves
    raw = mpnet_encode(sd, cfg, ids, mask, normalize=False)
    ref_raw = last[:, 0] if pool == "cls" else (last * mask[..., None]).sum(1) / mask.sum(1, keepdim=True)
    assert float((raw - ref_raw).abs().max()) < 1e-4 * float(ref_raw.abs().max())


def test_mpnet_encode_float64_agrees():
    cfg = tiny_mpnet()
    sd = make_mpnet_weights(cfg, seed=12)
    ids, mask = ragged_ids(4, 24, cfg.vocab, [24, 5, 12, 1], seed=2)
    a = mpnet_encode(sd, cfg, ids, mask)
    b = mpnet_encode(sd, cfg, ids, mask, dtype=torch.float64)
    assert b.dtype == torch.float64
    assert float((a.double() - b).abs().max()) < 1e-5


def test_library_buckets_match_transformers(native_lib):
    from transformers.models.mpnet.modeling_mpnet import MPNetEncoder
    from marqo_b200.engine import relative_position_buckets
    D = 1023
    d = torch.arange(-D, D + 1, dtype=torch.long)
    ref = MPNetEncoder.relative_position_bucket(d, num_buckets=32).numpy()
    got = relative_position_buckets(D)
    assert got.shape == ref.shape
    assert (got == ref).all(), np.nonzero(got != ref)[0][:10] - D
    # the thresholds the attention kernels' clamp at |d| = 91 relies on
    for n, b in ((7, 7), (8, 8), (11, 8), (12, 9), (16, 10), (23, 11), (32, 12), (46, 13), (64, 14), (90, 14), (91, 15)):
        assert got[D - n] == b and got[D + n] == b + 16, n


def _vocab_lines():
    words = ["hello", "world", "the", "a", "quick", "brown", "fox", "jump", "##s", "##ed", "##ing", "over", "lazy",
             "dog", "cafe", "naive", "un", "##believ", "##able", ".", ",", "!", "?", "'", "-", "(", ")", "1", "2",
             "##3", "mask", "[", "]", "<", ">", "s", "/", "pad", "cls", "sep", "unk", "é", "中", "文"]
    return ["<s>", "<pad>", "</s>", "<unk>", "[PAD]", "[UNK]", "[CLS]", "[SEP]", "[MASK]"] + words + ["<mask>"]


def _random_sentences(n, seed):
    rng = np.random.default_rng(seed)
    pool = ["hello", "world", "The", "quick", "brown", "fox", "jumps", "jumped", "over", "the", "lazy", "dog", "Café",
            "naïve", "unbelievable", "zebra", "!", "?", ",", ".", "(x)", "123", "<s>", "</s>", "<pad>", "<mask>",
            "[UNK]", "[MASK]", "[CLS]", "中文", "don't", "well-known", "  ", "\t"]
    out = []
    for _ in range(n):
        k = int(rng.integers(0, 30))
        out.append(" ".join(pool[int(i)] for i in rng.integers(0, len(pool), k)))
    return out


@pytest.mark.parametrize("max_length", [6, 16, 128])
def test_wordpiece_special_matches_mpnet_tokenizer(native_lib, tmp_path, max_length):
    from transformers import MPNetTokenizerFast
    from marqo_b200.tokenizers import WordPieceTokenizer
    lines = _vocab_lines()
    vocab_file = tmp_path / "vocab.txt"
    vocab_file.write_text("\n".join(lines) + "\n", encoding="utf-8")
    ref_tok = MPNetTokenizerFast(vocab={t: i for i, t in enumerate(lines)})
    assert ref_tok.pad_token_id == 1
    tok = WordPieceTokenizer(str(vocab_file), cls_token="<s>", sep_token="</s>", pad_token="<pad>", unk_token="[UNK]")
    for seed in range(4):
        texts = _random_sentences(24, seed)
        ref = ref_tok(texts, padding=True, truncation=True, max_length=max_length, return_tensors="np")
        got = tok(texts, padding=True, truncation=True, max_length=max_length, return_tensors="np")
        assert got["input_ids"].shape == ref["input_ids"].shape
        assert (got["input_ids"] == ref["input_ids"]).all(), texts
        assert (got["attention_mask"] == ref["attention_mask"]).all()


def test_wordpiece_default_entry_point_unchanged(native_lib, tmp_path):
    """b200_tokenizer_create_wordpiece and the [CLS] / [SEP] / [PAD] / [UNK] case of the special-token entry point (what
    WordPieceTokenizer now calls by default) give the same ids."""
    import ctypes as C
    from marqo_b200 import _native as N
    from marqo_b200.tokenizers import WordPieceTokenizer, _read
    lines = _vocab_lines()
    vocab_file = tmp_path / "vocab.txt"
    vocab_file.write_text("\n".join(lines) + "\n", encoding="utf-8")
    texts = _random_sentences(40, 7)
    special = WordPieceTokenizer(str(vocab_file))(texts, max_length=32)
    data = _read(str(vocab_file))
    h = C.c_void_p()
    N.check(N.load().b200_tokenizer_create_wordpiece(data, len(data), 1, C.byref(h)))
    plain = WordPieceTokenizer.__new__(WordPieceTokenizer)
    plain._lib, plain._h, plain.model_max_length = N.load(), h, 512
    base = plain(texts, max_length=32)
    plain.close()
    assert (special["input_ids"] == base["input_ids"]).all()
    assert (special["attention_mask"] == base["attention_mask"]).all()
    assert base["input_ids"][0, 0] == lines.index("[CLS]")
    assert (base["input_ids"] == lines.index("[MASK]")).any()   # "[MASK]" in the text is matched verbatim
    # a vocabulary without the requested specials is rejected
    with pytest.raises(N.NativeError):
        WordPieceTokenizer(b"hello\nworld\n", cls_token="<s>", sep_token="</s>", pad_token="<pad>", unk_token="[UNK]")


def test_registry_and_loader_pick_mpnet():
    from marqo_b200 import model_registry as R, weights as Wt
    for name, repo in (("hf/all-mpnet-base-v1", "sentence-transformers/all-mpnet-base-v1"),
                       ("hf/all-mpnet-base-v2", "sentence-transformers/all-mpnet-base-v2"),
                       ("hf/all_datasets_v3_mpnet-base", "flax-sentence-embeddings/all_datasets_v3_mpnet-base"),
                       ("hf/all_datasets_v4_mpnet-base", "flax-sentence-embeddings/all_datasets_v4_mpnet-base")):
        p = R.get_model_properties(name)
        assert p["name"] == repo and p["dimensions"] == 768 and p["tokens"] == 128 and p["type"] == R.TYPE_HF
        a = p["arch"]
        assert (a["family"], a["vocab"], a["max_pos"], a["buckets"], a["ln_eps"]) == ("mpnet", 30527, 514, 32, 1e-5)
    # the numpy random weights carry exactly the restatement's parameter names and shapes
    arch = dict(R.get_model_properties("hf/all-mpnet-base-v2")["arch"], layers=1)
    sd = Wt.random_mpnet_weights(arch, seed=1)
    ref = make_mpnet_weights(MpnetCfg(768, 1, 12, 3072), seed=1)
    assert {k: tuple(v.shape) for k, v in sd.items()} == {k: tuple(v.shape) for k, v in ref.items()}
    # a MPNetForXxx checkpoint's "mpnet." prefix is stripped
    assert set(Wt.strip_hf_prefix({"mpnet." + k: v for k, v in sd.items()}, "mpnet.")) == set(sd)
