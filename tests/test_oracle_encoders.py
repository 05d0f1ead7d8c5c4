"""Pin the encoder oracle (oracle/encoders.py) against INDEPENDENT implementations of the same architectures:
transformers' CLIPVisionModelWithProjection / CLIPTextModelWithProjection / BertModel instantiated from config
(offline) with the oracle's weights copied in.  open_clip itself is not installed here (SURVEY §8c)."""
import numpy as np
import pytest
import torch

from oracle import encoders as E


def _copy_clip_block(hf_layer, sd, p, width):
    w, b = sd[p + "attn.in_proj_weight"], sd[p + "attn.in_proj_bias"]
    sa = hf_layer.self_attn
    sa.q_proj.weight.data.copy_(w[:width]); sa.q_proj.bias.data.copy_(b[:width])
    sa.k_proj.weight.data.copy_(w[width:2 * width]); sa.k_proj.bias.data.copy_(b[width:2 * width])
    sa.v_proj.weight.data.copy_(w[2 * width:]); sa.v_proj.bias.data.copy_(b[2 * width:])
    sa.out_proj.weight.data.copy_(sd[p + "attn.out_proj.weight"]); sa.out_proj.bias.data.copy_(sd[p + "attn.out_proj.bias"])
    hf_layer.layer_norm1.weight.data.copy_(sd[p + "ln_1.weight"]); hf_layer.layer_norm1.bias.data.copy_(sd[p + "ln_1.bias"])
    hf_layer.layer_norm2.weight.data.copy_(sd[p + "ln_2.weight"]); hf_layer.layer_norm2.bias.data.copy_(sd[p + "ln_2.bias"])
    hf_layer.mlp.fc1.weight.data.copy_(sd[p + "mlp.c_fc.weight"]); hf_layer.mlp.fc1.bias.data.copy_(sd[p + "mlp.c_fc.bias"])
    hf_layer.mlp.fc2.weight.data.copy_(sd[p + "mlp.c_proj.weight"]); hf_layer.mlp.fc2.bias.data.copy_(sd[p + "mlp.c_proj.bias"])


@pytest.mark.parametrize("act", ["gelu", "quickgelu"])
def test_clip_vision_matches_hf(act):
    from transformers import CLIPVisionConfig, CLIPVisionModelWithProjection
    cfg = E.tiny_clip(act)
    sd = E.make_clip_weights(cfg, seed=7)
    v = cfg.vision
    hc = CLIPVisionConfig(hidden_size=v.width, intermediate_size=v.mlp, num_hidden_layers=v.layers,
                          num_attention_heads=v.heads, image_size=v.image_size, patch_size=v.patch,
                          projection_dim=cfg.embed_dim, hidden_act="gelu" if act == "gelu" else "quick_gelu",
                          layer_norm_eps=1e-5, attn_implementation="eager")
    m = CLIPVisionModelWithProjection(hc).eval()
    vm = m.vision_model
    vm.embeddings.patch_embedding.weight.data.copy_(sd["visual.conv1.weight"])
    vm.embeddings.class_embedding.data.copy_(sd["visual.class_embedding"])
    vm.embeddings.position_embedding.weight.data.copy_(sd["visual.positional_embedding"])
    pre = getattr(vm, "pre_layrnorm", None) or getattr(vm, "pre_layernorm")
    pre.weight.data.copy_(sd["visual.ln_pre.weight"]); pre.bias.data.copy_(sd["visual.ln_pre.bias"])
    vm.post_layernorm.weight.data.copy_(sd["visual.ln_post.weight"]); vm.post_layernorm.bias.data.copy_(sd["visual.ln_post.bias"])
    for i, layer in enumerate(vm.encoder.layers):
        _copy_clip_block(layer, sd, f"visual.transformer.resblocks.{i}.", v.width)
    m.visual_projection.weight.data.copy_(sd["visual.proj"].t())
    x = torch.randn(3, 3, 224, 224, generator=torch.Generator().manual_seed(1))
    with torch.no_grad():
        ref = m(pixel_values=x).image_embeds
    got = E.clip_encode_image(sd, cfg, x, normalize=False)
    torch.testing.assert_close(got, ref, rtol=1e-4, atol=1e-4)
    gn = E.clip_encode_image(sd, cfg, x, normalize=True)
    assert torch.allclose(gn.norm(dim=-1), torch.ones(3), atol=1e-6)


def test_clip_text_matches_hf():
    from transformers import CLIPTextConfig, CLIPTextModelWithProjection
    cfg = E.tiny_clip()
    sd = E.make_clip_weights(cfg, seed=8)
    t = cfg.text
    hc = CLIPTextConfig(vocab_size=t.vocab, hidden_size=t.width, intermediate_size=t.mlp, num_hidden_layers=t.layers,
                        num_attention_heads=t.heads, max_position_embeddings=t.ctx, projection_dim=cfg.embed_dim,
                        hidden_act="gelu", layer_norm_eps=1e-5, eos_token_id=t.vocab - 1, bos_token_id=t.vocab - 2,
                        pad_token_id=0, attn_implementation="eager")
    m = CLIPTextModelWithProjection(hc).eval()
    tm = m.text_model
    tm.embeddings.token_embedding.weight.data.copy_(sd["token_embedding.weight"])
    tm.embeddings.position_embedding.weight.data.copy_(sd["positional_embedding"])
    tm.final_layer_norm.weight.data.copy_(sd["ln_final.weight"]); tm.final_layer_norm.bias.data.copy_(sd["ln_final.bias"])
    for i, layer in enumerate(tm.encoder.layers):
        _copy_clip_block(layer, sd, f"transformer.resblocks.{i}.", t.width)
    m.text_projection.weight.data.copy_(sd["text_projection"].t())
    g = torch.Generator().manual_seed(2)
    ids = torch.zeros(4, t.ctx, dtype=torch.long)
    for b, L in enumerate([5, 20, 77, 33]):                       # SOT, tokens, EOT (largest id), zero padding
        ids[b, 0] = t.vocab - 2
        ids[b, 1:L - 1] = torch.randint(1, t.vocab - 2, (L - 2,), generator=g)
        ids[b, L - 1] = t.vocab - 1
    with torch.no_grad():
        ref = m(input_ids=ids).text_embeds
    got = E.clip_encode_text(sd, cfg, ids, normalize=False)
    torch.testing.assert_close(got, ref, rtol=1e-4, atol=1e-4)


@pytest.mark.parametrize("pool", ["mean", "cls"])
def test_bert_matches_hf(pool):
    from transformers import BertConfig, BertModel
    cfg = E.tiny_bert(pool)
    sd = E.make_bert_weights(cfg, seed=9)
    hc = BertConfig(vocab_size=cfg.vocab, hidden_size=cfg.width, num_hidden_layers=cfg.layers,
                    num_attention_heads=cfg.heads, intermediate_size=cfg.mlp, max_position_embeddings=cfg.max_pos,
                    type_vocab_size=cfg.type_vocab, hidden_act="gelu", layer_norm_eps=cfg.ln_eps,
                    hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0, attn_implementation="eager")
    m = BertModel(hc, add_pooling_layer=False).eval()
    missing = m.load_state_dict(sd, strict=False)
    assert not missing.unexpected_keys and all("position_ids" in k for k in missing.missing_keys)
    g = torch.Generator().manual_seed(3)
    ids = torch.randint(1, cfg.vocab, (5, 48), generator=g)
    mask = torch.ones(5, 48, dtype=torch.long)
    for b, L in enumerate([48, 7, 30, 1, 16]):
        mask[b, L:] = 0
        ids[b, L:] = 0
    with torch.no_grad():
        out = m(input_ids=ids, attention_mask=mask)
    # Marqo's pooling + normalise, restated from hugging_face_model.py:194-214
    if pool == "mean":
        last = out.last_hidden_state.masked_fill(~mask[..., None].bool(), 0.0)
        ref = last.sum(dim=1) / mask.sum(dim=1)[..., None]
    else:
        ref = out[0][:, 0]
    ref = torch.nn.functional.normalize(ref, p=2, dim=1)
    got = E.bert_encode(sd, cfg, ids, mask, normalize=True)
    torch.testing.assert_close(got, ref, rtol=1e-4, atol=1e-5)


def test_preprocess_identity_size_is_pure_normalise():
    """For 224x224 inputs Resize/CenterCrop are identities, so the transform is (u8/255 - mean)/std."""
    rng = np.random.default_rng(0)
    img = rng.integers(0, 256, size=(2, 224, 224, 3), dtype=np.uint8)
    got = E.clip_preprocess_u8(img)
    ref = (torch.from_numpy(img).permute(0, 3, 1, 2).float() / 255.0
           - torch.tensor(E.OPENAI_CLIP_MEAN).view(1, 3, 1, 1)) / torch.tensor(E.OPENAI_CLIP_STD).view(1, 3, 1, 1)
    torch.testing.assert_close(got, ref, rtol=0, atol=1e-6)


@pytest.mark.parametrize("arch", ["clip_gelu", "clip_quickgelu", "bert_mean", "bert_cls"])
def test_oracle_dtype_argument(arch):
    """The oracle's compute type is a parameter (float64 gives the high-precision reference of the GPU tests): the
    tiny configurations agree across float32 / float64 to cosine 1 - 1e-6, and each output keeps its dtype."""
    outs = {}
    for dt in (torch.float32, torch.float64):
        if arch.startswith("clip"):
            cfg = E.tiny_clip(arch.split("_")[1])
            sd = E.make_clip_weights(cfg, seed=5)
            px = torch.randn(3, 3, 224, 224, generator=torch.Generator().manual_seed(1))
            ids = torch.zeros(3, 77, dtype=torch.int64)
            ids[:, 0] = cfg.text.vocab - 2
            ids[:, 1:20] = torch.randint(1, cfg.text.vocab - 2, (3, 19), generator=torch.Generator().manual_seed(2))
            ids[:, 20] = cfg.text.vocab - 1
            ids[1, 3:] = 0
            ids[1, 2] = cfg.text.vocab - 1
            outs[dt] = [E.clip_encode_image(sd, cfg, px, dtype=dt), E.clip_encode_text(sd, cfg, ids, dtype=dt),
                        E.clip_encode_image(sd, cfg, px, normalize=False, dtype=dt)]
        else:
            cfg = E.tiny_bert(arch.split("_")[1])
            sd = E.make_bert_weights(cfg, seed=6)
            ids = torch.randint(1, cfg.vocab, (4, 30), generator=torch.Generator().manual_seed(4))
            mask = torch.ones(4, 30, dtype=torch.int64)
            mask[1, 7:] = 0
            mask[3, 1:] = 0
            outs[dt] = [E.bert_encode(sd, cfg, ids, mask, dtype=dt), E.bert_encode(sd, cfg, ids, None, dtype=dt),
                        E.bert_encode(sd, cfg, ids, mask, normalize=False, dtype=dt)]
    for a, b in zip(outs[torch.float32], outs[torch.float64]):
        assert a.dtype == torch.float32 and b.dtype == torch.float64
        cos = torch.nn.functional.cosine_similarity(a.double(), b, dim=-1)
        assert float((1 - cos).max()) < 1e-6, f"float32 vs float64 oracle: min cosine {float(cos.min())}"
        torch.testing.assert_close(a.double().norm(dim=-1), b.norm(dim=-1), rtol=1e-5, atol=0)
