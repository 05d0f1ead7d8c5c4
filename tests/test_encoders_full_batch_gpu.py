"""Every item of the encoders' headline batches, through the entry points the benchmark and the serving path call,
against the encoder oracle (oracle/encoders.py) run on the GPU in float64.

test_encoders_gpu.py checks a few items of each batch against the CPU fp32 oracle at the cosine contract; here every
item of every batch is compared with a reference whose own error is negligible, so the bars can sit close to what
the kernels actually achieve:
  * the contract, on every item: cosine >= 1 - 1e-3 and unit norm to 1e-5;
  * regression bars, each ~10x the worst value measured on a B200 (written beside it): the worst per-item 1 - cos,
    the worst per-item |got - ref|_2 (relative to |ref| for un-normalised outputs) and the batch mean of |got - ref|_2.
One batch per model also goes through every entry point -- host buffers, device buffers with sync=True, device buffers
with sync=False on a caller's torch stream (bench.py's headline path), the private stream again after
set_stream(None), and per-kernel profiling on -- and the results must be bit-identical: every reduction on the path
has a fixed order (GEMM k-loop, LayerNorm row sums, attention key blocks, head_proj_kernel's K-slice partials summed
in slice order), so nothing may depend on the stream, the timing events or the launch mode.
"""
import numpy as np
import pytest
import torch

from oracle import encoders as E

pytestmark = pytest.mark.gpu

COS_CONTRACT = 1e-3          # BASELINE.json north star: cosine >= 1 - 1e-3 per vector
NORM_CONTRACT = 1e-5

# Regression bars: (worst 1 - cos, worst |got - ref|_2, mean |got - ref|_2), ~10x the worst value measured on a B200
# (NVIDIA B200, 1000 W power limit) against the fp64 reference, capped at the contract (1e-3 / 0.045).  Measured:
BARS = {
    "vit_l14_image": (4e-5, 2.7e-2, 2.5e-2),     # 3.6e-6, 2.7e-3, 2.5e-3
    "vit_b32_image": (9e-5, 4.2e-2, 3.5e-2),     # 8.8e-6, 4.2e-3, 3.5e-3 (graph / sub-batch / resize runs: within)
    "vit_b32_text": (9e-5, 4.2e-2, 3.3e-2),      # 8.6e-6, 4.1e-3, 3.3e-3
    "vit_l14_text": (9e-5, 4.2e-2, 3.4e-2),      # 8.9e-6, 4.2e-3, 3.4e-3
    # post-LN BERT with these random weights loses ~30x more than the pre-LN CLIP towers: 10x would pass the contract
    "e5_large": (1e-3, 4.5e-2, 4.5e-2),          # 1.4e-4, 1.7e-2, 1.5e-2
    "e5_base": (8.5e-4, 4.5e-2, 4.5e-2),         # 8.5e-5, 1.3e-2, 1.0e-2 (mask runs: within)
}
# normalize=False: |got - ref| / |ref| takes the place of |got - ref| (same measured values as the normalised runs),
# and the norm itself gets a bar of its own: worst | |got| / |ref| - 1 |, measured 3.9e-4 (ViT-B-32 image), 3.3e-4
# (ViT-B-32 text), 1.2e-4 (e5-base)
NORM_BAR = 3e-3

VIT_L14 = "open_clip/ViT-L-14/laion2b_s32b_b82k"     # bench.py's headline model
VIT_B32 = "open_clip/ViT-B-32/laion2b_s34b_b79k"
E5_LARGE = "hf/e5-large-v2"
E5_BASE = "hf/e5-base-v2"


# ------------------------------------------------------------------------------------------------ set-up
def _arch(name, **over):
    from marqo_b200 import model_registry as R
    return dict(R.get_model_properties(name)["arch"], **over)


def _clip_cfg(arch) -> E.ClipCfg:
    v, t = arch.get("vision"), arch.get("text")
    vt = E.TowerCfg(v["width"], v["layers"], v["heads"], v["mlp"], image_size=v.get("image_size", 224),
                    patch=v["patch"]) if v else None
    tt = E.TowerCfg(t["width"], t["layers"], t["heads"], t["mlp"], ctx=t["ctx"], vocab=t["vocab"]) if t else None
    return E.ClipCfg(arch["embed_dim"], vt, tt, act=arch["act"], mean=tuple(arch["mean"]), std=tuple(arch["std"]))


def _bert_cfg(arch) -> E.BertCfg:
    return E.BertCfg(arch["width"], arch["layers"], arch["heads"], arch["mlp"], vocab=arch["vocab"],
                     max_pos=arch["max_pos"], type_vocab=arch["type_vocab"], pool=arch["pool"])


def _clip(arch, max_batch):
    """(Encoder, weights as float64 on the GPU) for seeded random weights of `arch` (as bench.py draws them)."""
    from marqo_b200 import weights as Wt
    from marqo_b200.engine import Encoder
    sd = Wt.random_clip_weights(arch, 1234)
    enc = Encoder("clip", arch, sd, max_batch=max_batch)
    return enc, {k: torch.from_numpy(v).to("cuda", torch.float64) for k, v in sd.items()}


def _bert(arch, max_batch):
    from marqo_b200 import weights as Wt
    from marqo_b200.engine import Encoder
    sd = Wt.random_bert_weights(arch, 1234)
    enc = Encoder("bert", arch, sd, max_batch=max_batch)
    return enc, {k: torch.from_numpy(v).to("cuda", torch.float64) for k, v in sd.items()}


def _text_ids(seed, n, ctx, vocab):
    """CLIP token rows: start token, random ids, end token (the arg-max id) at a random length 3..ctx."""
    g = torch.Generator().manual_seed(seed)
    ids = torch.zeros(n, ctx, dtype=torch.int32)
    for b in range(n):
        L = int(torch.randint(3, ctx + 1, (1,), generator=g))
        ids[b, 0] = vocab - 2
        ids[b, 1:L - 1] = torch.randint(1, vocab - 2, (L - 2,), generator=g, dtype=torch.int32)
        ids[b, L - 1] = vocab - 1
    return ids


def _bert_ids(seed, n, S, lens=None):
    """[CLS] random ids [SEP] rows of S tokens; with `lens`, right-padded to those lengths (prefix mask)."""
    g = torch.Generator().manual_seed(seed)
    ids = torch.cat([torch.full((n, 1), 101), torch.randint(1000, 30000, (n, S - 2), generator=g),
                     torch.full((n, 1), 102)], 1).to(torch.int32)
    if lens is None:
        return ids, None
    mask = (torch.arange(S)[None, :] < torch.tensor(lens)[:, None]).to(torch.int32)
    return ids * mask, mask


def _ref_images(sd64, cfg, img, normalize=True, chunk=64):
    """float64 reference on the GPU; pixels through PIL exactly as the reference's download threads prepare them."""
    out = []
    for lo in range(0, img.shape[0], chunk):
        px = E.clip_preprocess_u8(img[lo:lo + chunk], mean=cfg.mean, std=cfg.std).to("cuda")
        out.append(E.clip_encode_image(sd64, cfg, px, normalize=normalize, dtype=torch.float64))
    return torch.cat(out)


def _ref_text(sd64, cfg, ids, normalize=True):
    return E.clip_encode_text(sd64, cfg, ids.to("cuda"), normalize=normalize, dtype=torch.float64)


def _ref_bert(sd64, cfg, ids, mask, normalize=True):
    return E.bert_encode(sd64, cfg, ids.to("cuda"), None if mask is None else mask.to("cuda"), normalize=normalize,
                         dtype=torch.float64)


# ------------------------------------------------------------------------------------------------ entry points
def _device_runs(enc, n, call):
    """The batch through the device entry point in every mode -> name -> [n, E] fp32 numpy.  `call(d_out, sync)`
    launches one encode into the device buffer d_out; the output is poisoned with NaN before each run."""
    d_out = torch.empty(n, enc.embed_dim, dtype=torch.float32, device="cuda")
    out = {}

    def run(name, sync, stream=None):
        d_out.fill_(float("nan"))
        torch.cuda.synchronize()
        call(d_out, sync)
        if stream is not None:
            stream.synchronize()
        elif not sync:
            torch.cuda.synchronize()
        out[name] = d_out.cpu().numpy()

    run("device sync=True", True)
    s = torch.cuda.Stream()
    enc.set_stream(s.cuda_stream)
    try:
        run("device sync=False on a caller's stream", False, s)
        enc.set_profiling(True)
        run("device sync=False on a caller's stream, profiling on", False, s)
    finally:
        enc.set_profiling(False)
        enc.set_stream(None)
    run("device sync=False on the private stream after set_stream(None)", False)
    return out


def _image_entry_points(enc, img, normalize=True):
    n, h, w, _ = img.shape
    out = {"host": enc.encode_images_u8(img, normalize=normalize)}
    d_img = torch.from_numpy(img).to("cuda")
    out.update(_device_runs(enc, n, lambda d_out, sync: enc.encode_images_u8_device(
        d_img.data_ptr(), n, h, w, d_out.data_ptr(), normalize=normalize, sync=sync)))
    return out


def _token_entry_points(enc, ids, mask=None, normalize=True):
    n, S = ids.shape
    out = {"host": enc.encode_tokens(ids.numpy(), None if mask is None else mask.numpy(), normalize=normalize)}
    d_ids = ids.to(torch.int32).to("cuda")
    d_mask = None if mask is None else mask.to(torch.int32).to("cuda")
    out.update(_device_runs(enc, n, lambda d_out, sync: enc.encode_tokens_device(
        d_ids.data_ptr(), None if d_mask is None else d_mask.data_ptr(), n, S, d_out.data_ptr(), normalize=normalize,
        sync=sync)))
    return out


def _assert_bit_identical(outs):
    host = outs["host"]
    for name, got in outs.items():
        assert np.array_equal(got, host), (f"{name} differs from the host entry point: "
                                           f"max |diff| {np.nanmax(np.abs(got - host))}, NaN {np.isnan(got).sum()}")


# ------------------------------------------------------------------------------------------------ bars
def _check(got, ref, bars, tag, normalized=True):
    """Contract on every item + the regression bars -> (worst 1 - cos, worst dist, mean dist)."""
    g = torch.from_numpy(np.asarray(got)).to("cuda", torch.float64)
    assert g.shape == ref.shape and bool(torch.isfinite(g).all())
    one_m_cos = 1 - torch.nn.functional.cosine_similarity(g, ref, dim=-1)
    dist = (g - ref).norm(dim=-1)
    if not normalized:
        dist = dist / ref.norm(dim=-1)
    wc, wd, md = float(one_m_cos.max()), float(dist.max()), float(dist.mean())
    norm_err = (g.norm(dim=-1) / ref.norm(dim=-1) - 1).abs()
    print(f"ERRSTAT {tag} n={g.shape[0]} worst_1mcos={wc:.3e} (item {int(one_m_cos.argmax())}) worst_dist={wd:.3e} "
          f"mean_dist={md:.3e} worst_norm_err={float(norm_err.max()):.3e}")
    assert wc < COS_CONTRACT, f"{tag}: worst 1 - cos {wc:.3e} at item {int(one_m_cos.argmax())}"
    if normalized:
        assert float((g.norm(dim=-1) - 1).abs().max()) < NORM_CONTRACT
    else:
        assert float(norm_err.max()) < NORM_BAR, f"{tag}: worst norm error {float(norm_err.max()):.3e} at item {int(norm_err.argmax())}"
    bc, bd, bm = bars
    assert wc < bc, f"{tag}: worst 1 - cos {wc:.3e} (bar {bc:.1e}) at item {int(one_m_cos.argmax())}"
    assert wd < bd, f"{tag}: worst |got - ref| {wd:.3e} (bar {bd:.1e}) at item {int(dist.argmax())}"
    assert md < bm, f"{tag}: mean |got - ref| {md:.3e} (bar {bm:.1e})"
    return wc, wd, md


# ------------------------------------------------------------------------------------------------ reference check
def test_fp64_gpu_reference_matches_cpu_oracle(gpu_required):
    """The float64 GPU reference the bars below rest on == the CPU fp32 oracle (itself pinned to transformers and to
    the reference's goldens by the CPU tests) on two items of the headline configuration."""
    arch = _arch(VIT_L14, text=None)
    from marqo_b200 import weights as Wt
    sd = {k: torch.from_numpy(v) for k, v in Wt.random_clip_weights(arch, 1234).items()}
    cfg = _clip_cfg(arch)
    img = np.random.default_rng(0).integers(0, 256, size=(2, 224, 224, 3), dtype=np.uint8)
    cpu = E.clip_encode_image(sd, cfg, E.clip_preprocess_u8(img, mean=cfg.mean, std=cfg.std))
    sd64 = {k: v.to("cuda", torch.float64) for k, v in sd.items()}
    gpu = _ref_images(sd64, cfg, img)
    assert cpu.dtype == torch.float32 and gpu.dtype == torch.float64
    cos = torch.nn.functional.cosine_similarity(cpu.double(), gpu.cpu(), dim=-1)
    assert float((1 - cos).max()) < 1e-6, f"fp64 GPU reference vs CPU fp32 oracle: min cosine {float(cos.min())}"


# ------------------------------------------------------------------------------------------------ every item
def test_vit_l_14_image_batch_256_every_item(gpu_required):
    """bench.py's headline workload restated: ViT-L-14 (laion2b_s32b_b82k arch, image tower only), weights
    random_clip_weights(arch, 1234), 256 images of 224 x 224 uint8 (the first 16 from default_rng(0), the rest from a
    torch generator seeded 0), max_batch 256, the device entry point on a caller's stream."""
    arch = _arch(VIT_L14, text=None)
    enc, sd64 = _clip(arch, 256)
    img = np.empty((256, 224, 224, 3), np.uint8)
    img[:16] = np.random.default_rng(0).integers(0, 256, size=(16, 224, 224, 3), dtype=np.uint8)
    img[16:] = torch.randint(0, 256, (240, 224, 224, 3), dtype=torch.uint8,
                             generator=torch.Generator().manual_seed(0)).numpy()
    outs = _image_entry_points(enc, img)
    enc.close()
    _check(outs["host"], _ref_images(sd64, _clip_cfg(arch), img), BARS["vit_l14_image"], "vit_l14_image")
    _assert_bit_identical(outs)


def test_vit_b_32_image_and_text_batch_256_every_item(gpu_required):
    arch = _arch(VIT_B32)
    cfg = _clip_cfg(arch)
    enc, sd64 = _clip(arch, 256)
    img = np.random.default_rng(1).integers(0, 256, size=(256, 224, 224, 3), dtype=np.uint8)
    ids = _text_ids(4, 256, 77, 49408)
    ids[5, :] = 0
    ids[5, 0], ids[5, 1] = 49406, 49407                        # shortest possible text
    outs_i = _image_entry_points(enc, img)
    outs_t = _token_entry_points(enc, ids)
    # normalize=False on both towers: the norm is checked as well as the direction
    un_i = enc.encode_images_u8(img[:32], normalize=False)
    un_t = enc.encode_tokens(ids[:32].numpy(), normalize=False)
    enc.close()
    _check(outs_i["host"], _ref_images(sd64, cfg, img), BARS["vit_b32_image"], "vit_b32_image")
    _check(outs_t["host"], _ref_text(sd64, cfg, ids), BARS["vit_b32_text"], "vit_b32_text")
    _check(un_i, _ref_images(sd64, cfg, img[:32], normalize=False), BARS["vit_b32_image"], "vit_b32_image_unnorm",
           normalized=False)
    _check(un_t, _ref_text(sd64, cfg, ids[:32], normalize=False), BARS["vit_b32_text"], "vit_b32_text_unnorm",
           normalized=False)
    _assert_bit_identical(outs_i)
    _assert_bit_identical(outs_t)


def test_vit_l_14_text_batch_64_every_item(gpu_required):
    arch = _arch(VIT_L14, vision=None)
    enc, sd64 = _clip(arch, 64)
    ids = _text_ids(3, 64, 77, 49408)
    ids[63, :] = 0
    ids[63, 0], ids[63, 1] = 49406, 49407
    outs = _token_entry_points(enc, ids)
    enc.close()
    _check(outs["host"], _ref_text(sd64, _clip_cfg(arch), ids), BARS["vit_l14_text"], "vit_l14_text")
    _assert_bit_identical(outs)


def test_e5_large_512_tokens_every_item(gpu_required):
    """8 x 512: every row full length, then ragged (key lengths 1, 511, 512 and around 256) with a device mask."""
    arch = _arch(E5_LARGE)
    cfg = _bert_cfg(arch)
    enc, sd64 = _bert(arch, 8)
    ids, _ = _bert_ids(0, 8, 512)
    full = _token_entry_points(enc, ids)
    rids, mask = _bert_ids(0, 8, 512, lens=[512, 1, 511, 256, 255, 257, 129, 384])
    ragged = _token_entry_points(enc, rids, mask)
    enc.close()
    _check(full["host"], _ref_bert(sd64, cfg, ids, None), BARS["e5_large"], "e5_large_full")
    _check(ragged["host"], _ref_bert(sd64, cfg, rids, mask), BARS["e5_large"], "e5_large_ragged")
    _assert_bit_identical(full)
    _assert_bit_identical(ragged)


@pytest.mark.parametrize("pool", ["mean", "cls"])
def test_e5_base_pooling_every_item(gpu_required, pool):
    """8 x 128 ragged (one row full length: the mean's divisor is S there), plus normalize=False for the BERT head."""
    arch = _arch(E5_BASE, pool=pool)
    cfg = _bert_cfg(arch)
    enc, sd64 = _bert(arch, 8)
    ids, mask = _bert_ids(1, 8, 128, lens=[128, 1, 16, 64, 127, 100, 65, 128])
    outs = _token_entry_points(enc, ids, mask)
    un = enc.encode_tokens(ids.numpy(), mask.numpy(), normalize=False)
    enc.close()
    _check(outs["host"], _ref_bert(sd64, cfg, ids, mask), BARS["e5_base"], f"e5_base_{pool}")
    _check(un, _ref_bert(sd64, cfg, ids, mask, normalize=False), BARS["e5_base"], f"e5_base_{pool}_unnorm",
           normalized=False)
    _assert_bit_identical(outs)


# ------------------------------------------------------------------------------------------------ device-path edges
def test_device_entry_graph_replay_with_new_contents(gpu_required):
    """ViT-B-32, n = 16 on the private stream: the 1st call of a shape runs eagerly, the 2nd is captured into a CUDA
    graph, the 3rd replays it.  New pixels go into the SAME device buffer each time; every result must equal the host
    entry point bit for bit (the graph reads the buffer, it does not bake the first contents in)."""
    arch = _arch(VIT_B32)
    enc, sd64 = _clip(arch, 256)
    rng = np.random.default_rng(7)
    d_img = torch.empty(16, 224, 224, 3, dtype=torch.uint8, device="cuda")
    d_out = torch.empty(16, enc.embed_dim, dtype=torch.float32, device="cuda")
    batches, got = [], []
    for _ in range(3):
        img = rng.integers(0, 256, size=(16, 224, 224, 3), dtype=np.uint8)
        d_img.copy_(torch.from_numpy(img))
        d_out.fill_(float("nan"))
        torch.cuda.synchronize()
        enc.encode_images_u8_device(d_img.data_ptr(), 16, 224, 224, d_out.data_ptr(), sync=True)
        batches.append(img)
        got.append(d_out.cpu().numpy())
    host = [enc.encode_images_u8(img) for img in batches]
    enc.close()
    cfg = _clip_cfg(arch)
    for i in range(3):
        assert np.array_equal(got[i], host[i]), f"call {i + 1} (eager, captured, replayed) differs from the host entry"
        _check(got[i], _ref_images(sd64, cfg, batches[i]), BARS["vit_b32_image"], f"graph_call_{i + 1}")
    assert not np.array_equal(got[1], got[2])


def test_device_entry_sub_batches(gpu_required):
    """n > max_batch on both device entry points: the call runs in sub-batches of max_batch; every item, in
    particular the ones either side of each sub-batch boundary, matches the reference."""
    arch = _arch(VIT_B32)
    cfg = _clip_cfg(arch)
    enc, sd64 = _clip(arch, 8)
    n = 20                                                          # sub-batches [0, 8), [8, 16), [16, 20)
    img = np.random.default_rng(8).integers(0, 256, size=(n, 224, 224, 3), dtype=np.uint8)
    ids = _text_ids(9, n, 77, 49408)
    d_img, d_ids = torch.from_numpy(img).to("cuda"), ids.to("cuda")
    d_oi = torch.full((n, enc.embed_dim), float("nan"), device="cuda")
    d_ot = torch.full((n, enc.embed_dim), float("nan"), device="cuda")
    torch.cuda.synchronize()
    enc.encode_images_u8_device(d_img.data_ptr(), n, 224, 224, d_oi.data_ptr(), sync=True)
    enc.encode_tokens_device(d_ids.data_ptr(), None, n, 77, d_ot.data_ptr(), sync=True)
    gi, gt = d_oi.cpu().numpy(), d_ot.cpu().numpy()
    whole_i = enc.encode_images_u8(img[:8])                       # one whole sub-batch through the host entry
    enc.close()
    ri, rt = _ref_images(sd64, cfg, img), _ref_text(sd64, cfg, ids)
    _check(gi, ri, BARS["vit_b32_image"], "sub_batch_image")
    _check(gt, rt, BARS["vit_b32_text"], "sub_batch_text")
    assert np.array_equal(gi[:8], whole_i)


def test_device_entry_resize(gpu_required):
    """480 x 640 uint8 images through encode_images_u8_device: the bicubic resize + centre crop kernel runs first;
    the reference resizes with PIL (clip_preprocess_u8)."""
    arch = _arch(VIT_B32)
    enc, sd64 = _clip(arch, 256)
    img = np.random.default_rng(10).integers(0, 256, size=(16, 480, 640, 3), dtype=np.uint8)
    img[3] = (np.linspace(0, 255, 640)[None, :, None] * np.ones((480, 1, 3))).astype(np.uint8)   # smooth gradient
    outs = _image_entry_points(enc, img)
    enc.close()
    _check(outs["host"], _ref_images(sd64, _clip_cfg(arch), img), BARS["vit_b32_image"], "resize_480x640")
    _assert_bit_identical(outs)


def test_device_entry_tokens_with_and_without_mask(gpu_required):
    """encode_tokens_device on e5-base: no mask (every key counts), an all-ones device mask (the same result), and a
    ragged device mask."""
    arch = _arch(E5_BASE)
    cfg = _bert_cfg(arch)
    enc, sd64 = _bert(arch, 16)
    ids, _ = _bert_ids(11, 6, 96)
    rids, mask = _bert_ids(11, 6, 96, lens=[96, 40, 1, 95, 48, 72])
    ones = torch.ones_like(ids)
    outs = {}
    for name, i, m in (("none", ids, None), ("ones", ids, ones), ("ragged", rids, mask)):
        d_i = i.to("cuda")
        d_m = None if m is None else m.to("cuda")
        d_o = torch.full((6, enc.embed_dim), float("nan"), device="cuda")
        torch.cuda.synchronize()
        enc.encode_tokens_device(d_i.data_ptr(), None if d_m is None else d_m.data_ptr(), 6, 96, d_o.data_ptr(),
                                 sync=True)
        outs[name] = d_o.cpu().numpy()
    enc.close()
    assert np.array_equal(outs["none"], outs["ones"])
    _check(outs["none"], _ref_bert(sd64, cfg, ids, None), BARS["e5_base"], "mask_none")
    _check(outs["ragged"], _ref_bert(sd64, cfg, rids, mask), BARS["e5_base"], "mask_ragged")
