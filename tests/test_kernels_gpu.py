"""Kernel-level numerics tests: each CUDA kernel of the encoder vs a plain PyTorch reference of the same op, computed
on the GPU in float64 (inputs pre-rounded to bf16 where the kernel consumes bf16, so the comparison isolates the
kernel's arithmetic).  Besides the small shapes that reach each kernel's edge cases, every kernel runs at the shapes
the encoders time it at (ViT-L-14 / ViT-B-32 at batch 256, CLIP text at 256 x 77, e5 at 8 x 512 and 8 x 128).

Two kinds of bar: the elementwise one (assert_close) is set by the worst element, and a whole-output one -- the
relative RMS error ||got - ref|| / ||ref|| and the relative signed error sum((got - ref) sign(ref)) / sum|ref| -- is set
from the error the compute type allows and from the value measured on a B200, so that a systematic error of a fraction
of a percent (a mis-scaled tile, head or sub-batch) fails even where every element stays inside the elementwise bar."""
import math

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

# One bf16 rounding (8 significant bits, round to nearest): an error uniform in +-ulp/2, ulp = 2^-7 of the binade, over
# values spread log-uniformly across a binade gives a relative RMS of 2^-7 / sqrt(12) * sqrt(3 / (8 ln 2)) = 1.66e-3 --
# measured 1.66e-3 on every bf16-output GEMM below.  It is the floor of every bf16-output bar; a systematic error shows
# in the signed error, whose floor is ~0.
BF16_ROUND_RMS = 1.66e-3
# Bars on a B200 (NVIDIA B200, 1000 W power limit), each ~10x the worst value measured over the cases of its test, except
# the bf16-output RMS bars: their floor is the format's (above), so they sit at 1.5x it (2.5e-3).
FP32_RMS_BAR, FP32_BIAS_BAR = 3e-5, 2e-5        # fp32-output GEMMs: worst measured 3.1e-6 / 1.9e-6 (K = 4096)
BF16_RMS_BAR, BF16_BIAS_BAR = 2.5e-3, 1.5e-4   # bf16-output GEMMs: worst measured 1.72e-3 (GELU) / 1.3e-5


def _bf16(x: torch.Tensor) -> torch.Tensor:
    return x.to(torch.bfloat16).to(torch.float32)


def _dev64(x: torch.Tensor) -> torch.Tensor:
    return x.to("cuda", torch.float64)


def _rel_rms(got: torch.Tensor, ref: torch.Tensor, dim=None) -> torch.Tensor:
    """||got - ref|| / ||ref|| in fp64 on the reference's device (per slice along `dim` when given)."""
    d = _dev64(got) - ref
    if dim is None:
        return d.norm() / ref.norm()
    return d.pow(2).sum(dim).sqrt() / ref.pow(2).sum(dim).sqrt()


def _rel_bias(got: torch.Tensor, ref: torch.Tensor) -> float:
    """Error along the reference's sign, relative to its mean magnitude: ~0 for unbiased rounding, s for a scale 1 + s."""
    return float(((_dev64(got) - ref) * ref.sign()).sum() / ref.abs().sum())


# production Linears, (M, N, K): every Linear of ViT-L-14 at batch 256 (M = 256 x 257 = 65 792: 1 000 - 4 000 tiles, i.e.
# 7 - 28 per CTA pair); ViT-B-32 image at batch 256 (M = 12 800); the ViT-B-32 text tower at 256 x 77 (M = 19 712);
# e5-large at 8 x 512 (M = 4 096).  Order in each group: qkv, out_proj, fc1, fc2.
VIT_L14_LINEARS = [(65792, 3072, 1024), (65792, 1024, 1024), (65792, 4096, 1024), (65792, 1024, 4096)]
OTHER_LINEARS = [(12800, 768, 768), (12800, 3072, 768), (12800, 768, 3072),
                 (19712, 1536, 512), (19712, 512, 512), (19712, 2048, 512), (19712, 512, 2048),
                 (4096, 3072, 1024), (4096, 1024, 1024), (4096, 4096, 1024)]


def _gemm_inputs(M, N, K, seed, residual=False):
    g = torch.Generator().manual_seed(seed)
    A = _bf16(torch.randn(M, K, generator=g))
    W = _bf16(torch.randn(N, K, generator=g) / math.sqrt(K))
    bias = torch.randn(N, generator=g)
    res = torch.randn(M, N, generator=g) if residual else None
    return A, W, bias, res


@pytest.mark.parametrize("M,N,K", [
    (128, 256, 64), (128, 64, 64), (200, 96, 128), (50, 512, 768), (1000, 768, 768), (257 * 3, 3072, 1024),
    (4096, 1024, 4096), (392, 768, 3072), (12800, 2304, 768), (300, 128, 640),
    *VIT_L14_LINEARS, *OTHER_LINEARS,
])
def test_gemm_matches_torch(gpu_required, M, N, K):
    from marqo_b200.engine import debug_gemm
    A, W, bias, _ = _gemm_inputs(M, N, K, M + N + K)
    got = torch.from_numpy(debug_gemm(A.numpy(), W.numpy(), bias.numpy()))
    ref = _dev64(A) @ _dev64(W).t() + _dev64(bias)
    torch.testing.assert_close(_dev64(got), ref, rtol=2e-4, atol=2e-4)   # fp32 accumulate, different summation order
    # fp32 accumulation of K bf16 products: measured 7e-7 relative RMS at K = 1024, 3.1e-6 at K = 4096, with a small
    # negative signed error (-0.6x the RMS: the accumulator rounds towards zero)
    rr, rb = float(_rel_rms(got, ref)), _rel_bias(got, ref)
    print(f"ERRSTAT gemm M={M} N={N} K={K} rel_rms={rr:.3e} rel_bias={rb:.3e}")
    assert rr < FP32_RMS_BAR, f"relative RMS error {rr:.3e}"
    assert abs(rb) < FP32_BIAS_BAR, f"relative signed error {rb:.3e}"


# the old cases keep their ids ("1", "2"): an activation with a separate residual (fp32) and without one (bf16 out).
# The production cases run the epilogue the model uses for that Linear: qkv = bias, bf16 out; fc1 = bias + GELU /
# QuickGELU, bf16 out; out_proj / fc2 = bias + residual, fp32 out, from a separate residual buffer and in place (the
# output aliases the residual, as the model writes the residual stream x over itself).
_QKV, _OUT, _FC1, _FC2 = VIT_L14_LINEARS


@pytest.mark.parametrize("act,M,N,K,mode", [
    pytest.param(1, 333, 1024, 256, "both", id="1"), pytest.param(2, 333, 1024, 256, "both", id="2"),
    (0, *_QKV, "bf16"), (1, *_FC1, "bf16"), (2, *_FC1, "bf16"),
    (0, *_OUT, "residual"), (0, *_FC2, "residual"), (0, *_OUT, "in_place"), (0, *_FC2, "in_place"),
    (0, 12800, 768, 768, "in_place"), (0, 19712, 512, 2048, "in_place"), (0, 4096, 1024, 4096, "in_place"),
    (1, 12800, 3072, 768, "bf16"), (1, 19712, 2048, 512, "bf16"), (1, 4096, 4096, 1024, "bf16"),
    (0, 4096, 3072, 1024, "bf16"),
])
def test_gemm_epilogues(gpu_required, act, M, N, K, mode):
    from marqo_b200.engine import debug_gemm
    A, W, bias, res = _gemm_inputs(M, N, K, act if mode == "both" else M + N + K + act, residual=mode != "bf16")
    z = _dev64(A) @ _dev64(W).t() + _dev64(bias)
    a = torch.nn.functional.gelu(z) if act == 1 else z * torch.sigmoid(1.702 * z) if act == 2 else z
    del z
    if mode in ("both", "residual", "in_place"):
        got = torch.from_numpy(debug_gemm(A.numpy(), W.numpy(), bias.numpy(), res.numpy(), act=act,
                                          in_place=mode == "in_place"))
        ref = a + _dev64(res)
        torch.testing.assert_close(_dev64(got), ref, rtol=2e-4, atol=3e-4)
        # fp32 output: accumulation noise (measured worst 2.5e-6 at K = 4096, in place or not)
        rr, rb = float(_rel_rms(got, ref)), _rel_bias(got, ref)
        print(f"ERRSTAT epi act={act} M={M} N={N} K={K} mode={mode} f32 rel_rms={rr:.3e} rel_bias={rb:.3e}")
        assert rr < FP32_RMS_BAR, f"relative RMS error {rr:.3e}"
        assert abs(rb) < FP32_BIAS_BAR, f"relative signed error {rb:.3e}"
        del got, ref
    if mode in ("both", "bf16"):
        got_b = torch.from_numpy(debug_gemm(A.numpy(), W.numpy(), bias.numpy(), None, act=act, out_bf16=True))
        torch.testing.assert_close(_dev64(got_b), a, rtol=1e-2, atol=1e-2)     # bf16 output rounding
        # one bf16 rounding of the output: BF16_ROUND_RMS, unbiased (+ the packed-fp16 erf-GELU: 1.72e-3 measured)
        rr, rb = float(_rel_rms(got_b, a)), _rel_bias(got_b, a)
        print(f"ERRSTAT epi act={act} M={M} N={N} K={K} mode={mode} bf16 rel_rms={rr:.3e} rel_bias={rb:.3e}")
        assert rr < BF16_RMS_BAR, f"relative RMS error {rr:.3e}"
        assert abs(rb) < BF16_BIAS_BAR, f"relative signed error {rb:.3e}"


@pytest.mark.parametrize("n,S,patch,N", [
    (3, 224, 14, 1024),    # ViT-L-14: 42-byte pixel rows, one 64-slot k-block each, 3 of its 4 UMMA_K steps issued
    (5, 224, 32, 768),     # ViT-B-32: 96-byte pixel rows = 2 k-blocks, a warp's 32 patches straddle images (49 per image)
    (2, 224, 16, 128),     # ViT-B-16 grid with the BN = 128 tile
    (300, 224, 32, 128),   # more tiles than CTA pairs: the smem ring and the strip buffers wrap
    (1, 112, 8, 256),      # small image: 336-byte rows
    (256, 224, 14, 1024),  # ViT-L-14 at batch 256
    (256, 224, 32, 768),   # ViT-B-32 at batch 256
])
def test_patch_embed_gather_matches_conv(gpu_required, n, S, patch, N):
    """SURVEY §8 (a2): uint8 HWC -> ToTensor -> Normalize -> conv1 fused into the GEMM's operand load.  Reference: the
    torchvision formula (u8/255 - mean)/std in fp32, rounded to bf16 like the kernel's A operand, conv2d in fp32."""
    from marqo_b200.engine import debug_patch_embed
    g = torch.Generator().manual_seed(n * 31 + patch)
    img = torch.randint(0, 256, (n, S, S, 3), generator=g, dtype=torch.uint8)
    K = 3 * patch * patch
    w = _bf16(torch.randn(N, 3, patch, patch, generator=g) / math.sqrt(K))
    G = (S // patch) ** 2
    pos = torch.randn(G + 1, N, generator=g)
    mean = torch.tensor([0.48145466, 0.4578275, 0.40821073])
    std = torch.tensor([0.26862954, 0.26130258, 0.27577711])
    x = (img.permute(0, 3, 1, 2).float() / 255.0 - mean[None, :, None, None]) / std[None, :, None, None]
    ref = torch.nn.functional.conv2d(_dev64(_bf16(x)), _dev64(w), stride=patch)          # [n, N, g, g]
    ref = ref.flatten(2).transpose(1, 2) + _dev64(pos[None, 1:, :])                       # [n, G, N]
    got = torch.from_numpy(debug_patch_embed(img.numpy(), patch, w.numpy(), mean.numpy(), std.numpy(), pos.numpy()))
    got = got.view(n, G + 1, N)
    assert float(got[:, 0].abs().max()) == 0.0                                            # class rows are not this kernel's
    # the kernel normalises with one fma (u * 1/(255 std) - mean/std): a few values land on the other side of a bf16
    # rounding boundary (2^-9 relative) -> compare at bf16-product accuracy, and against the im2col path the same way
    g1 = _dev64(got[:, 1:])
    torch.testing.assert_close(g1, ref, rtol=0, atol=2e-2)
    assert float((g1 - ref).abs().mean()) < 1e-3
    # fp32 output: accumulation noise (measured worst 2.3e-6 / signed 1.5e-6, K = 3072 for patch 32)
    rr, rb = float(_rel_rms(g1, ref)), _rel_bias(g1, ref)
    print(f"ERRSTAT patch n={n} patch={patch} N={N} rel_rms={rr:.3e} rel_bias={rb:.3e}")
    assert rr < FP32_RMS_BAR, f"relative RMS error {rr:.3e}"
    assert abs(rb) < FP32_BIAS_BAR, f"relative signed error {rb:.3e}"
    del g1, ref
    old = torch.from_numpy(debug_patch_embed(img.numpy(), patch, w.numpy(), mean.numpy(), std.numpy(), pos.numpy(),
                                             use_gather=False)).view(n, G + 1, N)
    torch.testing.assert_close(got, old, rtol=0, atol=2e-2)


@pytest.mark.parametrize("B,S,H,mask", [
    (2, 50, 12, 0), (3, 257, 4, 0), (2, 77, 8, 1), (4, 128, 12, 2), (2, 512, 2, 2), (1, 1, 2, 0), (2, 64, 2, 1), (1, 65, 2, 1),
    (2, 129, 2, 0), (2, 136, 2, 2), (2, 137, 2, 0), (3, 385, 2, 2), (2, 129, 2, 1), (2, 260, 2, 1), (1, 300, 2, 1), (2, 256, 4, 0),
    (1, 1025, 2, 0),
    # more work items than the persistent grid (2 x 148 CTAs): every CTA loops over several (batch, head, query block)
    # items, so barrier phases, the K/V ring and the remainder-key staging wrap around
    (40, 257, 8, 0), (32, 385, 4, 2), (160, 129, 2, 1), (80, 128, 4, 2), (12, 512, 8, 2), (100, 130, 3, 0),
    # the one-shot kernel (129 <= S <= 257, attention_os.cu): key-length masks shorter than one / two tiles, the 257th
    # token with a key-length mask, more (batch, head) units than CTAs (Q ring, K / V hand-back and TMEM reuse wrap)
    (5, 200, 2, 2), (6, 257, 2, 2), (3, 256, 2, 2), (90, 257, 4, 0), (170, 197, 2, 2), (2, 255, 3, 0),
    # the encoders' own shapes: ViT-L-14 image at batch 256 (16 heads, one-shot kernel), ViT-B-32 image (packed short
    # sequences) and text at batch 256, ViT-L-14 text at batch 64, e5-large at 8 x 512 (key lengths 1, 511, 512 and
    # around 256) and e5-base at 8 x 128
    (256, 257, 16, 0), (256, 50, 12, 0), (256, 77, 8, 1), (64, 77, 12, 1), (8, 512, 16, 2), (8, 128, 12, 2),
])
def test_attention_matches_torch(gpu_required, B, S, H, mask):
    from marqo_b200.engine import debug_attention
    g = torch.Generator().manual_seed(B * 1000 + S)
    W = H * 64
    qkv = _bf16(torch.randn(B * S, 3 * W, generator=g))
    kv_len = None
    if mask == 2:
        kv_len = torch.randint(1, S + 1, (B,), generator=g).to(torch.int32)
        kv_len[0] = S
        if (B, S) == (8, 512):
            kv_len = torch.tensor([512, 1, 511, 256, 255, 257, 129, 384], dtype=torch.int32)
    q, k, v = _dev64(qkv).view(B, S, 3, H, 64).permute(2, 0, 3, 1, 4)
    att = (q @ k.transpose(-1, -2)) / 8.0
    if mask == 1:
        att = att + torch.full((S, S), float("-inf"), dtype=att.dtype, device=att.device).triu_(1)
    if mask == 2:
        keep = torch.arange(S, device=att.device)[None, :] < kv_len.to(att.device)[:, None]
        att = att.masked_fill(~keep[:, None, None, :], float("-inf"))
    ref = (att.softmax(-1) @ v).permute(0, 2, 1, 3).reshape(B * S, W)
    del att, q, k, v
    got = torch.from_numpy(debug_attention(qkv.numpy(), B, S, W, H, mask, None if kv_len is None else kv_len.numpy()))
    g64 = _dev64(got)
    torch.testing.assert_close(g64, ref, rtol=2e-2, atol=2e-2)     # P and the output are rounded to bf16
    assert (g64 - ref).abs().mean() < 3e-3
    # per (batch item, head) slice: P rounded to bf16 + one rounding of the output (BF16_ROUND_RMS): measured 1.9e-3 -
    # 2.7e-3 on every shape above, so the bar sits at 1.5x the worst (a 1.6 % scale error of one head's scores gives
    # ~1.6e-2 there); signed error: worst 6.2e-5 measured
    per_head = _rel_rms(g64.view(B, S, H, 64), ref.view(B, S, H, 64), dim=(1, 3))
    rr, rb = float(per_head.max()), _rel_bias(g64, ref)
    print(f"ERRSTAT attn B={B} S={S} H={H} mask={mask} worst_head_rel_rms={rr:.3e} rel_bias={rb:.3e}")
    assert rr < 4e-3, f"worst (item, head) relative RMS error {rr:.3e}"
    assert abs(rb) < 6e-4, f"relative signed error {rb:.3e}"


@pytest.mark.parametrize("B,S,H,mask", [(3, 257, 2, 0), (4, 200, 2, 2), (3, 512, 2, 2), (4, 77, 2, 1), (4, 257, 16, 0)])
def test_attention_peaked_scores(gpu_required, B, S, H, mask):
    """Scores with a spread of +-40 (one key dominates most rows): the exponent reference must be the row's true maximum."""
    from marqo_b200.engine import debug_attention
    g = torch.Generator().manual_seed(S)
    W = H * 64
    qkv = torch.randn(B * S, 3 * W, generator=g)
    qkv[:, : 2 * W] *= 3.0                                          # q and k: score std 9, extremes beyond 40
    qkv = _bf16(qkv)
    kv_len = None
    if mask == 2:
        kv_len = torch.randint(1, S + 1, (B,), generator=g).to(torch.int32)
        kv_len[0] = S
    q, k, v = _dev64(qkv).view(B, S, 3, H, 64).permute(2, 0, 3, 1, 4)
    att = (q @ k.transpose(-1, -2)) / 8.0
    if mask == 1:
        att = att + torch.full((S, S), float("-inf"), dtype=att.dtype, device=att.device).triu_(1)
    if mask == 2:
        keep = torch.arange(S, device=att.device)[None, :] < kv_len.to(att.device)[:, None]
        att = att.masked_fill(~keep[:, None, None, :], float("-inf"))
    ref = (att.softmax(-1) @ v).permute(0, 2, 1, 3).reshape(B * S, W)
    got = torch.from_numpy(debug_attention(qkv.numpy(), B, S, W, H, mask, None if kv_len is None else kv_len.numpy()))
    assert torch.isfinite(got).all()
    torch.testing.assert_close(_dev64(got), ref, rtol=3e-2, atol=3e-2)
    # as in test_attention_matches_torch (measured 1.6e-3 - 2.3e-3 here)
    per_head = _rel_rms(got.view(B, S, H, 64), ref.view(B, S, H, 64), dim=(1, 3))
    rr = float(per_head.max())
    print(f"ERRSTAT attn_peaked B={B} S={S} H={H} mask={mask} worst_head_rel_rms={rr:.3e}")
    assert rr < 4e-3, f"worst (item, head) relative RMS error {rr:.3e}"


@pytest.mark.parametrize("rows,w,eps", [(5, 128, 1e-5), (77, 512, 1e-5), (1000, 768, 1e-12), (33, 1024, 1e-5),
                                         (65792, 1024, 1e-5)])   # ViT-L-14 at batch 256
def test_layernorm_matches_torch(gpu_required, rows, w, eps):
    from marqo_b200.engine import debug_layernorm
    g = torch.Generator().manual_seed(rows)
    x = torch.randn(rows, w, generator=g) * 3 + 1
    gamma, beta = torch.randn(w, generator=g), torch.randn(w, generator=g)
    ref = torch.nn.functional.layer_norm(_dev64(x), (w,), _dev64(gamma), _dev64(beta), eps)
    got = torch.from_numpy(debug_layernorm(x.numpy(), gamma.numpy(), beta.numpy(), eps))
    torch.testing.assert_close(_dev64(got), ref, rtol=1e-5, atol=1e-5)
    # fp32 statistics over w values and an fp32 output: a few 2^-24 relative (measured 5.9e-8 / signed 2.4e-8 worst)
    rr, rb = float(_rel_rms(got, ref)), _rel_bias(got, ref)
    print(f"ERRSTAT ln rows={rows} w={w} rel_rms={rr:.3e} rel_bias={rb:.3e}")
    assert rr < 6e-7, f"relative RMS error {rr:.3e}"
    assert abs(rb) < 2.5e-7, f"relative signed error {rb:.3e}"


@pytest.mark.parametrize("h,w", [(480, 640), (640, 480), (224, 224), (300, 224), (256, 256), (1000, 750), (225, 400), (100, 150)])
def test_resize_matches_pillow_bit_exact(gpu_required, h, w):
    """Resize(224, BICUBIC) + CenterCrop(224) on PIL images (clip_utils.py:48-67) — Pillow is the third-party
    implementation the reference runs; the CUDA kernel restates its fixed-point two-pass resampler bit for bit."""
    from PIL import Image
    from torchvision.transforms import CenterCrop, InterpolationMode, Resize
    from marqo_b200.engine import debug_resize
    rng = np.random.default_rng(h * 7 + w)
    imgs = rng.integers(0, 256, size=(3, h, w, 3), dtype=np.uint8)
    imgs[1] = (np.linspace(0, 255, w)[None, :, None] * np.ones((h, 1, 3))).astype(np.uint8)   # smooth gradient
    tf = [Resize(224, interpolation=InterpolationMode.BICUBIC), CenterCrop(224)]
    ref = []
    for a in imgs:
        im = Image.fromarray(a)
        for t in tf:
            im = t(im)
        ref.append(np.asarray(im.convert("RGB")))
    got = debug_resize(imgs, 224)
    np.testing.assert_array_equal(got, np.stack(ref))
