#!/usr/bin/env python
"""bench.py — the measurement contract of this repo (see DESIGN.md §Measurement).

Headline workload (BASELINE.json `metric`): open_clip/ViT-L-14 image vectorise, batch 256 per GPU, synthetic
224x224 uint8 RGB, random-init weights of that architecture.  One "step" = one pass of the hot path over one batch:
uint8 pixels -> patch-embed GEMM whose gather warps read the pixels, apply ToTensor/Normalize and fill the tcgen05 A
operand in shared memory (no patch matrix in HBM) -> ViT-L-14 (tcgen05 GEMMs with fused epilogues, one-shot tcgen05
attention with P in TMEM) -> projection -> L2-normalised fp32 embeddings.  Weak scaling: every rank encodes its own batch of 256 (doc-sharded, no collective).

Blocks in the same JSON line (all driver-visible):
  topk     exact top-10 of 64 queries over a 10 M x 768 fp16 corpus row-sharded across the ranks; the per-shard blocks
           are exchanged by ONE fused peer-store kernel over NVLink (NCCL all-gather when IPC is unavailable) and merged
           on the device; `e2e` = host queries in -> merged ids out, max over ranks.
  api_e2e  the repo's public Python API driven from 8 threads: s2_inference.vectorise() and GpuTensorIndex.query().
  cfg2     open_clip/ViT-B-32 image + text vectorise, batch 256 (BASELINE.json configs[1]).
  cfg3     add_documents fast path sample: image + caption towers + index append (configs[2] shape, bounded docs/GPU).

Full-size secondary configurations run behind --config:
    python bench.py --config cfg3 [--docs 100000]     ViT-L-14 add_documents, 100 k image-text docs over the ranks
    python bench.py --config cfg4 [--chunks 1000000]  e5-large-v2, 512-token chunks from on-device ids
    python bench.py --config cfg2                     ViT-B-32 b256 image + text

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--skip-topk] [--skip-api]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

`--dump-outputs DIR` writes what the last timed step returned, as DIR/<name>.npy: the headline's embeddings and, unless
--skip-topk, the merged top-k (doc, row, score).  Inputs and weights are seeded, so two builds run with the same
arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

MODEL = "open_clip/ViT-L-14/laion2b_s32b_b82k"
MODEL_B32 = "open_clip/ViT-B-32/laion2b_s34b_b79k"
MODEL_E5L = "hf/e5-large-v2"
BATCH = 256
IMG = 224
TOPK_ROWS_TOTAL = 10_000_000
TOPK_DIM = 768
TOPK_NQ = 64
TOPK_K = 10
METRIC = "embeddings/s (open_clip/ViT-L-14 image vectorise, batch 256 per GPU)"
REF_SUB_BATCH = 16      # MARQO_MAX_VECTORISE_BATCH_SIZE default (src/marqo/api/configs.py:38): the reference's own sub-batch

_REAL_STDOUT = None


def claim_stdout():
    """Libraries (NCCL's version banner, torchrun warnings) write to fd 1; the contract is ONE JSON line on stdout.
    Everything else is diverted to stderr and the JSON line is written to the original stdout at the end."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line: dict):
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def host_threads() -> int:
    """Threads this process may actually use: the affinity mask capped by the cgroup CPU quota (a 128-CPU mask
    under an 8-CPU quota runs torch 16x oversubscribed and several times slower), not the box's core count."""
    try:
        n = max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        n = os.cpu_count() or 1
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            with open(path) as f:
                parts = f.read().split()
            if path.endswith("cpu.max"):
                if parts[0] != "max":
                    n = min(n, max(1, -(-int(parts[0]) // int(parts[1]))))
            else:
                quota = int(parts[0])
                if quota > 0:
                    with open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as f:
                        n = min(n, max(1, -(-quota // int(f.read().split()[0]))))
            break
        except (OSError, ValueError, IndexError):
            continue
    return n


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


def load_traffic():
    """DRAM bytes per launch of the dominant kernels, read from the committed ncu capture summary (profiles/)."""
    for name in ("r02_traffic.json", "r01_traffic.json"):
        p = os.path.join(ROOT, "profiles", name)
        if os.path.exists(p):
            with open(p) as f:
                d = json.load(f)
            d["_file"] = name
            return d
    return {}


def vit_flops(arch_vision: dict, batch: int):
    """Algorithmic FLOPs of one step: (total, in GEMM kernels, in attention)."""
    w, L, mlp, p = arch_vision["width"], arch_vision["layers"], arch_vision["mlp"], arch_vision["patch"]
    g = arch_vision.get("image_size", 224) // p
    S = g * g + 1
    gemm = L * 2 * S * (4 * w * w + 2 * w * mlp) + 2 * (S - 1) * 3 * p * p * w
    attn = L * 4 * S * S * w
    return batch * (gemm + attn), batch * gemm, batch * attn


def text_flops(t: dict, batch: int, seq: int):
    w, L, mlp = t["width"], t["layers"], t["mlp"]
    return batch * (L * 2 * seq * (4 * w * w + 2 * w * mlp) + L * 4 * seq * seq * w)


def headline_config(world: int) -> dict:
    return {"workload": "open_clip/ViT-L-14 image vectorise: uint8 224x224x3 -> 768-d L2-normalised fp32 "
                        "embeddings, batch 256 per GPU, random-init weights (seed 1234)",
            "model": MODEL, "global_batch": BATCH * world, "parallelism": f"doc-shard x{world} (no collective)",
            "l2_flush": "not needed: each step streams ~1.6 GB of activations + 0.6 GB of weights, far larger "
                        "than the 126 MB L2",
            "residual_stream": "fp32", "accumulate": "fp32"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu_index = gpu_index
        self.proc = None
        self.lines = []
        self.thread = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu_index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._pump, daemon=True)
        self.thread.start()

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.perf_counter(), line.strip()))

    def stop(self, t0: float, t1: float) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, pw = [], [], set(), []
        for ts, line in self.lines:
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 8 or not (t0 - 0.05 <= ts <= t1 + 0.15):
                continue
            try:
                sm.append(float(parts[1]))
                mx.append(float(parts[2]))
                pw.append(float(parts[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), parts[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------ reference arm
def oracle_embed_step(sd, cfg, pixels_u8):
    """The reference's CPU path for this workload, restated by the oracle: per-image PIL transform
    (add_docs.py:129-134) then OPEN_CLIP.encode_image in sub-batches of 16 (MARQO_MAX_VECTORISE_BATCH_SIZE default)."""
    import torch
    from oracle import encoders as E
    px = E.clip_preprocess_u8(pixels_u8, mean=cfg.mean, std=cfg.std)
    outs = []
    for i in range(0, px.shape[0], REF_SUB_BATCH):
        outs.append(E.clip_encode_image(sd, cfg, px[i:i + REF_SUB_BATCH]))
    return torch.cat(outs)


def make_oracle_model():
    import torch
    from oracle import encoders as E
    from marqo_b200 import model_registry as R, weights as Wt
    arch = R.get_model_properties(MODEL)["arch"]
    cfg = E.ClipCfg(arch["embed_dim"], E.CLIP_VIT_L_14.vision, E.CLIP_VIT_L_14.text, act=arch["act"], mean=arch["mean"],
                    std=arch["std"])
    varch = dict(arch, text=None)
    sd = {k: torch.from_numpy(v) for k, v in Wt.random_clip_weights(varch, 1234).items()}
    return sd, cfg


def reference_sample_images(n: int) -> np.ndarray:
    """The first n images of rank 0's synthetic batch (same generator as the b200 arm's host copy)."""
    rng = np.random.default_rng(0)
    return rng.integers(0, 256, size=(n, IMG, IMG, 3), dtype=np.uint8)


def run_reference(args, rank: int, world: int):
    """`--impl reference`: the CPU restatement of the reference's PyTorch path (kind "port": the reference package
    itself cannot be installed here — DESIGN.md §4).  One step = ONE sub-batch of 16 images (the reference's default
    vectorise sub-batch), torch threads = the cores this process may use, warm-up on the same shape.  If a step is so
    slow that K + W of them would not finish in a few minutes the sample shrinks (and says so)."""
    if rank != 0:
        return
    import torch
    threads = host_threads()
    torch.set_num_threads(threads)
    sd, cfg = make_oracle_model()
    sample = REF_SUB_BATCH
    img = reference_sample_images(sample)
    t0 = time.perf_counter()
    oracle_embed_step(sd, cfg, img)              # first touch: allocator, thread pool
    first = time.perf_counter() - t0
    budget_s = 200.0
    total_steps = args.steps + max(args.warmup, 1)
    if first * total_steps > budget_s:
        sample = max(2, int(sample * budget_s / (first * total_steps)))
        img = img[:sample]
    for _ in range(max(args.warmup, 1)):
        oracle_embed_step(sd, cfg, img)
    per_step = []
    for _ in range(args.steps):
        t0 = time.perf_counter()
        oracle_embed_step(sd, cfg, img)
        per_step.append(time.perf_counter() - t0)
    dt = sum(per_step)
    v = sample * args.steps / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": "embeddings/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": headline_config(world),
        "cpu_baseline": {"value": v, "unit": "embeddings/s", "cores": threads, "kind": "port",
                         "sample": f"one vectorise sub-batch of {sample} synthetic 224x224 images per step "
                                   f"(PIL-equivalent preprocess + ViT-L-14 fp32 on host cores)",
                         "step_spread": (max(per_step) - min(per_step)) / statistics.median(per_step)},
        "e2e": {"value": v, "unit": "embeddings/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ------------------------------------------------------------------------------------------------ helpers for our arm
class Ctx:
    pass


def make_ctx(args):
    import torch
    import torch.distributed as dist
    c = Ctx()
    c.args = args
    c.rank = int(os.environ.get("RANK", "0"))
    c.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    c.world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: marqo_b200 has no CPU fallback")
    torch.cuda.set_device(c.local_rank)
    c.dev = torch.device("cuda", c.local_rank)
    c.distributed = c.world > 1
    if c.distributed:
        dist.init_process_group("nccl", device_id=c.dev)
    c.peaks = load_peaks()
    c.traffic = load_traffic()
    c.stream = torch.cuda.Stream(device=c.dev)      # the engine and the timing events share this stream
    torch.cuda.set_stream(c.stream)

    def barrier():
        if c.distributed:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if not c.distributed:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=c.dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(x: float) -> float:
        if not c.distributed:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=c.dev)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    c.barrier, c.max_over_ranks, c.sum_over_ranks = barrier, max_over_ranks, sum_over_ranks
    c.outputs = {}                                  # name -> array returned by the last timed step (--dump-outputs)
    return c


def dump_outputs(directory: str, outputs: dict):
    """DIR/<name>.npy per array: float32 stays float32, any other dtype (ids, fp64 scores) is written as float64."""
    os.makedirs(directory, exist_ok=True)
    for name, a in outputs.items():
        a = np.asarray(a)
        np.save(os.path.join(directory, name + ".npy"), a if a.dtype == np.float32 else a.astype(np.float64))


def timed_steps(c, step, steps: int, warmup: int):
    """W untimed + exactly K timed steps between barriers; device time by CUDA events on the launching stream; max over
    ranks.  -> ms per step."""
    import torch
    for _ in range(warmup):
        step()
    c.barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(c.stream)
    for _ in range(steps):
        step()
    ev1.record(c.stream)
    c.barrier()
    return c.max_over_ranks(ev0.elapsed_time(ev1)) / steps


# ------------------------------------------------------------------------------------------------ headline
def bench_headline(c):
    import torch
    from marqo_b200 import model_registry as R, weights as Wt
    from marqo_b200.engine import Encoder
    args, dev = c.args, c.dev
    props = R.get_model_properties(MODEL)
    arch = dict(props["arch"], text=None)      # image tower only: the metric is image embeddings/s
    sd = Wt.random_clip_weights(arch, 1234)
    enc = Encoder("clip", arch, sd, device=c.local_rank, max_batch=BATCH)
    del sd
    enc.set_stream(c.stream.cuda_stream)
    E = enc.embed_dim
    img_host = torch.empty(BATCH, IMG, IMG, 3, dtype=torch.uint8).pin_memory()
    if c.rank == 0:
        img_host.numpy()[:REF_SUB_BATCH] = reference_sample_images(REF_SUB_BATCH)   # shared with the reference arm
        g = torch.Generator().manual_seed(0)
        img_host[REF_SUB_BATCH:] = torch.randint(0, 256, (BATCH - REF_SUB_BATCH, IMG, IMG, 3), dtype=torch.uint8, generator=g)
    else:
        g = torch.Generator().manual_seed(c.rank)
        img_host.copy_(torch.randint(0, 256, (BATCH, IMG, IMG, 3), dtype=torch.uint8, generator=g))
    img_dev = img_host.to(dev)
    out_dev = torch.empty(BATCH, E, dtype=torch.float32, device=dev)
    flops_total, flops_gemm, flops_attn = vit_flops(arch["vision"], BATCH)

    def step():
        enc.encode_images_u8_device(img_dev.data_ptr(), BATCH, IMG, IMG, out_dev.data_ptr(), normalize=True, sync=False)

    # ---- `value`: K steps, NO per-kernel events inside the timed region
    enc.set_profiling(False)
    for _ in range(args.warmup):
        step()
    c.barrier()
    sampler = ClockSampler(c.local_rank)
    if c.rank == 0:
        sampler.start()
        time.sleep(0.25)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    c.barrier()
    w0 = time.perf_counter()
    ev0.record(c.stream)
    for _ in range(args.steps):
        step()
    ev1.record(c.stream)
    c.barrier()
    w1 = time.perf_counter()
    if args.dump_outputs:
        c.outputs["embeddings"] = out_dev.cpu().numpy()
    launches = enc.last_timing()[1] * args.steps
    step_ms = c.max_over_ranks(ev0.elapsed_time(ev1)) / args.steps
    clocks = sampler.stop(w0, w1) if c.rank == 0 else None
    value = BATCH * c.world / (step_ms / 1e3)
    assert bool(torch.isfinite(out_dev).all()), "non-finite embeddings"

    # ---- roofline numerator: the same steps again with per-kernel-class CUDA events (separate region)
    prof_steps = max(3, min(args.steps, 10))
    enc.set_profiling(True)
    step()
    c.barrier()
    enc.set_profiling(True)                    # resets the sums
    p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    p0.record(c.stream)
    for _ in range(prof_steps):
        step()
    p1.record(c.stream)
    c.barrier()
    prof_ms = p0.elapsed_time(p1)
    pr = enc.profile()
    gemm_ms, gemm_n, attn_ms, attn_n = pr["gemm_ms"], pr["gemm_launches"], pr["attention_ms"], pr["attention_launches"]
    enc.set_profiling(False)

    # ---- e2e: C-ABI call with HOST buffers (H2D + encode + D2H inside the timed region)
    img_host_np = img_host.numpy()
    e2e_steps = max(3, min(args.steps, 10))
    out_host = enc.encode_images_u8(img_host_np, normalize=True)
    c.barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        out_host = enc.encode_images_u8(img_host_np, normalize=True)    # H2D + encode + D2H, synchronous
    torch.cuda.synchronize()
    e2e_ms = c.max_over_ranks((time.perf_counter() - t0) * 1e3) / e2e_steps
    e2e_value = BATCH * c.world / (e2e_ms / 1e3)
    e2e_launches = enc.last_timing()[1]
    assert np.isfinite(out_host).all()
    enc.close()
    del img_dev, out_dev
    torch.cuda.empty_cache()

    peak_tf = c.peaks["bf16_tflops_sustained"]
    gemm_avg_ms = gemm_ms / max(gemm_n, 1)
    ach_tf = (flops_gemm * prof_steps / max(gemm_n, 1)) / (gemm_avg_ms / 1e3) / 1e12 if gemm_n else 0.0
    tr = c.traffic.get("gemm_gemm_kernel_256", {})
    res = {
        "value": value, "step_ms": step_ms, "clocks": clocks, "tflops": flops_total / (step_ms / 1e3) / 1e12,
        "roofline": {"bound": "tensor", "achieved": ach_tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": ach_tf / peak_tf,
                     "traffic": tr.get("avg"),
                     "traffic_note": f"mean dram__bytes_read+write per launch over the GEMMs of a ViT-L-14 layer "
                                     f"(ncu --set full, profiles/{c.traffic.get('_file', 'n/a')})",
                     "kernel": "gemm::gemm_kernel (all shapes of the step)",
                     "launches_timed": gemm_n, "avg_launch_ms": gemm_avg_ms,
                     "flops_per_launch_avg": flops_gemm * prof_steps / max(gemm_n, 1),
                     "peak_source": f"{c.peaks['source']} bf16 sustained",
                     "step_share": gemm_ms / max(prof_ms, 1e-9), "attention_share": attn_ms / max(prof_ms, 1e-9),
                     "attention_ms_per_launch": attn_ms / max(attn_n, 1),
                     "attention_tflops": (flops_attn * prof_steps / max(attn_n, 1)) / (attn_ms / max(attn_n, 1) / 1e3) / 1e12
                     if attn_n else None,
                     "timed_in": f"a separate region of {prof_steps} steps with per-kernel-class CUDA events; `value` is "
                                 "timed without them"},
        "e2e": {"value": e2e_value, "unit": "embeddings/s", "h2d_bytes_per_step": int(img_host_np.nbytes),
                "d2h_bytes_per_step": int(out_host.nbytes), "ms_per_step": e2e_ms,
                "api": "b200_model_encode_images_u8 (host uint8 in pinned memory -> host fp32)"},
        "gpu_launches": launches + e2e_launches * e2e_steps,
        "out_host": out_host,
    }
    return res


# ------------------------------------------------------------------------------------------------ top-k
def bench_topk(c):
    import torch
    from marqo_b200.distributed import ShardedRowStore, unpack_blocks
    from marqo_b200.engine import RowStore
    args, dev, world, rank = c.args, c.dev, c.world, c.rank
    rows_local = args.topk_rows // world + (1 if rank < args.topk_rows % world else 0)
    row_base = rank * (args.topk_rows // world) + min(rank, args.topk_rows % world)
    store = RowStore(TOPK_DIM, "prenormalized-angular", device=c.local_rank, capacity=rows_local)
    gc = torch.Generator(device=dev).manual_seed(1000 + rank)
    chunk = 250_000
    for lo in range(0, rows_local, chunk):
        m = min(chunk, rows_local - lo)
        x = torch.nn.functional.normalize(torch.randn(m, TOPK_DIM, device=dev, generator=gc), dim=1).contiguous()
        torch.cuda.synchronize()
        store.add_device(x.data_ptr(), m)
    del x
    sharded = ShardedRowStore(store, rank, world, device=dev, exchange=args.exchange, max_k=16)
    store.set_doc_offset(row_base)                 # shard-local document numbers -> global
    stream = sharded._stream
    gq = torch.Generator(device=dev).manual_seed(99)
    q = torch.nn.functional.normalize(torch.randn(TOPK_NQ, TOPK_DIM, device=dev, generator=gq), dim=1).contiguous()
    nk = TOPK_NQ * TOPK_K
    fin = torch.empty(nk * 16, dtype=torch.uint8, device=dev)
    torch.cuda.synchronize()

    def search_step():
        sharded.search_device(q.data_ptr(), TOPK_NQ, TOPK_K, fin.data_ptr(), sync=False)

    scan, merge = [], []
    for _ in range(3):
        search_step()
    c.barrier()
    s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s0.record(stream)
    for _ in range(args.steps):
        search_step()                 # back to back: no host synchronisation inside the timed region
    s1.record(stream)
    c.barrier()
    t_ms = c.max_over_ranks(s0.elapsed_time(s1)) / args.steps
    if args.dump_outputs:
        D, R, S = unpack_blocks(fin.cpu().numpy(), 1, TOPK_NQ, TOPK_K)
        c.outputs.update(topk_doc=D[0], topk_row=R[0], topk_score=S[0])
    for _ in range(max(5, min(args.steps, 20))):   # per-kernel times (roofline numerator): CUDA events around the scan
        search_step()
        a, b = store.last_timing()
        scan.append(a)
        merge.append(b)
    torch.cuda.synchronize()
    D, R, S = unpack_blocks(fin.cpu().numpy(), 1, TOPK_NQ, TOPK_K)
    md, msc = D[0], S[0]
    assert (md >= 0).all() and np.all(np.diff(msc, axis=1) <= 0) and md.max() < args.topk_rows
    stats = store.search_stats()
    scan_ms = statistics.median(scan)
    bytes_per_launch = rows_local * TOPK_DIM * 2
    ach = bytes_per_launch / (scan_ms / 1e3) / 1e9
    tsc = c.traffic.get("score_scan_kernel", {})
    topk = {
        "metric": "queries/s (exact top-10, batch 64, 10M x 768 fp16 corpus)", "value": TOPK_NQ / (t_ms / 1e3),
        "unit": "queries/s", "ms_per_batch": t_ms, "rows_total": args.topk_rows, "rows_per_gpu": rows_local,
        "scan_ms": scan_ms, "merge_ms": statistics.median(merge), "scaling": "strong",
        "exactness": {"guard_failures": stats["flagged"], "unresolved_async": stats["unresolved_async"],
                      "note": "every batch runs the exact-selection guard; 0 failures = the one-pass answer was proven exact"},
        "config": {"l2_flush": "not needed: every launch streams the whole shard (>= 1.9 GB), far larger than the 126 MB L2",
                   "exchange": {"peer": "ONE fused kernel: peer stores of the packed [64,10] block (10 KB) into every rank's "
                                        "symmetric buffer over NVLink + release flag + device merge (no NCCL call), inside the "
                                        "timed region",
                                "nccl": "one all-gather of the packed [64,10] result block (10 KB per rank) + device-side merge, "
                                        "inside the timed region",
                                "single": "single GPU: no exchange", "host": "host"}[sharded.mode],
                   "exchange_mode": sharded.mode},
        "roofline": {"bound": "hbm", "achieved": ach, "peak": c.peaks["hbm_gbs"], "unit": "GB/s",
                     "frac": ach / c.peaks["hbm_gbs"],
                     "traffic": (tsc.get("dram_bytes_per_launch") if rows_local == tsc.get("rows") else None),
                     "traffic_note": f"ncu dram bytes of one launch (profiles/{c.traffic.get('_file', 'n/a')}); null when "
                                     f"this run's shard size differs from the captured one",
                     "peak_source": c.peaks["source"],
                     "kernel": "score::scan_kernel", "bytes_per_launch": bytes_per_launch},
    }
    # e2e: host queries in -> MERGED global ids out through ShardedRowStore.search (H2D + scan + exchange + merge + D2H),
    # every rank takes part, max over ranks
    qh = q.cpu().numpy()
    sharded.search(qh, TOPK_K)
    e2e_n = max(5, min(args.steps, 20))
    c.barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_n):
        ed, er, es = sharded.search(qh, TOPK_K)
    dt = c.max_over_ranks(time.perf_counter() - t0)
    assert (ed == md).all()
    topk["e2e"] = {"value": TOPK_NQ / (dt / e2e_n), "unit": "queries/s",
                   "h2d_bytes_per_step": int(qh.nbytes), "d2h_bytes_per_step": TOPK_NQ * TOPK_K * 16,
                   "note": "ShardedRowStore.search: host fp32 queries in, merged global (doc, row, score) out on every rank; "
                           "includes the exchange; max over ranks"}
    # larger k through the same path (single pass up to k = 160)
    if not args.quick:
        k100 = 100
        store.search(qh[:16], k100)
        before = store.search_stats()
        t0 = time.perf_counter()
        for _ in range(3):
            store.search(qh[:16], k100)
        dt100 = (time.perf_counter() - t0) / 3
        after = store.search_stats()
        topk["k100"] = {"ms_per_batch_of_16": dt100 * 1e3, "collect_passes": after["collect_passes"] - before["collect_passes"],
                        "note": "limit = 100 on this rank's shard through b200_index_search: one scan when the guard holds"}
    sharded.close()
    store.close()
    return topk


# ------------------------------------------------------------------------------------------------ public-API block
def bench_api(c):
    """The calls a Marqo process makes, from 8 threads (api/configs.py:27-28): s2_inference.vectorise() ->
    List[List[float]], and GpuTensorIndex.query() -> QueryResult on a 500 k-document index."""
    import torch
    from marqo_b200 import s2_inference as S2, model_registry as R
    from marqo_b200.gpu_tensor_index import DeviceChunks, GpuTensorIndex
    out = {"threads": 8}
    os.environ["MARQO_MAX_VECTORISE_BATCH_SIZE"] = str(BATCH)
    props = dict(R.get_model_properties(MODEL_B32), random_init=1234, max_batch=BATCH)
    rng = np.random.default_rng(3)
    imgs = [torch.from_numpy(rng.integers(0, 256, size=(IMG, IMG, 3), dtype=np.uint8)) for _ in range(BATCH)]
    dev_s = f"cuda:{c.local_rank}"
    v = S2.vectorise(MODEL_B32, imgs, model_properties=props, device=dev_s, normalize_embeddings=True,
                     modality=S2.Modality.IMAGE)
    assert len(v) == BATCH and len(v[0]) == 512
    t0 = time.perf_counter()
    for _ in range(3):
        S2.vectorise(MODEL_B32, imgs, model_properties=props, device=dev_s, normalize_embeddings=True,
                     modality=S2.Modality.IMAGE)
    one = (time.perf_counter() - t0) / 3

    def work():
        for _ in range(2):
            S2.vectorise(MODEL_B32, imgs, model_properties=props, device=dev_s, normalize_embeddings=True,
                         modality=S2.Modality.IMAGE)

    ths = [threading.Thread(target=work) for _ in range(8)]
    t0 = time.perf_counter()
    [t.start() for t in ths]
    [t.join() for t in ths]
    dt = time.perf_counter() - t0
    out["vectorise"] = {"model": MODEL_B32, "batch": BATCH, "single_thread_emb_per_s": BATCH / one,
                        "eight_threads_emb_per_s": 16 * BATCH / dt,
                        "note": "s2_inference.vectorise(list of 256 uint8 HWC tensors) -> List[List[float]]; includes batch "
                                "assembly, H2D, encode, D2H and .tolist()"}
    S2.clear_loaded_models()
    torch.cuda.empty_cache()

    # ---- GpuTensorIndex.query() from 8 threads
    n_docs, dim = 500_000, 768
    ix = GpuTensorIndex(device=c.local_rank)
    g = torch.Generator(device=c.dev).manual_seed(7)
    t0 = time.perf_counter()
    step = 50_000
    for lo in range(0, n_docs, step):
        x = torch.nn.functional.normalize(torch.randn(step, dim, device=c.dev, generator=g), dim=1).contiguous()
        torch.cuda.synchronize()
        batch = [{"id": str(lo + i), "fields": {"marqo__id": str(lo + i),
                                                "marqo__embeddings_body": DeviceChunks(["0"], x.data_ptr() + i * dim * 4, dim, x)}}
                 for i in range(step)]
        r = ix.feed_batch(batch, "bench")
        assert not r.errors
    feed_s = time.perf_counter() - t0
    out["feed_batch_device"] = {"docs": n_docs, "docs_per_s": n_docs / feed_s,
                                "note": "feed_batch with DeviceChunks (embeddings already in HBM): host bookkeeping + ONE "
                                        "device append per 50 k-document batch"}
    qs = torch.nn.functional.normalize(torch.randn(512, dim, generator=torch.Generator().manual_seed(8)), dim=1).numpy()
    yql = ("select * from bench where ({targetHits:10, approximate:False}nearestNeighbor(marqo__embeddings_body, "
           "marqo__query_embedding))")

    def ask(i):
        return ix.query(yql, hits=10, ranking="embedding_similarity", model_restrict="bench",
                        query_features={"marqo__query_embedding": qs[i].tolist()})

    ask(0)
    t0 = time.perf_counter()
    for i in range(64):
        ask(i)
    single = 64 / (time.perf_counter() - t0)

    def qwork(t):
        for i in range(t * 64, t * 64 + 64):
            ask(i)

    before = ix.coalescer_stats()
    ths = [threading.Thread(target=qwork, args=(t,)) for t in range(8)]
    t0 = time.perf_counter()
    [t.start() for t in ths]
    [t.join() for t in ths]
    dt = time.perf_counter() - t0
    after = ix.coalescer_stats()
    out["query"] = {"docs": n_docs, "dim": dim, "single_thread_qps": single, "eight_threads_qps": 512 / dt,
                    "scans_for_512_queries": after["batches"] - before["batches"],
                    "note": "GpuTensorIndex.query(yql, query_features) -> QueryResult with hits, match-features and coverage; "
                            "concurrent requests are coalesced into shared scans"}
    ix.close()
    torch.cuda.empty_cache()
    return out


# ------------------------------------------------------------------------------------------------ cfg2 / cfg3 / cfg4
def bench_cfg2(c, steps: int, warmup: int):
    """open_clip/ViT-B-32 image + text vectorise, batch 256 (BASELINE.json configs[1]); step = 256 images + 256 texts."""
    import torch
    from marqo_b200 import model_registry as R, weights as Wt
    from marqo_b200.engine import Encoder
    arch = R.get_model_properties(MODEL_B32)["arch"]
    enc = Encoder("clip", arch, Wt.random_clip_weights(arch, 1234), device=c.local_rank, max_batch=BATCH)
    enc.set_stream(c.stream.cuda_stream)
    g = torch.Generator(device=c.dev).manual_seed(c.rank)
    img = torch.randint(0, 256, (BATCH, IMG, IMG, 3), dtype=torch.uint8, device=c.dev, generator=g)
    ids = torch.randint(1, 49405, (BATCH, 77), dtype=torch.int32, device=c.dev, generator=g)
    ids[:, 0] = 49406
    ids[:, 76] = 49407
    oi = torch.empty(BATCH, 512, dtype=torch.float32, device=c.dev)
    ot = torch.empty(BATCH, 512, dtype=torch.float32, device=c.dev)

    def step():
        enc.encode_images_u8_device(img.data_ptr(), BATCH, IMG, IMG, oi.data_ptr(), normalize=True, sync=False)
        enc.encode_tokens_device(ids.data_ptr(), None, BATCH, 77, ot.data_ptr(), normalize=True, sync=False)

    ms = timed_steps(c, step, steps, warmup)
    fl = vit_flops(arch["vision"], BATCH)[0] + text_flops(arch["text"], BATCH, 77)
    ih, th = img.cpu().numpy(), ids.cpu().numpy()
    enc.encode_images_u8(ih)
    t0 = time.perf_counter()
    for _ in range(5):
        enc.encode_images_u8(ih)
        enc.encode_tokens(th)
    e2e = c.max_over_ranks(time.perf_counter() - t0) / 5
    assert bool(torch.isfinite(oi).all() and torch.isfinite(ot).all())
    enc.close()
    torch.cuda.empty_cache()
    return {"metric": "embeddings/s (open_clip/ViT-B-32 image + text vectorise, batch 256 + 256)",
            "value": 2 * BATCH * c.world / (ms / 1e3), "unit": "embeddings/s", "ms_per_step": ms,
            "tflops": fl / (ms / 1e3) / 1e12, "frac_of_sustained_peak": fl / (ms / 1e3) / 1e12 / c.peaks["bf16_tflops_sustained"],
            "e2e": {"value": 2 * BATCH * c.world / e2e, "unit": "embeddings/s", "h2d_bytes_per_step": int(ih.nbytes + th.nbytes),
                    "d2h_bytes_per_step": 2 * BATCH * 512 * 4}}


def bench_cfg3(c, docs_total: int, through_api: bool = True):
    """open_clip/ViT-L-14 add_documents: image + caption per document, doc-sharded across the ranks, embeddings appended
    to this rank's GPU index shard — both towers and the index append inside the timed region (configs[2])."""
    import torch
    from marqo_b200 import model_registry as R
    from marqo_b200.add_documents import add_documents_device
    from marqo_b200.gpu_tensor_index import GpuTensorIndex
    from marqo_b200.loaders import B200OpenCLIP
    lo = c.rank * (docs_total // c.world) + min(c.rank, docs_total % c.world)
    n_local = docs_total // c.world + (1 if c.rank < docs_total % c.world else 0)
    props = dict(R.get_model_properties(MODEL), random_init=1234, max_batch=BATCH)
    model = B200OpenCLIP(device=f"cuda:{c.local_rank}", model_properties=props)
    model.load()
    arch = props["arch"]
    ix = GpuTensorIndex(device=c.local_rank)
    g = torch.Generator(device=c.dev).manual_seed(17 + c.rank)
    n_img_variants = 4 * BATCH           # synthetic pixels are recycled (HBM-resident pool); every document is encoded
    pool = torch.randint(0, 256, (n_img_variants, IMG, IMG, 3), dtype=torch.uint8, device=c.dev, generator=g)
    cap_ids = torch.randint(1, 49405, (n_img_variants, 77), dtype=torch.int32, generator=torch.Generator().manual_seed(5))
    cap_ids[:, 0] = 49406
    cap_ids[:, 40:] = 0
    cap_ids[:, 40] = 49407
    cap_np = cap_ids.numpy()

    def run(n_docs: int, id_base: int):
        done = 0
        while done < n_docs:
            m = min(BATCH, n_docs - done)
            sel = (done % n_img_variants)
            imgs = pool[sel:sel + m] if sel + m <= n_img_variants else pool[:m]
            caps = cap_np[sel:sel + m] if sel + m <= n_img_variants else cap_np[:m]
            docs = [{"_id": f"doc{id_base + done + i}", "n": id_base + done + i} for i in range(m)]
            r = add_documents_device(ix, "cfg3", docs, {"image": (model, "image"), "caption": (model, "text")},
                                     device_contents={"image": imgs, "caption": caps})
            assert not r.errors
            done += m

    run(2 * BATCH, 10_000_000)           # warm-up (separate ids)
    c.barrier()
    t0 = time.perf_counter()
    run(n_local, lo)
    torch.cuda.synchronize()
    dt = c.max_over_ranks(time.perf_counter() - t0)
    assert ix.get_document_count("cfg3") == n_local + 2 * BATCH
    st = ix._schemas["cfg3"].stores
    assert len(st["marqo__embeddings_image"]) == n_local + 2 * BATCH == len(st["marqo__embeddings_caption"])
    fl = (vit_flops(arch["vision"], 1)[0] + text_flops(arch["text"], 1, 77)) * docs_total
    # a self-match through the index that was just built
    res = ix.query("select * from cfg3 where ({targetHits:3, approximate:False}nearestNeighbor(marqo__embeddings_image, "
                   "marqo__query_embedding))", hits=3, ranking="embedding_similarity", model_restrict="cfg3",
                   query_features={"marqo__query_embedding": st["marqo__embeddings_image"].get_rows([2 * BATCH + 5])[0].tolist()})
    assert abs(res.hits[0].relevance - 1.0) < 2e-3
    ix.close()
    model.close()
    torch.cuda.empty_cache()
    return {"metric": "documents/s (open_clip/ViT-L-14 add_documents: image + caption towers + index append)",
            "value": docs_total / dt, "unit": "documents/s", "docs_total": docs_total, "docs_per_gpu": n_local,
            "seconds": dt, "tflops": fl / dt / 1e12, "scaling": "strong (fixed document count, doc-sharded)",
            "api": "add_documents_device -> B200OpenCLIP.encode_to_device x2 -> GpuTensorIndex.feed_batch(DeviceChunks) -> "
                   "b200_index_add_device_docs",
            "note": "wall clock around the public fast-path API, max over ranks; pixels come from an HBM-resident pool "
                    "(what Marqo's download threads leave on the device, add_docs.py:129-134), captions as token ids"}


def bench_cfg4(c, chunks_total: int, seq: int = 512, batch: int = 64, pad_fraction: float = 0.0):
    """hf/e5-large-v2 text indexing: 512-token chunks generated from on-device ids (no 2 GB host traffic), sharded across
    the ranks, embeddings appended to the rank's row store (configs[3])."""
    import torch
    from marqo_b200 import model_registry as R, weights as Wt
    from marqo_b200.engine import Encoder, RowStore
    arch = R.get_model_properties(MODEL_E5L)["arch"]
    enc = Encoder("bert", arch, Wt.random_bert_weights(arch, 1234), device=c.local_rank, max_batch=batch)
    enc.set_stream(c.stream.cuda_stream)
    n_local = chunks_total // c.world + (1 if c.rank < chunks_total % c.world else 0)
    store = RowStore(arch["width"], device=c.local_rank, capacity=n_local + 4 * batch)
    store.set_stream(c.stream.cuda_stream)
    g = torch.Generator(device=c.dev).manual_seed(31 + c.rank)
    out = torch.empty(batch, arch["width"], dtype=torch.float32, device=c.dev)
    mask = None
    if pad_fraction > 0:
        lens = torch.randint(int(seq * (1 - 2 * pad_fraction)) + 1, seq + 1, (batch,), generator=torch.Generator().manual_seed(1))
        mask = (torch.arange(seq)[None, :] < lens[:, None]).to(torch.int32).to(c.dev)

    def one(m):
        ids = torch.randint(1000, 30000, (m, seq), dtype=torch.int32, device=c.dev, generator=g)   # counter-based RNG on the device
        ids[:, 0] = 101
        ids[:, seq - 1] = 102
        enc.encode_tokens_device(ids.data_ptr(), None if mask is None else mask.data_ptr(), m, seq, out.data_ptr(),
                                 normalize=True, sync=False)
        c.stream.synchronize()
        store.add_device(out.data_ptr(), m)

    for _ in range(3):
        one(batch)
    c.barrier()
    base_rows = len(store)
    t0 = time.perf_counter()
    done = 0
    while done < n_local:
        m = min(batch, n_local - done)
        one(m)
        done += m
    torch.cuda.synchronize()
    dt = c.max_over_ranks(time.perf_counter() - t0)
    assert len(store) == base_rows + n_local
    fl = text_flops(arch, 1, seq) * chunks_total
    enc.close()
    store.close()
    torch.cuda.empty_cache()
    return {"metric": "chunks/s (hf/e5-large-v2 indexing, 512-token chunks, incl. row-store append)",
            "value": chunks_total / dt, "unit": "chunks/s", "chunks_total": chunks_total, "chunks_per_gpu": n_local,
            "seconds": dt, "tflops": fl / dt / 1e12, "frac_of_sustained_peak": fl / dt / 1e12 / c.world / c.peaks["bf16_tflops_sustained"],
            "pad_fraction": pad_fraction, "batch": batch, "seq": seq}


def cpu_baseline_block(c, out_host, topk):
    """Rank 0, bounded sample: the oracle port on the host cores this process may use — the SAME 16 images the reference
    arm times (its own sub-batch size), and a 1 M-row slice for the score step."""
    import torch
    threads = host_threads()
    torch.set_num_threads(threads)
    sample = REF_SUB_BATCH
    sd_o, cfg_o = make_oracle_model()
    pix = reference_sample_images(sample)
    oracle_embed_step(sd_o, cfg_o, pix[:2])
    t0 = time.perf_counter()
    ref = oracle_embed_step(sd_o, cfg_o, pix)
    dt = time.perf_counter() - t0
    cos = torch.nn.functional.cosine_similarity(ref.double(), torch.from_numpy(out_host[:sample]).double())
    cpu = {"value": sample / dt, "unit": "embeddings/s", "cores": threads, "kind": "port",
           "sample": f"the first {sample} of the step's 256 images (one reference sub-batch), one pass, torch CPU fp32 oracle",
           "min_cosine_vs_gpu": float(cos.min())}
    if topk is not None:
        n_s = 1_000_000
        gcpu = torch.Generator().manual_seed(5)
        C = torch.nn.functional.normalize(torch.randn(n_s, TOPK_DIM, generator=gcpu), dim=1)
        qc = torch.nn.functional.normalize(torch.randn(TOPK_NQ, TOPK_DIM, generator=gcpu), dim=1)
        (qc[:4] @ C[:1000].t()).topk(TOPK_K, dim=1)
        t0 = time.perf_counter()
        (qc @ C.t()).topk(TOPK_K, dim=1)
        dt = time.perf_counter() - t0
        topk["cpu_baseline"] = {"value": TOPK_NQ / (dt * (c.args.topk_rows / n_s)), "unit": "queries/s",
                                "cores": threads, "kind": "port",
                                "sample": "fp32 q @ C^T + topk on a 1M-row slice, scaled x10 to the 10M corpus"}
    return cpu


# ------------------------------------------------------------------------------------------------ our arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="headline", choices=["headline", "cfg2", "cfg3", "cfg4"])
    ap.add_argument("--skip-topk", action="store_true")
    ap.add_argument("--skip-api", action="store_true")
    ap.add_argument("--skip-cfg", action="store_true")
    ap.add_argument("--skip-cpu-baseline", action="store_true")
    ap.add_argument("--quick", action="store_true", help="headline + topk only")
    ap.add_argument("--topk-rows", type=int, default=TOPK_ROWS_TOTAL)
    ap.add_argument("--exchange", default="auto", choices=["auto", "peer", "nccl"])
    ap.add_argument("--docs", type=int, default=100_000)
    ap.add_argument("--chunks", type=int, default=1_000_000)
    ap.add_argument("--pad-fraction", type=float, default=0.0)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's outputs as DIR/<name>.npy (headline configuration only)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.config != "headline"):
        ap.error("--dump-outputs covers the headline configuration of --impl b200 only")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.quick:
        args.skip_api = args.skip_cfg = True
    claim_stdout()

    if args.impl == "reference":
        run_reference(args, int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")))
        return

    import torch.distributed as dist
    c = make_ctx(args)

    if args.config != "headline":
        if args.config == "cfg2":
            blk = bench_cfg2(c, args.steps, args.warmup)
        elif args.config == "cfg3":
            blk = bench_cfg3(c, args.docs)
        else:
            blk = bench_cfg4(c, args.chunks, pad_fraction=args.pad_fraction)
        if c.rank == 0:
            line = dict(blk, n_gpus=c.world, higher_is_better=True, dtype="bf16", data="synthetic", vs_baseline=None,
                        config={"workload": blk["metric"], "baseline_config": args.config})
            emit(line)
        if c.distributed:
            dist.barrier()
            dist.destroy_process_group()
        return

    head = bench_headline(c)
    topk = None if args.skip_topk else bench_topk(c)
    cfg2 = cfg3 = api = None
    if not args.skip_cfg:
        cfg2 = bench_cfg2(c, max(5, min(args.steps, 20)), 3)
        cfg3 = bench_cfg3(c, 8192 * c.world)   # 32 batches per GPU: the row store's x1.5 growth steps are amortised
    if not args.skip_api and c.rank == 0:
        api = bench_api(c)
    cpu = None
    if c.rank == 0 and not args.skip_cpu_baseline:
        cpu = cpu_baseline_block(c, head["out_host"], topk)

    if c.rank == 0:
        line = {
            "metric": METRIC, "value": head["value"], "unit": "embeddings/s", "n_gpus": c.world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": head["step_ms"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": headline_config(c.world),
            "tflops": head["tflops"], "roofline": head["roofline"], "e2e": head["e2e"],
            "gpu_launches": head["gpu_launches"], "clocks": head["clocks"], "cpu_baseline": cpu, "topk": topk,
            "api_e2e": api, "cfg2": cfg2, "cfg3": cfg3,
        }
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, c.outputs)
        emit(line)
    if c.distributed:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
