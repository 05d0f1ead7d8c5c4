"""Probe: hf/all-mpnet-base-v2 against hf/e5-base-v2 (the same GEMM shapes; MPNet adds the relative-position bias to
the attention softmax) in one process, alternating between the two models.

For each shape it reports the median device time per encode call (CUDA events around the call, device-resident ids,
sync after every call) and the per-class device time of one call from b200_model_set_profiling (GEMM vs attention), so
the cost of the bias is visible as attention ms with and without it.  Shapes: b256 x 128 tokens full length and
ragged (lengths uniform in 1..128), and b8 x 128 (a small-batch query shape, CUDA-graph replayed).  Prints one JSON
line per (model, shape) and a summary line with the throughput ratio; the card's name and power limit go with them.

    python tools/mpnet_probe.py [--iters 20] [--out profiles/mpnet_probe.jsonl]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from marqo_b200 import model_registry as R, weights as Wt  # noqa: E402
from marqo_b200.engine import Encoder  # noqa: E402

MODELS = {"hf/all-mpnet-base-v2": ("mpnet", Wt.random_mpnet_weights), "hf/e5-base-v2": ("bert", Wt.random_bert_weights)}


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [s.strip() for s in q.split(",")]
        return {"gpu": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:   # the numbers are still printed, without the card's settings
        return {"gpu": torch.cuda.get_device_name(0), "power_limit": f"unknown ({e})"}


def inputs(B, S, ragged, vocab, seed):
    g = torch.Generator().manual_seed(seed)
    ids = torch.randint(1000, min(vocab, 30000), (B, S), generator=g, dtype=torch.int32)
    lens = torch.randint(1, S + 1, (B,), generator=g) if ragged else torch.full((B,), S)
    mask = (torch.arange(S)[None, :] < lens[:, None]).to(torch.int32)
    return ids.cuda(), mask.cuda(), int(lens.sum())


def time_calls(enc, ids, mask, out, iters):
    B, S = ids.shape
    run = lambda: enc.encode_tokens_device(ids.data_ptr(), mask.data_ptr(), B, S, out.data_ptr(), sync=True)
    for _ in range(3):
        run()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ms = []
    for _ in range(iters):
        torch.cuda.synchronize()
        e0.record()
        run()
        e1.record()
        e1.synchronize()
        ms.append(e0.elapsed_time(e1))
    enc.set_profiling(True)
    run()
    prof = enc.profile()
    enc.set_profiling(False)
    return float(np.median(ms)), float(np.min(ms)), prof


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3, help="alternations between the two models per shape")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    torch.cuda.set_device(0)
    info = card()
    encs = {}
    for name, (kind, rnd) in MODELS.items():
        arch = R.get_model_properties(name)["arch"]
        encs[name] = Encoder(kind, arch, rnd(arch, 1234), max_batch=256)
    shapes = [("b256x128 full", 256, 128, False), ("b256x128 ragged", 256, 128, True), ("b8x128", 8, 128, False)]
    lines = []
    for label, B, S, ragged in shapes:
        ids, mask, tokens = inputs(B, S, ragged, 30522, seed=B + S + int(ragged))
        out = torch.empty(B, 768, device="cuda")
        runs = {n: [] for n in encs}
        for _ in range(a.rounds):
            for name, enc in encs.items():
                runs[name].append(time_calls(enc, ids, mask, out, a.iters))
        for name in encs:
            med = float(np.median([r[0] for r in runs[name]]))
            prof = runs[name][-1][2]
            rec = {"model": name, "shape": label, "B": B, "S": S, "valid_tokens": tokens, "ms_median": round(med, 4),
                   "ms_min": round(min(r[1] for r in runs[name]), 4), "items_per_s": round(B / med * 1e3, 1),
                   "gemm_ms": round(prof["gemm_ms"], 4), "attention_ms": round(prof["attention_ms"], 4),
                   "attention_launches": prof["attention_launches"], **info}
            lines.append(rec)
            print(json.dumps(rec), flush=True)
        m, e = (next(r for r in lines if r.get("model") == n and r["shape"] == label) for n in MODELS)
        summ = {"shape": label, "mpnet_over_e5_throughput": round(m["items_per_s"] / e["items_per_s"], 4),
                "attention_ms_with_bias": m["attention_ms"], "attention_ms_without_bias": e["attention_ms"],
                "attention_ms_delta": round(m["attention_ms"] - e["attention_ms"], 4), **info}
        lines.append(summ)
        print(json.dumps(summ), flush=True)
    for enc in encs.values():
        enc.close()
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "w") as f:
            for r in lines:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
