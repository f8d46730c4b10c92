"""Time the tagged catalogue pass (HSemanticIdTokenizer.precompute_corpus_ids with concatenated ids) at the gin shape.

    python tools/bench_tag_heads.py [--items 1048576] [--reps 5] [--out result.json]

Variants, alternated in the same process: tag_precision="fused"; "torch" with fp32 matmuls (the tokenizer's setting
outside the trainer); "torch" with TF32 matmuls (the trainer's setting); and the untagged pass for scale.  Then a
torch.profiler run of the fused variant gives per-kernel times of the tag kernels, and the tag heads' TFLOP/s against
the algorithmic count (2 x MACs of every Linear of every level, gate included: 9.57 Mflop per item at the gin shape).
The catalogue (3 GB fp32) is larger than the L2, so every pass reads it from HBM.
"""
import argparse
import json
import os
import re
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "hid-vae_b200"), ROOT]

import torch  # noqa: E402

D, HIDDEN, COUNTS = 32, [512, 256, 128], [38, 168, 348]


def flops_per_item(d=D, first_hidden=HIDDEN[0], counts=COUNTS):
    total = 0
    for i, c in enumerate(counts):
        e, h = d * (i + 1), first_hidden // 2 * (i + 1)
        inner = int(h * 0.9)
        macs = e * (e // 4) + (e // 4) * (e // 2) + (e // 2) * e + e * h + 2 * (h * inner + inner * h) + h * inner
        macs += inner * (inner // 2) + (inner // 2) * c
        total += 2 * macs
    return total


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--items", type=int, default=1 << 20)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_tag_heads.py measures on a CUDA device; none found")
    from modules.tokenizer.h_semids import HSemanticIdTokenizer

    def tok(tagged, precision):
        torch.manual_seed(0)
        return HSemanticIdTokenizer(input_dim=768, output_dim=D, hidden_dims=HIDDEN, codebook_size=256, n_layers=3,
                                    tag_class_counts=COUNTS if tagged else None, use_concatenated_ids=tagged,
                                    tag_precision=precision).cuda()

    variants = {"fused": (tok(True, "fused"), False), "torch_fp32": (tok(True, "torch"), False),
                "torch_tf32": (tok(True, "torch"), True), "untagged": (tok(False, "torch"), False)}
    g = torch.Generator(device="cuda").manual_seed(1)
    items = torch.randn((args.items, 768), generator=g, device="cuda")

    def run(name):
        t, tf32 = variants[name]
        torch.backends.cuda.matmul.allow_tf32 = tf32
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = t.precompute_corpus_ids(items)
        torch.cuda.synchronize()
        torch.backends.cuda.matmul.allow_tf32 = False
        return time.perf_counter() - t0, out

    for name in variants:          # warm-up: module loads, cuBLAS heuristics, image packing
        run(name)
    times = {name: [] for name in variants}
    for _ in range(args.reps):
        for name in variants:
            times[name].append(run(name)[0])
    _, fused_ids = run("fused")
    _, torch_ids = run("torch_fp32")
    agree = [(fused_ids[:, 3 + i] == torch_ids[:, 3 + i]).float().mean().item() for i in range(3)]

    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        run("fused")
    kern = {}
    for e in prof.key_averages():
        m = re.search(r"\b(tag_[a-z_]+_kernel(?:<(?:\(int\))?\d+>)?|enc_mlp_kernel<[^>]*>|rq_fwd\w*)", e.key)
        if m and e.device_time_total > 0:
            k = kern.setdefault(m.group(1).replace("(int)", ""), {"calls": 0, "total_ms": 0.0})
            k["calls"] += e.count
            k["total_ms"] += e.device_time_total / 1e3
    tag_ms = sum(v["total_ms"] for k, v in kern.items() if k.startswith("tag_") and "pack" not in k)
    fl = flops_per_item() * args.items
    med = {k: sorted(v)[len(v) // 2] * 1e3 for k, v in times.items()}
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    res = {
        "gpu": gpu, "items": args.items, "reps": args.reps, "median_ms": med, "all_ms": {k: [x * 1e3 for x in v] for k, v in times.items()},
        "tag_ms": {k: med[k] - med["untagged"] for k in ("fused", "torch_fp32", "torch_tf32")},
        "speedup_vs_tf32": med["torch_tf32"] / med["fused"], "speedup_vs_fp32": med["torch_fp32"] / med["fused"],
        "tag_kernels_ms": tag_ms, "tag_kernels_tflops": fl / (tag_ms * 1e-3) / 1e12 if tag_ms else None,
        "tag_kernels_share_of_dense_fp16_2250": (fl / (tag_ms * 1e-3) / 1e12) / 2250 if tag_ms else None,
        "mflop_per_item": flops_per_item() / 1e6, "kernels": kern, "agreement_fused_vs_fp32": agree,
    }
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
