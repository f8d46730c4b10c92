#!/usr/bin/env python
"""Time the HiD-VAE training step in Gumbel-softmax mode, eager against CUDA graphs (GraphedTrainStep), on one GPU.

    python tools/bench_gumbel_graph.py [--steps 60] [--warmup 10] [--reps 200]

Three parts, one JSON line each, then a line with the card's name and power limit:
  step        HRqVae at the gin shapes (768-512-256-128-32, K = 256, L = 3, tag heads and uniqueness loss on), one optimisation
              step of batch 128 x 2 micro-steps and of batch 8,192 x 1, Gumbel-softmax and rotation trick (the reference for
              the comparison), eager (AdamW fused) and as graphs (AdamW fused + capturable).  Median / min ms per step over
              --steps steps after --warmup, each step bracketed by CUDA events.
  entries     one Gumbel level (D = 32, K = 256), forward + backward through autograd, host seed (hv_gumbel_forward /
              _backward) against device seed (the _devrng entries), at 8,192 and 65,536 rows; the two kinds alternate call
              by call in one process.  Median ms over --reps calls of each kind.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "hid-vae_b200"), ROOT]
import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

from data.schemas import TaggedSeqBatch  # noqa: E402
from hidvae_b200 import dist as hv_dist  # noqa: E402
from hidvae_b200 import ops  # noqa: E402
from hidvae_b200.graph_step import GraphedTrainStep  # noqa: E402
from modules.h_rqvae import HRqVae  # noqa: E402
from modules.quantize import QuantizeForwardMode  # noqa: E402

TAG_COUNTS = [37, 168, 353]
N_ITEMS = 32768


def card():
    q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader"], capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(), "nvidia_smi": q.stdout.strip() or q.stderr.strip()}


def timed(fn, steps):
    """Per-call ms of `steps` calls, each bracketed by CUDA events on the current stream."""
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for a, b in ev:
        a.record()
        fn()
        b.record()
    torch.cuda.synchronize()
    return [a.elapsed_time(b) for a, b in ev]


def step_times(mode, batch, micro, graphed, steps, warmup, data):
    dev = torch.device("cuda", 0)
    x, tags_emb, tags_idx = data
    torch.manual_seed(0)
    model = HRqVae(input_dim=768, embed_dim=32, hidden_dims=[512, 256, 128], codebook_size=256, codebook_kmeans_init=False,
                   codebook_normalize=True, codebook_mode=mode, n_layers=3, n_cat_features=0, commitment_weight=0.25,
                   tag_class_counts=TAG_COUNTS, tag_embed_dim=768, sem_id_uniqueness_weight=0.5,
                   sem_id_uniqueness_margin=0.5).to(dev).train()
    grads = hv_dist.FlatGradAllReduce(model.parameters())
    lr = torch.tensor(1e-4, device=dev) if graphed else 1e-4
    opt = torch.optim.AdamW(model.parameters(), lr=lr, fused=True, capturable=graphed)
    gen = torch.Generator(device=dev).manual_seed(7)
    fetch = lambda idx: TaggedSeqBatch(None, None, None, x[idx], None, None, tags_emb[idx], tags_idx[idx])
    if graphed:
        g = GraphedTrainStep(model, opt, grads, fetch, batch, N_ITEMS, gumbel_t=0.2, loss_divisor=micro, generator=gen)

        def step():
            grads.zero()
            for _ in range(micro):
                g.micro_step()
            grads.all_reduce()
            g.optimizer_step()
    else:
        def step():
            grads.zero()
            for _ in range(micro):
                out = model(fetch(torch.randint(0, N_ITEMS, (batch,), device=dev, generator=gen)), gumbel_t=0.2)
                grads.backward(out.loss / micro)
            grads.all_reduce()
            opt.step()
    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    ms = timed(step, steps)
    return {"median_ms": statistics.median(ms), "min_ms": min(ms)}


def entry_times(n, reps):
    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev).manual_seed(n)
    x = F.normalize(torch.randn(n, 32, generator=g, device=dev), dim=-1).requires_grad_(True)
    cb = F.normalize(torch.rand(256, 32, generator=g, device=dev), dim=-1).requires_grad_(True)
    g_emb = torch.randn(n, 32, generator=g, device=dev) * 0.1
    pair = torch.tensor([12345, 0], dtype=torch.int64, device=dev)

    def call(seed):
        emb, _ids, loss = ops.gumbel_apply(x, cb, 0.2, 0.25, seed=seed)
        torch.autograd.grad((emb * g_emb).sum() + loss.sum(), (x, cb))

    kinds = {"host_seed": 12345, "device_seed": pair}
    for seed in kinds.values():
        for _ in range(10):
            call(seed)
    ms = {name: [] for name in kinds}
    for _ in range(reps):
        for name, seed in kinds.items():
            ms[name] += timed(lambda: call(seed), 1)
    return {name: statistics.median(v) for name, v in ms.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=60)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--reps", type=int, default=200)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "tools/bench_gumbel_graph.py times the GPU: no CUDA device"
    torch.cuda.set_device(0)
    torch.set_float32_matmul_precision("high")                 # as train() does
    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev).manual_seed(3)
    data = (F.normalize(torch.randn(N_ITEMS, 768, generator=g, device=dev), dim=-1),
            torch.randn(N_ITEMS, 3, 768, generator=g, device=dev),
            torch.stack([torch.randint(0, c, (N_ITEMS,), generator=g, device=dev) for c in TAG_COUNTS], dim=1))
    for batch, micro in ((128, 2), (8192, 1)):
        for mode in (QuantizeForwardMode.GUMBEL_SOFTMAX, QuantizeForwardMode.ROTATION_TRICK):
            row = {"part": "step", "mode": mode.name, "batch": batch, "micro_steps": micro}
            for graphed in (False, True):
                row["graphs" if graphed else "eager"] = step_times(mode, batch, micro, graphed, args.steps, args.warmup, data)
            row["eager_over_graphs"] = row["eager"]["median_ms"] / row["graphs"]["median_ms"]
            print(json.dumps(row), flush=True)
    for n in (8192, 65536):
        row = {"part": "entries", "rows": n, "d": 32, "k": 256, **entry_times(n, args.reps)}
        row["device_over_host"] = row["device_seed"] / row["host_seed"]
        print(json.dumps(row), flush=True)
    print(json.dumps({"part": "card", **card()}), flush=True)


if __name__ == "__main__":
    main()
