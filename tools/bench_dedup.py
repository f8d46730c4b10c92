#!/usr/bin/env python
"""Time the semantic-ID collision digit (hv_semid_dedup through ops.semid_dedup) on one GPU.

    python tools/bench_dedup.py [--reps 10] [--warmup 3] [--skip-100mi]

Tables:
  bench_4mi   the [4 Mi, 3] id table the bench's tokenizer assigns to one GPU's shard (bench.make_tokenizer + synth_items)
  synth_32mi  32 Mi rows of uniform ids, 3 x 256 codes (24-bit keys)
  synth_100mi 100 Mi rows of the same (the catalogue size of BASELINE.json)
  c4_4mi      4 Mi rows of uniform ids, 4 x 4096 codes (48-bit keys)
Every timed call is preceded by a write of 512 MB, so that neither ids nor scratch are served from the 126 MB L2; the events
bracket the call alone.  Reported per table: median / min ms, algorithmic bytes (8 L read + 8 written per row) over time
against 7.7 TB/s of HBM, the torch formulation on the same GPU (1-D unique(return_inverse) of the same exact keys + stable
argsort), the kernel time by phase from torch.profiler (a separate, untimed call), and for bench_4mi the share of the bench
step (DESIGN.md section 5: 5.65-5.9 ms, measured earlier on other boards).  One JSON line per table, then a summary line
with the card's name and power limit.
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

import bench  # noqa: E402
from hidvae_b200 import ops  # noqa: E402

HBM_BYTES_PER_S = 7.7e12
BENCH_STEP_MS = (5.65, 5.9)


def card():
    q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader"], capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(), "nvidia_smi": q.stdout.strip() or q.stderr.strip()}


def torch_digits(ids, bits):
    keys = ops.dedup_key(ids, bits)
    uniq, inv = torch.unique(keys, return_inverse=True)
    order = torch.argsort(inv, stable=True)
    counts = torch.bincount(inv, minlength=uniq.numel())
    pos = torch.empty_like(order)
    pos[order] = torch.arange(order.numel(), device=ids.device)
    return pos - (counts.cumsum(0) - counts)[inv]


def timed(fn, reps, warmup, flush):
    for _ in range(warmup):
        fn()
    times = []
    for _ in range(reps):
        flush.add_(1)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b))
    return statistics.median(times), min(times)


def phases(ids, bits):
    """Kernel time (ms) of one call by phase, from torch.profiler."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        ops.semid_dedup(ids, bits)
        torch.cuda.synchronize()
    out = {}
    for ev in prof.events():
        if ev.device_type != torch.autograd.DeviceType.CUDA:
            continue
        name = ev.name
        key = next((k for k in ("dedup_keys", "dedup_flags", "dedup_runs", "dedup_finish") if k in name), None)
        if key is None:
            key = "cub_radix_sort" if "RadixSort" in name else "cub_scan" if "Scan" in name else "other"
        out[key] = out.get(key, 0.0) + ev.time_range.elapsed_us() / 1e3
    return {k: round(v, 4) for k, v in sorted(out.items())}


def measure(name, ids, bits, args, flush):
    rows, width = ids.shape
    res = ops.semid_dedup(ids, bits)
    ref = torch_digits(ids, bits)
    same = bool(torch.equal(res.digits, ref))
    del ref
    ms, ms_min = timed(lambda: ops.semid_dedup(ids, bits), args.reps, args.warmup, flush)
    t_ms, t_min = timed(lambda: torch_digits(ids, bits), max(3, args.reps // 2), 1, flush)
    alg = rows * (8 * width + 8)
    line = dict(table=name, rows=rows, width=width, key_bits=width * bits, distinct=int(res.stats[0]), max_digit=int(res.stats[1]),
                ms=round(ms, 4), ms_min=round(ms_min, 4), rows_per_s=round(rows / ms * 1e3), alg_bytes=alg,
                alg_tb_per_s=round(alg / ms / 1e9, 3), of_hbm=round(alg / ms / 1e9 / (HBM_BYTES_PER_S / 1e12), 4),
                torch_ms=round(t_ms, 3), torch_ms_min=round(t_min, 3), speedup_vs_torch=round(t_ms / ms, 2),
                digits_equal_torch=same, phases_ms=phases(ids, bits))
    if name == "bench_4mi":
        line["share_of_bench_step"] = [round(ms / s, 4) for s in BENCH_STEP_MS]
    print(json.dumps(line), flush=True)
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--skip-100mi", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_dedup.py needs a CUDA device")
    dev = torch.device("cuda")
    info = card()
    flush = torch.empty(1 << 27, dtype=torch.float32, device=dev)    # 512 MB written before every timed call
    g = torch.Generator(device=dev).manual_seed(0)
    results = []

    tok = bench.make_tokenizer(dev)
    items = bench.synth_items(bench.ITEMS_PER_GPU, seed=0, device=dev)
    table = tok.precompute_corpus_ids(items).clone()
    del items, tok
    torch.cuda.empty_cache()
    results.append(measure("bench_4mi", table, 8, args, flush))
    del table

    sizes = [("synth_32mi", 32 << 20, 3, 8), ("c4_4mi", 4 << 20, 4, 12)]
    if not args.skip_100mi:
        sizes.insert(1, ("synth_100mi", 100 << 20, 3, 8))
    for name, n, width, bits in sizes:
        ids = torch.randint(0, 1 << bits, (n, width), generator=g, device=dev)
        results.append(measure(name, ids, bits, args, flush))
        del ids
        torch.cuda.empty_cache()
    print(json.dumps(dict(summary="semid_dedup", **info, tables=[r["table"] for r in results],
                          all_equal_torch=all(r["digits_equal_torch"] for r in results))), flush=True)


if __name__ == "__main__":
    main()
