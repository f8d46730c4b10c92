"""Time hv_kmeans_accumulate (one Lloyd update's sums and counts) at the shapes that matter, with CUDA events:

    K = 4096, N = 65,536, D = 64   the stress shape (segmented form: key sort + one warp per cluster)
    K = 256,  N = 20,000, D = 32   the bench's codebook init (scan form: one CTA per cluster)

Inputs are L2-resident after the first launch (17 MB and 2.6 MB), as they are inside the Lloyd loop.  Per shape, one JSON
line with the eager call time (host launches included) and the device time of calls replayed from a CUDA graph; then a
line with the card's name and power limit.  A/B of two builds: run it once per library,
HIDVAE_B200_LIB=path/to/libhidvae_b200.so python tools/bench_kmeans.py --tag NAME.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "hid-vae_b200"), ROOT]
import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

from hidvae_b200 import ops  # noqa: E402

SHAPES = {"stress_k4096_n65536_d64": (4096, 65536, 64), "init_k256_n20000_d32": (256, 20000, 32)}


def card():
    q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader"], capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(), "nvidia_smi": q.stdout.strip() or q.stderr.strip()}


def timed(fn, reps):
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    start.record()
    for _ in range(reps):
        fn()
    stop.record()
    torch.cuda.synchronize()
    return start.elapsed_time(stop) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=2000)
    ap.add_argument("--tag", default=os.path.basename(os.environ.get("HIDVAE_B200_LIB", "shipped")))
    args = ap.parse_args()
    torch.cuda.set_device(0)
    g = torch.Generator(device="cuda").manual_seed(0)
    for name, (k, n, d) in SHAPES.items():
        x = F.normalize(torch.randn(n, d, device="cuda", generator=g), dim=-1)
        assign = torch.randint(0, k, (n,), device="cuda", generator=g)
        prev = torch.randint(0, k, (n,), device="cuda", generator=g)
        call = lambda: ops.kmeans_accumulate(x, assign, k, prev)
        for _ in range(20):
            call()
        res = {"tag": args.tag, "shape": name, "eager_ms": timed(call, args.reps)}
        # device time alone: 50 calls captured in one CUDA graph, replayed (the eager figure includes the host's launches)
        graph = torch.cuda.CUDAGraph()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            call()
        torch.cuda.current_stream().wait_stream(side)
        with torch.cuda.graph(graph):
            for _ in range(50):
                call()
        graph.replay()
        res["graph_ms"] = timed(graph.replay, max(args.reps // 50, 10)) / 50
        print(json.dumps(res), flush=True)
    print(json.dumps(card()), flush=True)


if __name__ == "__main__":
    main()
