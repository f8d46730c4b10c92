#!/usr/bin/env python
"""bench.py -- items/s of HiD-VAE's residual-quantisation hot path on B200, through the reference-shaped module API.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl native|reference] [--no-sweep] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (BASELINE.json configs[4], "c5": bulk semantic-ID assignment, one GPU's share of the catalogue): a chunk of
4 Mi synthetic 768-d items per GPU through `HSemanticIdTokenizer.precompute_corpus_ids` (modules/tokenizer/h_semids.py:
109-195) -- encoder 768-512-256-128-32 (SiLU, L2 norm), 3 levels x 256 codes x dim 32, ids [N, 3] int64 out.  It is the
largest single-GPU configuration of BASELINE.json; C1 / C2 / C4 and the RQ-only launches are `sweep` entries.
ONE STEP = one pass over the GPU's 4 Mi items:
    per 1 Mi-item chunk     hv_encoder_forward  (enc_mlp_kernel: fused tcgen05 GEMM chain)     modules/encoder.py:23-36
                            hv_rq_forward       (rq_fwd_tc_v11_kernel: fused 3-level quantiser) modules/quantize.py:100-154
`value` = items / second with the items resident in HBM (12.9 GB: nothing survives in L2 between steps);
`e2e`   = the same call with the items in PINNED HOST memory: per-chunk H2D copies, the kernels and the D2H copy of the
          id table are all inside the timed region (PCIe-bound: 3,072 B in and 24 B out per item).
N > 1: every rank owns its own contiguous shard of 4 Mi items (weak scaling: the catalogue grows with the GPU count, as in
the 100 M-item job of BASELINE.json); no data-path collective -- the only exchange is ONE all_gather of the id tables
after the last step, inside the timed region.
--impl reference times the reference's own CPU algorithm (the oracle port, DESIGN.md section 8) on the host cores:
the batch-512 loop of precompute_corpus_ids over a bounded sample of the same catalogue, rank 0 only.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (os.path.join(ROOT, "hid-vae_b200"), ROOT):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

METRIC = "rq_encode_items_per_s"
UNIT = "items/s"
DIMS = [768, 512, 256, 128, 32]
N_LEVELS, CODEBOOK, EMBED = 3, 256, 32
ITEMS_PER_GPU = 1 << 22
CHUNK_ITEMS = 1 << 20
E2E_ITEMS = 1 << 20            # pinned-host leg: items per step (PCIe-bound; 3.2 GB of pinned memory per rank)
REF_SAMPLE_ITEMS = 1 << 16     # CPU arms: items per step (batches of 512, like the reference)
FLOP_ENCODER = 2.0 * sum(a * b for a, b in zip(DIMS[:-1], DIMS[1:]))        # 1,122,304 per item (SURVEY 8d)
FLOP_RQ = 2.0 * N_LEVELS * CODEBOOK * EMBED                                  # 49,152 per item
BYTES_ITEM = 4 * DIMS[0] + 8 * N_LEVELS                                      # 3,096 per item
WORKLOAD = dict(workload="c5: bulk semantic-ID assignment, per-GPU chunk of the catalogue through "
                         "HSemanticIdTokenizer.precompute_corpus_ids (encoder 768-512-256-128-32 + 3x256x32 quantiser)",
                items_per_gpu_per_step=ITEMS_PER_GPU, chunk_items=CHUNK_ITEMS, input_dim=DIMS[0], hidden_dims=DIMS[1:-1],
                embed_dim=EMBED, codebook_size=CODEBOOK, n_levels=N_LEVELS, encoder_precision="fused (fp16 operands, fp32 accumulate)",
                l2_between_steps="inputs larger than L2 (12.9 GB of items per step)")
MODE_ROT = 3


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(path):
        with open(path) as f:
            p = json.load(f)
        return dict(hbm=float(p["hbm_gbs"]), tensor=float(p["bf16_tflops"]), tensor_sustained=float(p["bf16_tflops_sustained"]),
                    source="MEASURED_PEAKS.json (measured)")
    return dict(hbm=6650.0, tensor=1590.0, tensor_sustained=1400.0, source="B200_PROFILING.md fallback")


def ncu_traffic():
    """dram read + write bytes per launch from the committed `ncu --set full` captures (profiles/r02_traffic.json)."""
    path = os.path.join(ROOT, "profiles", "r02_traffic.json")
    if os.path.isfile(path):
        with open(path) as f:
            return json.load(f)
    return {}


def synth_items(n, seed, device):
    """SURVEY 8d: item embeddings x = l2norm(randn(n, 768)), generated on the target device in slices."""
    g = torch.Generator(device=device).manual_seed(seed)
    x = torch.empty((n, DIMS[0]), dtype=torch.float32, device=device)
    for lo in range(0, n, 1 << 18):
        hi = min(lo + (1 << 18), n)
        x[lo:hi] = F.normalize(torch.randn(hi - lo, DIMS[0], generator=g, device=device), dim=-1)
    return x


def synth_codebook_weights(seed=1):
    """uniform(0,1) codebooks like the reference init (quantize.py:86-89), later levels centred and scaled to the
    residual magnitude ("trained-like", SURVEY 8d).  Level 0 is row-normalised by out_proj (codebook_normalize)."""
    g = torch.Generator().manual_seed(seed)
    cbs = torch.rand(N_LEVELS, CODEBOOK, EMBED, generator=g)
    for l in range(1, N_LEVELS):
        cbs[l] = (cbs[l] - 0.5) * (0.7 * 0.5 ** l)
    return cbs


def synth_rq(n, d, k, n_levels, seed, device="cpu"):
    """RQ-only inputs of the sweep / CPU legs: unit-norm encoder outputs, trained-like codebooks, upstream gradients."""
    g = torch.Generator().manual_seed(seed)
    x = F.normalize(torch.randn(n, d, generator=g), dim=-1)
    cbs = torch.rand(n_levels, k, d, generator=g)
    cbs[0] = F.normalize(cbs[0], dim=-1)
    for l in range(1, n_levels):
        cbs[l] = (cbs[l] - 0.5) * (0.7 * 0.5 ** l)
    g_emb = torch.randn(n_levels, n, d, generator=g) * 0.01
    g_loss = torch.full((n,), 1.0 / n)
    return x.to(device), cbs.to(device), g_emb.to(device), g_loss.to(device)


def make_tokenizer(device):
    from modules.tokenizer.h_semids import HSemanticIdTokenizer
    from oracle import encoder as OE  # seeded weights only (shared with the CPU arms so both sides encode the same model)
    tok = HSemanticIdTokenizer(input_dim=DIMS[0], output_dim=EMBED, hidden_dims=DIMS[1:-1], codebook_size=CODEBOOK,
                               n_layers=N_LEVELS, n_cat_feats=0, hrqvae_codebook_normalize=True, chunk_items=CHUNK_ITEMS,
                               encoder_precision="fused").to(device)
    with torch.no_grad():
        for lin, w in zip([m for m in tok.hrq_vae.encoder.mlp if isinstance(m, torch.nn.Linear)], OE.seeded_weights(DIMS, 2024)):
            lin.weight.copy_(w)
        for layer, w in zip(tok.hrq_vae.layers, synth_codebook_weights()):
            layer.embedding.weight.copy_(w)
    return tok.eval()


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 50 ms while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def stop(self, t0, t1):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        time.sleep(0.12)
        self.proc.terminate()
        rows = [r for (ts, r) in self.rows if t0 - 0.05 <= ts <= t1 + 0.05] or [r for (_, r) in self.rows]
        sm, smax, power, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            try:
                sm.append(float(r[0])), smax.append(float(r[1]))
                for nme, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(nme)
                power.append(float(r[2]))
            except Exception:
                pass
        # (the fused encoder runs the board at its power limit: SM clocks of 1.3-1.5 GHz under this step are the power cap at work,
        # whether or not a 50 ms sample happens to catch the sw_power_cap flag; the power draw is reported beside it)
        return dict(sm_mhz=statistics.median(sm) if sm else None, sm_max_mhz=max(smax) if smax else None,
                    reasons=sorted(reasons), samples=len(sm), power_w_max=max(power) if power else None)


def bind_host_memory_near(local_rank):
    """Best effort, before the pinned buffers of the end-to-end leg are allocated: run this process on the CPUs of the NUMA node
    the GPU hangs off and prefer that node's memory (set_mempolicy), so that eight ranks do not pull their 3 GB of pinned items
    through one socket's memory controllers and the inter-socket link.  A no-op on single-node hosts (the 1-GPU boxes are 16-vCPU
    single-node VMs).  Returns what it found and did, for the JSON line."""
    info = dict(gpu_numa_node=None, nodes=None, bound=False)
    try:
        nodes = sorted(int(d[4:]) for d in os.listdir("/sys/devices/system/node") if d.startswith("node") and d[4:].isdigit())
        info["nodes"] = len(nodes)
        pr = torch.cuda.get_device_properties(local_rank)
        bus = "%04x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read().strip())
        info["gpu_numa_node"] = node
        if node < 0 or len(nodes) < 2:
            return info
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
        import ctypes
        libc = ctypes.CDLL(None, use_errno=True)
        mask = ctypes.c_ulong(1 << node)
        MPOL_PREFERRED, SYS_set_mempolicy = 1, 238              # x86_64
        rc = libc.syscall(SYS_set_mempolicy, MPOL_PREFERRED, ctypes.byref(mask), ctypes.c_ulong(8 * ctypes.sizeof(mask)))
        info["bound"] = bool(cpus) and rc == 0
    except Exception as exc:                                     # never fail the bench over placement
        info["error"] = repr(exc)[:120]
    return info


DUMP_LIMIT_BYTES = 64 * 10 ** 6
DUMP_SAMPLE_ROWS = 1 << 21


def dump_outputs(out_dir, ids):
    """--dump-outputs: the id table the last timed step returned, as out_dir/sem_ids.npy in float32 (ids are < 2^24, so
    exact), for comparing two builds output for output.  A table above DUMP_LIMIT_BYTES (the gathered table of a multi-GPU
    run) is cut to a fixed seeded sample of DUMP_SAMPLE_ROWS rows, whose indices go to sem_ids_rows.npy (float64)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    ids = ids.cpu()
    if ids.numel() * 4 > DUMP_LIMIT_BYTES:
        rows = torch.randperm(ids.shape[0], generator=torch.Generator().manual_seed(0))[:DUMP_SAMPLE_ROWS].sort().values
        np.save(os.path.join(out_dir, "sem_ids_rows.npy"), rows.numpy().astype(np.float64))
        ids = ids[rows]
    np.save(os.path.join(out_dir, "sem_ids.npy"), ids.numpy().astype(np.float32))


def time_steps(fn, steps, warmup, flush=None):
    """W warm-ups, then K steps each bracketed by CUDA events on the current stream (optionally an L2 flush between
    steps); returns the per-step milliseconds."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    evs = []
    for _ in range(steps):
        if flush is not None:
            flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        evs.append((a, b))
    torch.cuda.synchronize()
    return [a.elapsed_time(b) for a, b in evs]


# ------------------------------------------------------------------------------------------------------------------
# native arm
# ------------------------------------------------------------------------------------------------------------------
def run_native(args):
    import torch.distributed as dist
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    assert torch.cuda.is_available(), "bench.py (native arm) needs a CUDA device; there is no CPU fallback"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import datetime
        dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=300))
    from hidvae_b200 import ops

    pk = peaks()
    tok = make_tokenizer(dev)
    n = ITEMS_PER_GPU
    x = synth_items(n, seed=1000 + rank, device=dev)          # this rank's shard of the catalogue
    n_chunks = (n + CHUNK_ITEMS - 1) // CHUNK_ITEMS
    tok.precompute_corpus_ids(x[:CHUNK_ITEMS])                # packs the weight image, sets kernel attributes
    torch.cuda.synchronize()

    sampler = ClockSampler(local) if rank == 0 else None
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t_mark0 = time.time()

    # ---- value: items resident in HBM; K steps + (N > 1) the final gather, barrier + synchronize on both sides ----
    step = lambda: tok.precompute_corpus_ids(x)
    for _ in range(args.warmup):
        step()
    if world > 1:
        tok.gather_shards()
        tok.cached_ids = None
        dist.barrier()
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    step_evs = []
    ev0.record()
    for _ in range(args.steps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        step()
        b.record()
        step_evs.append((a, b))
    gather_ms = None
    if world > 1:
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        table = tok.gather_shards()
        g1.record()
        assert table.shape == (world * n, N_LEVELS)
    ev1.record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
        gather_ms = g0.elapsed_time(g1)
    total_ms = ev0.elapsed_time(ev1)
    per_step = [a.elapsed_time(b) for a, b in step_evs]
    tm = torch.tensor([total_ms], device=dev)
    if world > 1:
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
    total_ms = float(tm.item())
    value = world * n * args.steps / (total_ms * 1e-3)
    t_mark1 = time.time()
    last_ids = tok.cached_ids.cpu() if args.dump_outputs and rank == 0 else None   # what the last timed step returned

    # ---- e2e: the same call on PINNED HOST items: chunk H2D + kernels + D2H of the id table inside the timed region ----
    n_e = min(E2E_ITEMS, n)
    cpus_before = os.sched_getaffinity(0)
    host_numa = bind_host_memory_near(local)
    x_host = torch.empty((n_e, DIMS[0]), dtype=torch.float32).pin_memory()
    x_host.copy_(x[:n_e])
    ids_host = torch.empty((n_e, N_LEVELS), dtype=torch.int64).pin_memory()
    if host_numa["bound"]:                                   # the pages are placed: give the CPU legs every core back
        import ctypes
        os.sched_setaffinity(0, cpus_before)
        ctypes.CDLL(None).syscall(238, 0, None, 0)           # set_mempolicy(MPOL_DEFAULT)

    def e2e_step():
        ids_host.copy_(tok.precompute_corpus_ids(x_host), non_blocking=True)

    if world > 1:
        dist.barrier()
    e2e_ms = time_steps(e2e_step, args.steps, args.warmup)
    te = torch.tensor([sum(e2e_ms)], device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_total = float(te.item())
    e2e_value = world * n_e * args.steps / (e2e_total * 1e-3)
    ids_dev = tok.precompute_corpus_ids(x[:n_e])
    torch.cuda.synchronize()
    e2e_same = bool(torch.equal(ids_dev.cpu(), ids_host))      # host-fed and device-resident passes agree bit for bit

    # ---- the same workload on a catalogue kept in HALF precision (a data format beside the path: half the HBM / PCIe bytes;
    #      the fused encoder rounds fp32 items to fp16 anyway, so the id table must equal the fp32 catalogue's bit for bit).
    #      Reported beside the headline, never instead of it: the reference's items are fp32. ----
    half_cat = None
    if not args.no_sweep:
        x16 = x.half()
        step16 = lambda: tok.precompute_corpus_ids(x16)
        ms16 = time_steps(step16, args.steps, args.warmup)
        ids16 = tok.precompute_corpus_ids(x16[:n_e]).clone()
        x16_host = torch.empty((n_e, DIMS[0]), dtype=torch.float16).pin_memory()
        x16_host.copy_(x16[:n_e])

        def e2e16_step():
            ids_host.copy_(tok.precompute_corpus_ids(x16_host), non_blocking=True)

        if world > 1:
            dist.barrier()
        e16 = time_steps(e2e16_step, args.steps, args.warmup)
        t16 = torch.tensor([sum(ms16), sum(e16)], device=dev)
        if world > 1:
            dist.all_reduce(t16, op=dist.ReduceOp.MAX)
        half_cat = dict(items="fp16 [N, 768] (x.half() of the same synthetic catalogue)",
                        value=world * n * args.steps / (float(t16[0]) * 1e-3), unit=UNIT, ms_per_step=float(t16[0]) / args.steps,
                        e2e=dict(value=world * n_e * args.steps / (float(t16[1]) * 1e-3), unit=UNIT, ms_per_step=float(t16[1]) / args.steps,
                                 h2d_bytes_per_step=n_e * DIMS[0] * 2, d2h_bytes_per_step=n_e * N_LEVELS * 8),
                        ids_equal_fp32_catalogue=bool(torch.equal(ids16, ids_dev)))
        del x16, x16_host

    # ---- per-kernel durations at the step's launch shape (CUDA events around each C-ABI call) -> roofline ----
    model = tok.hrq_vae
    image = model.encoder._weight_image()
    cbs = model.effective_codebooks().detach()
    packed = ops.pack_codebooks(cbs)
    z = torch.empty((CHUNK_ITEMS, EMBED), device=dev)
    ids_buf = torch.empty((CHUNK_ITEMS, N_LEVELS), dtype=torch.int64, device=dev)
    ci = [0]

    def enc_launch():   # walks the shard so that every launch reads fresh items from HBM, as in the step
        lo = (ci[0] % n_chunks) * CHUNK_ITEMS
        ci[0] += 1
        ops.encoder_forward(x[lo:lo + CHUNK_ITEMS], image, normalize=True, out=z)

    reps = 2 * n_chunks
    t_enc = statistics.mean(time_steps(enc_launch, reps, 3))
    t_rq = statistics.mean(time_steps(lambda: ops.rq_encode(z, cbs, ids_out=ids_buf, packed=packed), reps, 3))
    traffic = ncu_traffic()
    kernels = [
        dict(kernel="enc_mlp_kernel (fused encoder 768-512-256-128-32)", ms=t_enc, bound="tensor", rows_per_launch=CHUNK_ITEMS,
             achieved=FLOP_ENCODER * CHUNK_ITEMS / (t_enc * 1e-3) / 1e12, peak=pk["tensor_sustained"], unit="TFLOP/s",
             hbm_gbs=CHUNK_ITEMS * (4 * DIMS[0] + 4 * EMBED) / (t_enc * 1e-3) / 1e9, traffic=traffic.get("enc_mlp_kernel")),
        dict(kernel="rq_fwd_tc_v11_kernel (fused 3-level quantiser, ids only)", ms=t_rq, bound="tensor", rows_per_launch=CHUNK_ITEMS,
             achieved=FLOP_RQ * CHUNK_ITEMS / (t_rq * 1e-3) / 1e12, peak=pk["tensor_sustained"], unit="TFLOP/s",
             hbm_gbs=CHUNK_ITEMS * (4 * EMBED + 8 * N_LEVELS) / (t_rq * 1e-3) / 1e9, traffic=(int(traffic["rq_encode"]["dram_bytes"] * CHUNK_ITEMS / (1 << 22)) if "rq_encode" in traffic else None)),
    ]
    for kk in kernels:
        kk["frac"] = kk["achieved"] / kk["peak"]
        kk["frac_of_burst_peak"] = kk["achieved"] / pk["tensor"]
    dom = max(kernels, key=lambda kk: kk["ms"])
    step_ms = statistics.mean(per_step)
    roofline = dict(bound=dom["bound"], achieved=dom["achieved"], peak=dom["peak"], unit=dom["unit"], frac=dom["frac"],
                    traffic=dom["traffic"], kernel=dom["kernel"], kernel_ms=dom["ms"], rows_per_launch=CHUNK_ITEMS,
                    algorithmic_flop_per_item=FLOP_ENCODER, frac_of_burst_peak=dom["frac_of_burst_peak"],
                    share_of_step=dom["ms"] * n_chunks / step_ms,
                    peak_source=pk["source"] + ", sustained bf16 (the kernel is timed inside a long step; burst = %.1f)" % pk["tensor"],
                    traffic_source="profiles/r02_traffic.json (ncu --set full, dram read + write of one launch; the quantiser's 4 Mi-row capture is scaled to the rows of this launch)",
                    step=dict(items_per_s=n / (step_ms * 1e-3), tflops=(FLOP_ENCODER + FLOP_RQ) * n / (step_ms * 1e-3) / 1e12,
                              frac_of_sustained_peak=(FLOP_ENCODER + FLOP_RQ) * n / (step_ms * 1e-3) / 1e12 / pk["tensor_sustained"],
                              hbm_gbs=BYTES_ITEM * n / (step_ms * 1e-3) / 1e9),
                    kernels=kernels)

    train_dp = run_train_dp(rank, world, dev) if not args.no_sweep else None

    sweep = None
    if rank == 0 and world == 1 and not args.no_sweep:
        del x_host
        sweep = run_sweep(ops, pk, dev)

    clocks = sampler.stop(t_mark0, t_mark1) if sampler else None
    if rank == 0:
        cpu = cpu_baseline(budget_s=6.0) if world == 1 else None
        line = dict(metric=METRIC, value=value, unit=UNIT, n_gpus=world, steps=args.steps, warmup=args.warmup,
                    ms_per_step=total_ms / args.steps, higher_is_better=True, scaling="weak", vs_baseline=None,
                    dtype="f16 operands / f32 accumulate (encoder GEMMs, TF32-grade); bf16x3 split / f32 (quantiser scores); ids int64",
                    data="synthetic",
                    config=dict(WORKLOAD, parallelism=f"dp{world} (item shards, no data-path collective)",
                                step_ms_min=min(per_step), step_ms_max=max(per_step), step_ms_mean=step_ms,
                                final_gather_ms=gather_ms,
                                collective=("one all_gather of the [N, 3] int64 id tables after the last step, inside the timed region"
                                            if world > 1 else None)),
                    e2e=dict(value=e2e_value, unit=UNIT, h2d_bytes_per_step=n_e * DIMS[0] * 4, d2h_bytes_per_step=n_e * N_LEVELS * 8,
                             ms_per_step=e2e_total / args.steps, items_per_step_per_gpu=n_e,
                             call="HSemanticIdTokenizer.precompute_corpus_ids(pinned host tensor) + id table -> pinned host",
                             ids_equal_device_resident_pass=e2e_same, host_numa=host_numa,
                             pcie_gbs=(n_e * (DIMS[0] * 4 + N_LEVELS * 8)) / (e2e_total / args.steps * 1e-3) / 1e9),
                    gpu_launches=(2 * n_chunks + 1) * args.steps, roofline=roofline, cpu_baseline=cpu, clocks=clocks, impl="native")
        if half_cat is not None:
            line["half_precision_catalogue"] = half_cat
        if sweep is not None:
            line["sweep"] = sweep
        if train_dp is not None:
            line["train_dp"] = train_dp
        if last_ids is not None:
            dump_outputs(args.dump_outputs, last_ids)
        OUT.emit(json.dumps(line))
    if world > 1:
        torch.cuda.synchronize()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)   # (tearing NCCL down was seen to hang on 2 x B200 with NCCL 2.28.9; nothing is pending here)


# ------------------------------------------------------------------------------------------------------------------
# C3: KuaiRand-shaped data-parallel training (k-means codebook init, tag heads, uniqueness loss, ONE flat gradient exchange)
# ------------------------------------------------------------------------------------------------------------------
def run_train_dp(rank, world, dev):
    """BASELINE.json configs[2] through the module API: HRqVae.forward + backward on this rank's own batches (the
    reference's per-rank sampling, train_hidvae.py:213,233), the 29 MB flat gradient all-reduce of
    hidvae_b200.dist.FlatGradAllReduce (what DDP does inside accelerator.backward, train_hidvae.py:709) and the AdamW
    step.  Codebooks come from the sharded k-means init (init/kmeans.py through Kmeans(process_group=...)).  Before
    timing, hv_peer_allreduce and NCCL are run on the same buffer and compared.  Weak scaling: per-rank batch fixed."""
    import torch.distributed as dist
    from data.schemas import TaggedSeqBatch
    from hidvae_b200 import dist as hv_dist
    from modules.h_rqvae import HRqVae
    from modules.quantize import QuantizeForwardMode
    from train_hidvae import init_codebooks
    import numpy as np

    counts = [37, 168, 353]                                   # configs/h_rqvae_kuairand.gin:32
    torch.manual_seed(0)
    np.random.seed(0)
    model = HRqVae(input_dim=768, embed_dim=32, hidden_dims=[512, 256, 128], codebook_size=256, codebook_kmeans_init=True,
                   codebook_normalize=True, codebook_mode=QuantizeForwardMode.ROTATION_TRICK, n_layers=3, n_cat_features=0,
                   commitment_weight=0.5, tag_class_counts=counts, tag_embed_dim=768, sem_id_uniqueness_weight=0.5,
                   sem_id_uniqueness_margin=0.5).to(dev).train()
    hv_dist.broadcast_parameters(model)
    n_items = 32768                                            # per rank (the reference does not state KuaiRand's item count)
    g = torch.Generator(device=dev).manual_seed(77 + rank)
    x = F.normalize(torch.randn(n_items, 768, generator=g, device=dev), dim=-1)
    tags_emb = torch.randn(n_items, 3, 768, generator=g, device=dev)
    tags_idx = torch.stack([torch.randint(0, c, (n_items,), generator=g, device=dev) for c in counts], dim=1)
    tags_idx[torch.rand(n_items, 3, generator=g, device=dev) < 0.05] = -1
    res = dict(model="KuaiRand-shaped HiD-VAE (7.24 M parameters, tag heads, k-means init, uniqueness loss)", items_per_rank=n_items)

    # sharded k-means codebook init: min(20000, N) rows of the GLOBAL matrix, this rank's share of them
    lo, hi = hv_dist.shard_range(20000, rank, world)
    t0 = time.perf_counter()
    init_codebooks(model, x[: hi - lo], process_group=dist.group.WORLD if world > 1 else None)
    torch.cuda.synchronize()
    res["kmeans_init_s"] = time.perf_counter() - t0
    if world > 1:   # every rank must hold the same codebooks afterwards (the reference's ranks silently diverge)
        cb = torch.stack([l.embedding.weight.detach() for l in model.layers])
        ref = cb.clone()
        dist.broadcast(ref, src=0)
        same = torch.tensor([float(torch.equal(cb, ref))], device=dev)
        dist.all_reduce(same, op=dist.ReduceOp.MIN)
        res["codebooks_identical_on_all_ranks"] = bool(same.item())

    grads = hv_dist.FlatGradAllReduce(model.parameters())
    opt = torch.optim.AdamW(model.parameters(), lr=1e-4, weight_decay=0.01, fused=True)
    res["flat_gradient_bytes"] = grads.flat.numel() * 4
    res["matmul_precision"] = "tf32 (torch.set_float32_matmul_precision('high'), as the reference sets at modules/h_rqvae.py:21)"
    precision_before = torch.get_float32_matmul_precision()
    torch.set_float32_matmul_precision("high")

    if world > 1:   # the one-kernel peer-memory exchange against NCCL on the same data
        try:
            cb_n = sum(l.embedding.weight.numel() for l in model.layers)
            peer = hv_dist.PeerAllReduce(cb_n, dev)
            a = torch.randn(cb_n, generator=g, device=dev)
            b = a.clone()
            for _ in range(3):                                  # repeated calls exercise the flag parities
                a2, b2 = a.clone(), b.clone()
                peer(a2)
                dist.all_reduce(b2)
                ok = torch.allclose(a2, b2, rtol=1e-6, atol=1e-6)
            peer.check()                                        # no call gave up waiting for a rank
            okt = torch.tensor([float(ok)], device=dev)
            dist.all_reduce(okt, op=dist.ReduceOp.MIN)
            res["allreduce_checked"] = bool(okt.item())
            res["allreduce_check"] = "hv_peer_allreduce == NCCL all_reduce on the same 24,576-float buffer, 3 consecutive calls, every rank"
        except Exception as e:  # noqa: BLE001
            res["allreduce_checked"] = False
            res["allreduce_check"] = f"peer-memory exchange unavailable: {type(e).__name__}: {e}"

    from hidvae_b200.graph_step import GraphedTrainStep
    fetch = lambda idx: TaggedSeqBatch(None, None, None, x[idx], None, None, tags_emb[idx], tags_idx[idx])
    opt_g = torch.optim.AdamW(model.parameters(), lr=torch.tensor(1e-4, device=dev), weight_decay=0.01, capturable=True, fused=True)

    def timed(fn, reps):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            fn()
        b.record()
        torch.cuda.synchronize()
        ms = torch.tensor([a.elapsed_time(b) / reps], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    for bs in (128, 8192):
        last = {}

        def step():   # the eager step: what a line-by-line port of train_hidvae.py:700-770 costs (launch-bound)
            grads.zero()
            out = model(fetch(torch.randint(0, n_items, (bs,), device=dev, generator=g)), gumbel_t=0.2)
            grads.backward(out.loss)
            grads.all_reduce()
            opt.step()
            last["loss"] = out.loss.detach()   # (a live autograd graph would pin AccumulateGrad nodes to this stream)

        for _ in range(5):
            step()
        eager_ms = timed(step, 20)
        last.clear()
        # the same step as two CUDA-graph replays around the NCCL exchange (hidvae_b200/graph_step.py)
        graphed = GraphedTrainStep(model, opt_g, grads, fetch, bs, n_items, gumbel_t=0.2, generator=g, warmup=3)
        for _ in range(3):
            graphed()
        ms = timed(graphed, 50)
        # the exchange alone (NCCL, 29 MB) on the same buffer
        ar_ms = timed(lambda: dist.all_reduce(grads.flat), 20) if world > 1 else None
        res[f"batch{bs}_per_rank"] = dict(ms_per_step=ms, items_per_s=world * bs / (ms * 1e-3), eager_ms_per_step=eager_ms,
                                           eager_items_per_s=world * bs / (eager_ms * 1e-3), flat_allreduce_ms=ar_ms,
                                           loss=float(graphed.stats[0]), step="CUDA graphs: gather + forward + backward | NCCL "
                                           "all-reduce of the flat gradient | AdamW")
        del graphed
    torch.set_float32_matmul_precision(precision_before)
    return res


# ------------------------------------------------------------------------------------------------------------------
# sweep: the other BASELINE.json shapes and the RQ-only launches (supplementary, N = 1 only)
# ------------------------------------------------------------------------------------------------------------------
class GraphedStep:
    def __init__(self, fn):
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(3):
                fn()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.out = fn()

    def __call__(self):
        self.graph.replay()
        return self.out


def run_sweep(ops, pk, dev):
    res = []
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    mean = lambda fn, reps, fl=None: statistics.mean(time_steps(fn, reps, 3, fl))

    # RQ-only launches: C1 batch, the C5 chunk on 32-d encoder outputs, C4
    for name, (n, d, k, L) in {"c1_batch1024_rq_only": (1024, 32, 256, 3), "c5_rq_only_4Mi": (1 << 22, 32, 256, 3),
                               "c4_65536x64x4096x4": (65536, 64, 4096, 4)}.items():
        x, cbs, g_emb, g_loss = synth_rq(n, d, k, L, seed=7, device=dev)
        packed = ops.pack_codebooks(cbs)
        fl = None if n * d * 4 > (128 << 20) else flush
        t_enc = mean(lambda: ops.rq_encode(x, cbs, packed=packed), 20, fl)
        ent = dict(case=name, n=n, d=d, k=k, L=L, encode_ms=t_enc, encode_items_per_s=n / (t_enc * 1e-3),
                   encode_tflops=2.0 * k * d * L * n / (t_enc * 1e-3) / 1e12)
        ent["encode_frac_of_bf16_burst"] = ent["encode_tflops"] / pk["tensor"]
        ent["encode_frac_of_bf16_sustained"] = ent["encode_tflops"] / pk["tensor_sustained"]
        if d == 32:
            out = ops.rq_forward(x, cbs, MODE_ROT, True, 0.4, want_emb=True, want_loss=True, packed=packed)
            t_f = mean(lambda: ops.rq_forward(x, cbs, MODE_ROT, True, 0.4, want_emb=True, want_loss=True, packed=packed), 20, fl)
            t_b = mean(lambda: ops.rq_backward(x, cbs, out.ids, MODE_ROT, True, 0.4, g_emb, g_loss, None), 20, fl)
            byt = n * (4 * d * (3 + 2 * L) + 16 * L + 8)
            ent.update(train_fwd_ms=t_f, train_bwd_ms=t_b, train_items_per_s=n / ((t_f + t_b) * 1e-3),
                       train_hbm_gbs=byt / ((t_f + t_b) * 1e-3) / 1e9)
            ent["train_frac_of_hbm_peak"] = ent["train_hbm_gbs"] / pk["hbm"]
        res.append(ent)
        del x, cbs, g_emb, g_loss

    # C2: the Amazon-Beauty-shaped catalogue pass of round 1 (train forward + backward + eval encode, one CUDA graph)
    n, d, k, L, beta = 12101, 32, 256, 3, 0.4
    x, cbs, g_emb, g_loss = synth_rq(n, d, k, L, seed=0, device=dev)
    side = torch.cuda.Stream()

    def c2_step():
        main = torch.cuda.current_stream()
        packed = ops.pack_codebooks(cbs)
        side.wait_stream(main)
        with torch.cuda.stream(side):
            ids = ops.rq_encode(x, cbs, packed=packed)
        out = ops.rq_forward(x, cbs, MODE_ROT, True, beta, want_emb=True, want_loss=True, packed=packed)
        g = ops.rq_backward(x, cbs, out.ids, MODE_ROT, True, beta, g_emb, g_loss, None)
        main.wait_stream(side)
        packed.record_stream(side)
        return out, g, ids

    graphed = GraphedStep(c2_step)
    t_c2 = mean(graphed, 200, flush)
    res.append(dict(case="c2_catalogue_pass_12101_items (train fwd + bwd + eval encode, CUDA graph)", n=n, ms=t_c2,
                    items_per_s=n / (t_c2 * 1e-3), eager_ms=mean(c2_step, 50, flush)))
    del graphed

    # C1 through the module API: HRqVae.forward + backward, batch 1024, 768-d items, rotation trick, untagged
    from data.schemas import SeqBatch
    from modules.h_rqvae import HRqVae
    from modules.quantize import QuantizeForwardMode
    model = HRqVae(input_dim=768, embed_dim=32, hidden_dims=[512, 256, 128], codebook_size=256, codebook_kmeans_init=False,
                   codebook_normalize=True, codebook_mode=QuantizeForwardMode.ROTATION_TRICK, n_layers=3, n_cat_features=0,
                   commitment_weight=0.4, tag_class_counts=[38, 168, 348]).to(dev).train()
    xb = synth_items(1024, seed=5, device=dev)
    batch = SeqBatch(user_ids=None, ids=None, ids_fut=None, x=xb, x_fut=None, seq_mask=None)

    def c1_step():
        model.zero_grad(set_to_none=True)
        model(batch, gumbel_t=0.2).loss.backward()

    t_c1 = mean(c1_step, 30, flush)
    # the same forward + backward replayed as one CUDA graph (gradients accumulate into static buffers, as the trainer's
    # GraphedTrainStep does): what the launch-bound eager number hides
    for p_ in model.parameters():
        p_.grad = torch.zeros_like(p_)
    torch.cuda.synchronize()

    def c1_fwd_bwd():
        model(batch, gumbel_t=0.2).loss.backward()

    c1_graph = GraphedStep(c1_fwd_bwd)
    t_c1g = mean(c1_graph, 50, flush)
    res.append(dict(case="c1_HRqVae.forward+backward_batch1024_untagged (module API: PyTorch MLPs + fused RQ)", n=1024,
                    ms=t_c1g, items_per_s=1024 / (t_c1g * 1e-3), eager_ms=t_c1, note="ms = one CUDA-graph replay, eager_ms = eager PyTorch"))
    return res


# ------------------------------------------------------------------------------------------------------------------
# CPU arms: the oracle port of the reference algorithm (the one place besides tests/smoke that may execute oracle/)
# ------------------------------------------------------------------------------------------------------------------
def _cpu_model():
    from oracle import encoder as OE
    from oracle import rq as O
    enc_w = OE.seeded_weights(DIMS, 2024)
    cb_w = synth_codebook_weights()
    cbs = [O.effective_codebook(cb_w[l], l == 0) for l in range(N_LEVELS)]
    return enc_w, cb_w, cbs


def _timed(fn, budget_s, min_reps=3, max_reps=200, warm=1):
    for _ in range(warm):
        fn()
    times = []
    t_end = time.perf_counter() + budget_s
    while len(times) < min_reps or (time.perf_counter() < t_end and len(times) < max_reps):
        t0 = time.perf_counter()
        fn()
        times.append(time.perf_counter() - t0)
    return statistics.median(times), len(times)


def cpu_baseline(budget_s):
    """The five CPU legs of BASELINE.md section 3 on this box's host cores (oracle port, torch CPU, all threads); `value`
    is the leg that matches the headline workload: the batch-512 precompute_corpus_ids loop."""
    from oracle import encoder as OE
    from oracle import hrqvae as OH
    from oracle import kmeans as OK
    from oracle import rq as O
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    enc_w, cb_w, cbs = _cpu_model()
    legs = {}
    # (iv) the headline workload: precompute_corpus_ids loop, batch 512, encoder + quantiser
    xs = synth_items(REF_SAMPLE_ITEMS, seed=1000, device="cpu")
    t, reps = _timed(lambda: OH.precompute_corpus_ids(xs, enc_w, cbs, True), budget_s, min_reps=2)
    value = REF_SAMPLE_ITEMS / t
    legs["precompute_corpus_ids_batch512_65536_items"] = dict(items_per_s=value, ms=t * 1e3, reps=reps)
    # (i) C1 untagged HRqVae.forward + backward, batch 1024 (the tagged variant needs the tag heads, which are outside the
    #     hot path and have no oracle port: SURVEY section 2 row 11)
    dec_w = OE.seeded_weights(DIMS[::-1], 2025)
    x1 = xs[:1024]
    for mname, mode in (("ste", O.MODE_STE), ("rotation", O.MODE_ROTATION_TRICK)):
        params = [w.clone().requires_grad_(True) for w in (*enc_w, *dec_w, *cb_w)]
        ew, dw, cw = params[:4], params[4:8], params[8:]

        def step(mode=mode, ew=ew, dw=dw, cw=cw, params=params):
            for p in params:
                p.grad = None
            OH.untagged_step(x1, ew, dw, cw, mode, 0.4, True).backward()

        t, reps = _timed(step, budget_s / 3)
        legs[f"c1_hrqvae_forward_backward_untagged_{mname}"] = dict(items_per_s=1024 / t, ms=t * 1e3, reps=reps)
    # (ii) C1 RQ-only get_semantic_ids forward + backward
    xr, cr, _, _ = synth_rq(1024, 32, 256, 3, seed=7)
    for mname, mode in (("ste", O.MODE_STE), ("rotation", O.MODE_ROTATION_TRICK)):
        def step(mode=mode):
            xg = xr.clone().requires_grad_(True)
            cg = [cr[l].clone().requires_grad_(True) for l in range(3)]
            out = O.rq_forward(xg, cg, mode, 0.4, True)
            (out.embeddings.sum() + out.quantize_loss.sum()).backward()

        t, reps = _timed(step, budget_s / 4)
        legs[f"c1_rq_only_forward_backward_{mname}"] = dict(items_per_s=1024 / t, ms=t * 1e3, reps=reps)
    # (iii) eval encode at 65,536 rows: C1 shape, and C4 shape on a reduced row count (the [N, 4096] fp32 tables)
    xe, ce, _, _ = synth_rq(65536, 32, 256, 3, seed=7)
    with torch.no_grad():
        t, reps = _timed(lambda: O.rq_forward(xe, [ce[l] for l in range(3)], O.MODE_STE, 0.25, False), budget_s / 3, min_reps=2)
        legs["eval_encode_rq_only_65536x32_k256_l3"] = dict(items_per_s=65536 / t, ms=t * 1e3, reps=reps)
        x4, c4, _, _ = synth_rq(16384, 64, 4096, 4, seed=7)
        t, reps = _timed(lambda: O.rq_forward(x4, [c4[l] for l in range(4)], O.MODE_STE, 0.25, False), budget_s / 3, min_reps=2, warm=0)
        legs["eval_encode_rq_only_c4_shape_16384x64_k4096_l4 (N reduced from 65,536)"] = dict(items_per_s=16384 / t, ms=t * 1e3, reps=reps)
    # (v) Kmeans.run on 20,000 x 32, K = 256, fixed seed; bounded to 8 Lloyd iterations (the reference runs to 1e-10)
    xk = F.normalize(torch.randn(20000, 32, generator=torch.Generator().manual_seed(3)), dim=-1)
    import numpy as np
    init_idx = np.random.RandomState(0).choice(20000, 256, replace=False)
    t0 = time.perf_counter()
    km = OK.kmeans_run(xk, 256, max_iters=8, init_idx=init_idx)
    dt = time.perf_counter() - t0
    legs["kmeans_20000x32_k256"] = dict(ms_per_lloyd_iteration=dt / max(km.n_iters, 1) * 1e3, iterations=km.n_iters, total_ms=dt * 1e3,
                                        note="bounded to 8 Lloyd iterations; the reference runs to max shift < 1e-10 (51 iterations in the survey)")
    return dict(value=value, unit=UNIT, cores=cores, kind="port",
                sample=f"{REF_SAMPLE_ITEMS} items of the same synthetic catalogue per pass, batches of 512 (oracle/hrqvae.py "
                       f"precompute_corpus_ids: encoder + quantiser, torch {torch.__version__} CPU, {cores} threads)",
                legs=legs)


def run_reference(args):
    """The reference's own CPU algorithm (oracle port) on this box's host cores; rank 0 only."""
    if int(os.environ.get("RANK", 0)) != 0:
        return
    from oracle import hrqvae as OH
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    enc_w, _cb_w, cbs = _cpu_model()
    xs = synth_items(REF_SAMPLE_ITEMS, seed=1000, device="cpu")
    steps, warmup = args.steps, min(args.warmup, 5)
    for _ in range(warmup):
        OH.precompute_corpus_ids(xs, enc_w, cbs, True)
    t0 = time.perf_counter()
    for _ in range(steps):
        ids = OH.precompute_corpus_ids(xs, enc_w, cbs, True)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, ids)
    value = REF_SAMPLE_ITEMS * steps / dt
    sample = (f"{steps} steps x {REF_SAMPLE_ITEMS} items of the same synthetic catalogue, batches of 512 like the reference "
              f"(oracle/hrqvae.py, torch {torch.__version__} CPU, {cores} threads)")
    OUT.emit(json.dumps(dict(metric=METRIC, value=value, unit=UNIT, n_gpus=args.gpus, steps=steps, warmup=warmup,
                             ms_per_step=dt / steps * 1e3, higher_is_better=True, scaling="weak", vs_baseline=None,
                             dtype="f32", data="synthetic",
                             config=dict(WORKLOAD, parallelism="cpu", items_per_gpu_per_step=REF_SAMPLE_ITEMS, chunk_items=512,
                                         encoder_precision="fp32",
                                         l2_between_steps="n/a (host arm: a bounded sample of the same catalogue per step)"),
                             impl="reference", cpu_baseline=dict(value=value, unit=UNIT, cores=cores, kind="port", sample=sample),
                             e2e=dict(value=value, unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0))))


class QuietStdout:
    """Everything but the final JSON line goes to stderr: libraries print to fd 1 on their own (NCCL's version banner),
    and the contract is ONE line on stdout."""

    def __enter__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        os.dup2(2, 1)
        return self

    def emit(self, text):
        sys.stdout.flush()
        os.write(self.saved, (text + "\n").encode())

    def __exit__(self, *exc):
        sys.stdout.flush()
        os.dup2(self.saved, 1)
        os.close(self.saved)
        return False


OUT = None


def main():
    global OUT
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--no-sweep", action="store_true")
    ap.add_argument("--chunk-items", type=int, default=CHUNK_ITEMS, help="items per launch inside precompute_corpus_ids (tuning runs)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the id table of the last timed step to DIR/sem_ids.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    globals()["CHUNK_ITEMS"] = WORKLOAD["chunk_items"] = args.chunk_items
    args.warmup = max(args.warmup, 3) if args.impl == "native" else args.warmup
    with QuietStdout() as OUT:
        if args.impl == "reference":
            run_reference(args)
        else:
            run_native(args)


if __name__ == "__main__":
    main()
