"""torchrun check of the sharded collision digit (HSemanticIdTokenizer(use_dedup_dim=True) with shard=(rank, world)) on
real GPUs over NCCL:
  - every rank's shard, before gather_shards, already holds the digits of the whole catalogue on its rows;
  - the gathered table equals the single-process table, and dedup_stats agree.

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 tools/check_dedup_shards.py
Prints one JSON line {"ok": true, ...} on rank 0.
"""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "hid-vae_b200"), ROOT]
import torch  # noqa: E402

import bench  # noqa: E402
from hidvae_b200 import dist as hv  # noqa: E402
from modules.tokenizer.h_semids import HSemanticIdTokenizer  # noqa: E402

rank, world, local = hv.init_from_env("nccl")
dev = torch.device("cuda", local)

plain = bench.make_tokenizer(dev)
tok = HSemanticIdTokenizer(input_dim=bench.DIMS[0], output_dim=bench.EMBED, hidden_dims=bench.DIMS[1:-1],
                           codebook_size=bench.CODEBOOK, n_layers=bench.N_LEVELS, n_cat_feats=0, hrqvae_codebook_normalize=True,
                           chunk_items=1 << 17, encoder_precision="fused", use_dedup_dim=True).to(dev).eval()
tok.load_state_dict(plain.state_dict())
items = bench.synth_items(300001, seed=9, device=dev)          # a ragged catalogue, identical on every rank

whole = tok.precompute_corpus_ids(items).clone()
whole_stats = tok.dedup_stats
_, inv = torch.unique(whole[:, :3], dim=0, return_inverse=True)  # torch formulation of the digits, as a cross-check
order = torch.argsort(inv, stable=True)
counts = torch.bincount(inv)
pos = torch.empty_like(order)
pos[order] = torch.arange(order.numel(), device=dev)
assert torch.equal(whole[:, 3], pos - (counts.cumsum(0) - counts)[inv]), "single-process digits differ from torch"
assert int(whole[:, 3].max()) > 0, "the catalogue has no collision: nothing to check"

tok.reset()
shard = tok.precompute_corpus_ids(items, shard=(rank, world)).clone()
per = (whole.shape[0] + world - 1) // world
lo, hi = min(rank * per, whole.shape[0]), min((rank + 1) * per, whole.shape[0])
assert torch.equal(shard, whole[lo:hi]), f"rank {rank}: the shard's digits are not the catalogue's"
assert tok.dedup_stats == whole_stats, f"rank {rank}: dedup_stats {tok.dedup_stats} != {whole_stats}"
gathered = tok.gather_shards()
assert torch.equal(gathered, whole), "gathered shards differ from the single-process table"

if rank == 0:
    print(json.dumps({"ok": True, "world": world, "rows": whole_stats[0], "distinct": whole_stats[1],
                      "max_digit": whole_stats[2]}))
torch.distributed.destroy_process_group()
