"""Bulk semantic-ID assignment with the interface of the reference's `HSemanticIdTokenizer`
(modules/tokenizer/h_semids.py): `precompute_corpus_ids`, `cached_ids`, `exists_prefix`, `_tokenize_seq_batch_from_cached`, `forward`, `sem_ids_dim`,
`reset`.

The reference walks the catalogue in DataLoader batches of 512, runs encode + the L-level loop, then -- in the
concatenated / interleaved id modes the trainer uses -- runs encode + the L-level loop a SECOND time inside
`predict_tags`, and concatenates Python lists of small tensors (h_semids.py:109-195).  Here the catalogue is cut into
large chunks; per chunk one encoder pass and ONE fused L-level kernel write the ids straight into their columns of
the preallocated `cached_ids [N, L (+ L_tags)]` table, and the tag heads reuse that launch's per-level embeddings.
`shard=(rank, world)` assigns a contiguous item range to every rank; `gather_shards` is the only collective of the id table.
With `use_dedup_dim` a last column numbers the items that share a semantic-id tuple (the TIGER-style collision digit,
ops.semid_dedup); sharded, the ranks exchange only their lists of distinct tuples to make those digits global.
"""
from typing import List, Optional, Tuple

import torch
from torch import Tensor, nn

from data.schemas import SeqBatch, TokenizedSeqBatch
from hidvae_b200 import ops
from modules.h_rqvae import HRqVae
from modules.utils import eval_mode

BATCH_SIZE = 16


def _features_of(dataset, lo: int, hi: int) -> Tensor:
    """Rows [lo, hi) of the item-feature matrix of an ItemData-like dataset or of a plain [N, F] tensor."""
    if isinstance(dataset, Tensor):
        return dataset[lo:hi]
    item = dataset[lo:hi] if hasattr(dataset, "__getitem__") else None
    x = getattr(item, "x", item)
    if isinstance(x, Tensor) and x.dim() == 2 and x.shape[0] == hi - lo:
        return x
    rows = [getattr(dataset[i], "x", dataset[i]) for i in range(lo, hi)]  # datasets that only index single items
    return torch.stack([r if isinstance(r, Tensor) else torch.as_tensor(r) for r in rows])


def _column_view(rows: Tensor, cols: List[int]) -> Optional[Tensor]:
    """rows[:, cols] as a strided view when the columns are evenly spaced (the concatenated and interleaved layouts)."""
    step = cols[1] - cols[0] if len(cols) > 1 else 1
    if step < 1 or cols != list(range(cols[0], cols[0] + step * len(cols), step)):
        return None
    return rows[:, cols[0]: cols[-1] + 1: step]


class HSemanticIdTokenizer(nn.Module):
    def __init__(
        self,
        input_dim: int,
        output_dim: int,
        hidden_dims: List[int],
        codebook_size: int,
        n_layers: int = 3,
        n_cat_feats: int = 18,
        commitment_weight: float = 0.25,
        hrqvae_weights_path: Optional[str] = None,
        hrqvae_codebook_normalize: bool = False,
        hrqvae_sim_vq: bool = False,
        tag_alignment_weight: float = 0.5,
        tag_prediction_weight: float = 0.5,
        tag_class_counts: Optional[List[int]] = None,
        tag_embed_dim: int = 768,
        use_dedup_dim: bool = False,
        use_concatenated_ids: bool = False,
        use_interleaved_ids: bool = False,
        chunk_items: int = 1 << 18,
        encoder_precision: str = "fused",
        tag_precision: str = "torch",
    ) -> None:
        super().__init__()
        if sum(map(bool, (use_dedup_dim, use_concatenated_ids, use_interleaved_ids))) > 1:
            raise ValueError("use_dedup_dim, use_concatenated_ids and use_interleaved_ids are mutually exclusive")
        if use_dedup_dim and n_layers * ops.dedup_bits(codebook_size) > 63:
            raise ValueError(f"use_dedup_dim: {n_layers} levels of {codebook_size} codes do not fit an exact 63-bit tuple key")
        # The reference sets torch.set_float32_matmul_precision('high') at import (modules/h_rqvae.py:21), i.e. TF32 encoder
        # GEMMs on a GPU.  encoder_precision (modules/encoder.py): "fused" = the one-kernel tcgen05 encoder with fp16
        # operands (the same 11-bit significand, fp32 accumulation); "tf32" / "fp32" = the PyTorch layers on cuBLAS
        # ("fp32": ids match the CPU reference bit for bit outside near-ties).
        self.encoder_precision = encoder_precision
        self.hrq_vae = HRqVae(
            input_dim=input_dim, embed_dim=output_dim, hidden_dims=hidden_dims, codebook_size=codebook_size,
            codebook_kmeans_init=False, codebook_normalize=hrqvae_codebook_normalize, codebook_sim_vq=hrqvae_sim_vq,
            n_layers=n_layers, n_cat_features=n_cat_feats, commitment_weight=commitment_weight,
            tag_alignment_weight=tag_alignment_weight, tag_prediction_weight=tag_prediction_weight,
            tag_class_counts=tag_class_counts, tag_embed_dim=tag_embed_dim)
        if hrqvae_weights_path is not None:
            self.hrq_vae.load_pretrained(hrqvae_weights_path)
        self.hrq_vae.eval()
        self.hrq_vae.encoder.inference_precision = encoder_precision
        # tag_precision (HRqVae.tag_inference_precision): "torch" = the PyTorch tag heads; "fused" = the tcgen05 tag-head
        # kernels (fp16 operands, fp32 accumulation), which write the predicted tags straight into their id-table columns
        self.hrq_vae.tag_inference_precision = tag_precision
        self.codebook_size = codebook_size
        self.n_layers = n_layers
        self.use_dedup_dim = use_dedup_dim
        self.use_concatenated_ids = use_concatenated_ids
        self.use_interleaved_ids = use_interleaved_ids
        self.tag_class_counts = tag_class_counts
        self.chunk_items = chunk_items
        self.reset()

    def reset(self) -> None:
        self.cached_ids = None
        self._dedup_stats = None

    @property
    def dedup_stats(self) -> Optional[Tuple[int, int, int]]:
        """(rows, distinct semantic-id tuples, largest collision digit) over the whole catalogue after
        `precompute_corpus_ids` with `use_dedup_dim` (None otherwise).  The last id position takes largest digit + 1 values."""
        return None if self._dedup_stats is None else tuple(int(v) for v in self._dedup_stats)

    def _get_hits(self, query: Tensor, key: Tensor) -> Tensor:
        return (key.unsqueeze(0) == query.unsqueeze(1)).all(dim=-1)

    @property
    def _with_tags(self) -> bool:
        return (self.use_concatenated_ids or self.use_interleaved_ids) and self.tag_class_counts is not None

    @property
    def sem_ids_dim(self) -> int:
        if self.use_dedup_dim:
            return self.n_layers + 1
        if self._with_tags:
            return self.n_layers + len(self.tag_class_counts)
        return self.n_layers

    def _columns(self) -> Tuple[List[int], List[int]]:
        """Column of every semantic level / tag level inside one row of `cached_ids`."""
        n_sem = self.n_layers
        n_tag = self.hrq_vae.n_layers if (self.use_concatenated_ids or self.use_interleaved_ids) else 0
        if self.use_interleaved_ids:   # s1 t1 s2 t2 ... (h_semids.py:148-171)
            sem, tag, col = [], [], 0
            for i in range(max(n_sem, n_tag)):
                if i < n_sem:
                    sem.append(col); col += 1
                if i < n_tag:
                    tag.append(col); col += 1
            return sem, tag
        return list(range(n_sem)), list(range(n_sem, n_sem + n_tag))

    @torch.no_grad()
    @eval_mode
    def precompute_corpus_ids(self, movie_dataset, shard: Optional[Tuple[int, int]] = None, process_group=None) -> Tensor:
        """cached_ids [N, sem_ids_dim] int64 for the whole catalogue (or this rank's contiguous shard of it).  With
        `use_dedup_dim`, column L holds every item's collision digit over the whole catalogue in item order, also on a
        shard (the ranks of `process_group` exchange their distinct tuples), so `gather_shards` stays a concatenation."""
        model = self.hrq_vae
        dev = model.device
        n_total = movie_dataset.shape[0] if isinstance(movie_dataset, Tensor) else len(movie_dataset)
        lo_all, hi_all = 0, n_total
        if shard is not None:
            rank, world = shard
            per = (n_total + world - 1) // world
            lo_all, hi_all = min(rank * per, n_total), min((rank + 1) * per, n_total)
        sem_cols, tag_cols = self._columns()
        width = len(sem_cols) + len(tag_cols) + int(self.use_dedup_dim)
        table = torch.empty((hi_all - lo_all, width), dtype=torch.int64, device=dev)
        contiguous_sem = sem_cols == list(range(len(sem_cols)))
        codebooks = model.effective_codebooks().detach()
        packed = ops.pack_codebooks(codebooks)          # one tensor-core operand image for every chunk
        fused = model._can_fuse()
        for lo in range(lo_all, hi_all, self.chunk_items):
            hi = min(lo + self.chunk_items, hi_all)
            x = _features_of(movie_dataset, lo, hi).to(dev, non_blocking=True)
            enc = model.encode(x)
            rows = table[lo - lo_all: hi - lo_all]
            if fused:
                ids_view = rows[:, : len(sem_cols)] if contiguous_sem else None
                out = ops.rq_forward(enc, codebooks, ops.HV_MODE_STE, False, 0.0, want_emb=bool(tag_cols),
                                     ids_out=ids_view, packed=packed)
                ids, level_emb = out.ids, out.emb_out
            else:  # Gumbel / cosine configurations: level-by-level modules
                level_emb, _res, ids, _loss = model.quantize_all_levels(enc)
            if not (fused and contiguous_sem):
                rows[:, sem_cols] = ids
            if tag_cols and model.predict_tags_into(level_emb, _column_view(rows, tag_cols)):
                pass  # the fused heads wrote the tag columns in place
            elif tag_cols:
                tags = model.predict_tags(x, level_embeddings=level_emb)["predictions"]
                if tags.shape[0] != ids.shape[0]:
                    raise ValueError(f"Semantic ID batch size ({ids.shape[0]}) does not match predicted tag batch size ({tags.shape[0]})")
                rows[:, tag_cols] = tags
        if self.use_dedup_dim:
            world = shard[1] if shard is not None else 1
            self._dedup_stats = self._assign_digits(table, n_total, shard[0] if world > 1 else 0, world, process_group)
        self.cached_ids = table
        return self.cached_ids

    def _assign_digits(self, table: Tensor, n_total: int, rank: int, world: int, process_group) -> Tensor:
        """table[:, L] <- collision digits of table[:, :L], in place; returns (rows, distinct, largest digit) of the catalogue.
        Sharded: every rank sorts its shard once to get its distinct tuples, the run lists are all-gathered (16 B per
        distinct tuple of each shard), and rank r sorts again with the merged lists of ranks < r as prior counts."""
        L, bits = self.n_layers, ops.dedup_bits(self.codebook_size)
        ids, digits = table[:, :L], table[:, L]
        local = ops.semid_dedup(ids, bits, digits_out=digits)
        if world == 1:
            return torch.stack([torch.full_like(local.stats[0], n_total), local.stats[0], local.stats[1]])
        import torch.distributed as dist
        dev = table.device
        sizes = [torch.zeros(1, dtype=torch.int64, device=dev) for _ in range(world)]
        dist.all_gather(sizes, local.stats[:1].clone(), group=process_group)
        sizes = [int(v) for v in sizes]
        padded = torch.zeros((2, max(sizes)), dtype=torch.int64, device=dev)
        padded[0, : sizes[rank]] = local.run_keys[: sizes[rank]]
        padded[1, : sizes[rank]] = local.run_counts[: sizes[rank]]
        parts = [torch.empty_like(padded) for _ in range(world)]
        dist.all_gather(parts, padded, group=process_group)
        lists = [(p[0, :n], p[1, :n]) for p, n in zip(parts, sizes)]
        top = local.stats[1:2].clone()
        if rank > 0:
            top = ops.semid_dedup(ids, bits, prior=ops.merge_runs(lists[:rank]), digits_out=digits).stats[1:2].clone()
        dist.all_reduce(top, op=dist.ReduceOp.MAX, group=process_group)
        distinct = ops.merge_runs(lists)[0].numel()
        return torch.tensor([n_total, distinct, int(top)], dtype=torch.int64)

    def gather_shards(self, process_group=None) -> Tensor:
        """all_gather of every rank's shard of `cached_ids` (the only collective of bulk assignment)."""
        import torch.distributed as dist
        world = dist.get_world_size(process_group)
        sizes = [torch.zeros(1, dtype=torch.int64, device=self.cached_ids.device) for _ in range(world)]
        dist.all_gather(sizes, torch.tensor([self.cached_ids.shape[0]], device=self.cached_ids.device), group=process_group)
        longest = int(max(int(s) for s in sizes))
        padded = torch.zeros((longest, self.cached_ids.shape[1]), dtype=torch.int64, device=self.cached_ids.device)
        padded[: self.cached_ids.shape[0]] = self.cached_ids
        parts = [torch.empty_like(padded) for _ in range(world)]
        dist.all_gather(parts, padded, group=process_group)
        self.cached_ids = torch.cat([p[: int(s)] for p, s in zip(parts, sizes)])
        return self.cached_ids

    @torch.no_grad()
    @eval_mode
    def exists_prefix(self, sem_id_prefix: Tensor) -> Tensor:
        """True where a prefix [..., P] equals the first P columns of some cached row (h_semids.py:197-240).
        Sort + binary search over 64-bit row keys instead of the O(B x N x P) broadcast compare."""
        if self.cached_ids is None:
            raise Exception("No match found in empty cache.")
        p = min(sem_id_prefix.shape[-1], self.cached_ids.shape[-1])
        cache, query = self.cached_ids[:, :p], sem_id_prefix[..., :p].reshape(-1, p).to(self.cached_ids.device)
        base = int(max(int(cache.max()) if cache.numel() else 0, int(query.max()) if query.numel() else 0)) + 2
        if p * torch.log2(torch.tensor(float(base))) < 62:       # exact mixed-radix key
            weights = torch.tensor([base ** (p - 1 - i) for i in range(p)], dtype=torch.int64, device=cache.device)
            ckey, qkey = ((cache + 1) * weights).sum(-1), ((query + 1) * weights).sum(-1)
            ckey = torch.sort(ckey).values
            pos = torch.searchsorted(ckey, qkey).clamp(max=max(ckey.numel() - 1, 0))
            hit = (ckey[pos] == qkey) if ckey.numel() else torch.zeros_like(qkey, dtype=torch.bool)
        else:                                                     # very wide prefixes: chunked exact compare
            hit = torch.cat([self._get_hits(query[i:i + BATCH_SIZE], cache).any(dim=-1)
                             for i in range(0, query.shape[0], BATCH_SIZE)]) if query.shape[0] else query.new_zeros(0, dtype=torch.bool)
        return hit.reshape(sem_id_prefix.shape[:-1]).to(sem_id_prefix.device)

    # ------------------------------------------------------------------------------------------------------------
    # cached-id consumers: the wire format to stage 2 (SURVEY.md section 8f rank 2)
    # ------------------------------------------------------------------------------------------------------------
    def _tokenize_seq_batch_from_cached(self, ids: Tensor) -> Tensor:
        """ids [B, N] of items -> their cached id rows laid side by side, [B, N * sem_ids_dim] (h_semids.py:241-258).
        Ids beyond the cache read row 0, like the reference."""
        b, n = ids.shape
        rows = ids.to(self.cached_ids.device).reshape(-1)
        rows = torch.where(rows >= self.cached_ids.shape[0], torch.zeros_like(rows), rows)
        return self.cached_ids.index_select(0, rows).reshape(b, n * self.cached_ids.shape[-1])

    def _ids_of_features(self, x: Tensor) -> Tensor:
        """[M, F] item features -> [M, sem_ids_dim] id rows in the cache's column order: one encoder pass and one fused
        L-level launch; the tag heads reuse its per-level embeddings (the reference encodes and quantises twice)."""
        model = self.hrq_vae
        sem_cols, tag_cols = self._columns()
        enc = model.encode(x.to(model.device))
        level_emb, _res, ids, _loss = model.quantize_all_levels(enc)
        rows = torch.empty((x.shape[0], len(sem_cols) + len(tag_cols)), dtype=torch.int64, device=ids.device)
        rows[:, sem_cols] = ids
        if tag_cols and not model.predict_tags_into(level_emb, _column_view(rows, tag_cols)):
            rows[:, tag_cols] = model.predict_tags(x, level_embeddings=level_emb)["predictions"]
        return rows

    @torch.no_grad()
    @eval_mode
    def forward(self, batch: SeqBatch) -> TokenizedSeqBatch:
        """SeqBatch -> TokenizedSeqBatch (h_semids.py:260-451): per sequence position the item's id row (semantic ids,
        plus concatenated / interleaved predicted tag ids), masked positions -1, token type = column inside the row.
        Items of the cache are gathered; when there is no cache, or an id lies beyond it, the ids are computed from the
        batch's features (the reference's version of that branch passes a 3-D tensor to the quantiser and cannot run,
        SURVEY.md section 8f; here the sequence is flattened to rows)."""
        b, n = batch.ids.shape
        use_cache = self.cached_ids is not None and not bool((batch.ids.max() >= self.cached_ids.shape[0]).item())
        if use_cache:
            width = self.cached_ids.shape[-1]
            sem_ids = self._tokenize_seq_batch_from_cached(batch.ids)
            sem_ids_fut = self._tokenize_seq_batch_from_cached(batch.ids_fut)
        else:
            feat = batch.x.shape[-1]
            rows = self._ids_of_features(batch.x.reshape(b * n, feat))
            width = rows.shape[-1]
            sem_ids = rows.reshape(b, n * width)
            sem_ids_fut = self._ids_of_features(batch.x_fut.reshape(b, feat)) if batch.x_fut is not None else None
        seq_mask = None
        if batch.seq_mask is not None:
            seq_mask = batch.seq_mask.to(sem_ids.device).repeat_interleave(width, dim=1)
            sem_ids = sem_ids.masked_fill(~seq_mask, -1)
        types = torch.arange(width, device=sem_ids.device)
        return TokenizedSeqBatch(user_ids=batch.user_ids, sem_ids=sem_ids, sem_ids_fut=sem_ids_fut, seq_mask=seq_mask,
                                 token_type_ids=types.repeat(b, n), token_type_ids_fut=types.repeat(b, 1))
