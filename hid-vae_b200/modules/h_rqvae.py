"""HiD-VAE model with the module API of the reference's modules/h_rqvae.py -- `HRqVae` (`forward`,
`get_semantic_ids`, `encode`, `decode`, `predict_tags`, `load_pretrained`, `update_class_counts`, `config`,
`device`), `SemanticIdUniquenessLoss`, `TagPredictor` -- with the residual-quantisation hot path on the sm_100a
kernels of libhidvae_b200.so.

Where the reference loops `res -> layer(res) -> res - emb` over the levels (h_rqvae.py:515-552, ~100 small launches
per level per forward+backward), `get_semantic_ids` here runs ALL levels in one fused launch (forward) and one in
backward; the tag heads only read the per-level `emb_out`, so they run afterwards on PyTorch exactly as in the
reference (they are HiD-VAE's supervision, not part of the hot path).  The per-level path is kept for the first
call (lazy k-means init is sequential across levels, quantize.py:103-104) and for GUMBEL_SOFTMAX.

Parameter / buffer names equal the reference's (`layers.{i}.embedding.weight`, `encoder.mlp.*`,
`tag_predictors.{i}.classifier.7.weight`, ...) so `load_pretrained` reads its checkpoints.

Reference quirk kept on purpose (SURVEY.md section 0, quirk 1): `forward` hands the uniqueness loss the TRANSPOSED
id tensor [L, B] (h_rqvae.py:630-631), which makes that loss 0 in practice.  `uniqueness_as_reference = False`
switches to the intended [B, L] semantics.
"""
from functools import cached_property
from typing import Dict, List, Optional

import torch
import torch.nn.functional as F
from torch import Tensor, nn

from data.schemas import HRqVaeComputedLosses, HRqVaeOutput, SeqBatch
from hidvae_b200 import ops
from modules.encoder import MLP
from modules.loss import (CategoricalReconstructionLoss, QuantizeLoss, ReconstructionLoss,  # noqa: F401
                          TagAlignmentLoss, TagPredictionLoss)
from modules.normalize import l2norm
from modules.quantize import Quantize, QuantizeForwardMode

try:  # the reference mixes this in for push_to_hub/from_pretrained; optional here
    from huggingface_hub import PyTorchModelHubMixin as _HubMixin
except Exception:  # pragma: no cover
    class _HubMixin:  # type: ignore
        pass


class SemanticIdUniquenessLoss(nn.Module):
    """weight * mean over pairs i<j of rows with identical id tuples of relu(cos(f_i, f_j) - margin); 0 when the
    batch has fewer than two rows or no identical pair (reference h_rqvae.py:25-105).  One tiled kernel instead of
    the [B, B, L] equality tensor + torch.where host sync."""

    def __init__(self, margin: float = 0.5, weight: float = 1.0):
        super().__init__()
        self.margin = margin
        self.weight = weight

    def forward(self, sem_ids: Tensor, encoded_features: Tensor) -> Tensor:
        n_rows, _ = sem_ids.shape
        if n_rows <= 1:
            return torch.tensor(0.0, device=sem_ids.device)
        if encoded_features.shape[0] < n_rows:
            raise IndexError(f"uniqueness loss: {n_rows} id rows but only {encoded_features.shape[0]} feature rows")
        return ops.uniqueness_loss(sem_ids, encoded_features, self.margin, self.weight)


def _norm(width: int, on: bool) -> nn.Module:
    return nn.LayerNorm(width) if on else nn.Identity()


def _res_block(width: int, inner: int, p: float, norm: bool) -> nn.Sequential:
    return nn.Sequential(nn.Linear(width, inner), _norm(inner, norm), nn.ReLU(), nn.Dropout(p),
                         nn.Linear(inner, width), nn.ReLU(), nn.Dropout(p), _norm(width, norm))


class TagPredictor(nn.Module):
    """Per-level tag classifier over the concatenated code embeddings: sigmoid feature gate, projection, two
    residual MLP blocks, 3-layer classifier (architecture and sub-module names of reference h_rqvae.py:108-227)."""

    def __init__(self, embed_dim: int, num_classes: int, hidden_dim: Optional[int] = None, dropout_rate: float = 0.2,
                 use_batch_norm: bool = True, layer_idx: int = 0) -> None:
        super().__init__()
        hidden_dim = embed_dim * 2 if hidden_dim is None else hidden_dim
        p = min(0.55, dropout_rate + 0.075 * layer_idx)  # deeper levels drop more
        inner = int(hidden_dim * 0.9)
        self.attention = nn.Sequential(nn.Linear(embed_dim, embed_dim // 4), nn.ReLU(),
                                       nn.Linear(embed_dim // 4, embed_dim // 2), nn.GELU(),
                                       nn.Linear(embed_dim // 2, embed_dim), nn.Sigmoid())
        self.feature_extractor = nn.Sequential(nn.Linear(embed_dim, hidden_dim), _norm(hidden_dim, use_batch_norm),
                                               nn.ReLU(), nn.Dropout(p))
        self.residual_block1 = _res_block(hidden_dim, inner, p, use_batch_norm)
        self.residual_block2 = _res_block(hidden_dim, inner, p, use_batch_norm)
        self.classifier = nn.Sequential(nn.Linear(hidden_dim, inner), _norm(inner, use_batch_norm), nn.ReLU(), nn.Dropout(p),
                                        nn.Linear(inner, inner // 2), nn.ReLU(), nn.Dropout(p * 0.5),
                                        nn.Linear(inner // 2, num_classes))
        self.label_smoothing = 0.1 if layer_idx > 0 else 0.05
        self.apply_norm = layer_idx > 0

    def forward(self, x: Tensor) -> Tensor:
        gated = x * self.attention(x)
        if self.apply_norm:
            gated = F.normalize(gated, p=2, dim=-1)
        h = self.feature_extractor(gated)
        h = h + self.residual_block1(h)
        h = h + self.residual_block2(h)
        return self.classifier(h)


class HRqVae(nn.Module, _HubMixin):
    def __init__(
        self,
        input_dim: int,
        embed_dim: int,
        hidden_dims: List[int],
        codebook_size: int,
        codebook_kmeans_init: bool = True,
        codebook_normalize: bool = False,
        codebook_sim_vq: bool = False,
        codebook_mode: QuantizeForwardMode = QuantizeForwardMode.GUMBEL_SOFTMAX,
        n_layers: int = 3,
        commitment_weight: float = 0.25,
        n_cat_features: int = 18,
        tag_alignment_weight: float = 0.5,
        tag_prediction_weight: float = 0.5,
        tag_class_counts: Optional[List[int]] = None,
        tag_embed_dim: int = 768,
        use_focal_loss: bool = False,
        focal_loss_params: Optional[Dict] = None,
        dropout_rate: float = 0.2,
        use_batch_norm: bool = True,
        alignment_temperature: float = 0.1,
        sem_id_uniqueness_weight: float = 0.5,
        sem_id_uniqueness_margin: float = 0.5,
    ) -> None:
        self._config = {k: v for k, v in locals().items() if k not in ("self", "__class__")}
        super().__init__()

        self.input_dim = input_dim
        self.embed_dim = embed_dim
        self.hidden_dims = hidden_dims
        self.n_layers = n_layers
        self.codebook_size = codebook_size
        self.commitment_weight = commitment_weight
        self.n_cat_feats = n_cat_features
        self.tag_alignment_weight = tag_alignment_weight
        self.tag_prediction_weight = tag_prediction_weight
        self.tag_embed_dim = tag_embed_dim
        self.use_focal_loss = use_focal_loss
        self.focal_loss_params = focal_loss_params or {"gamma": 2.0}
        self.dropout_rate = dropout_rate
        self.use_batch_norm = use_batch_norm
        self.alignment_temperature = alignment_temperature
        self.sem_id_uniqueness_weight = sem_id_uniqueness_weight
        self.uniqueness_as_reference = True   # transposed-ids call of h_rqvae.py:630-631 (see module docstring)
        self.fuse_levels = True               # False forces the reference's level-by-level loop
        # "torch": predict_tags runs the PyTorch heads; "fused": eval-mode, no-grad CUDA calls of a served shape run the
        # tcgen05 tag-head kernels (csrc/tag_heads.cu: fp16 operands, fp32 accumulation); training always uses PyTorch
        self.tag_inference_precision = "torch"
        self._tag_image, self._tag_image_key = None, None

        self.tag_class_counts = ([10, 100, 1000] if tag_class_counts is None else list(tag_class_counts))[:n_layers]
        assert len(self.tag_class_counts) == n_layers, (
            f"Number of tag classes {len(self.tag_class_counts)} does not match number of layers {n_layers}")

        self.layers = nn.ModuleList([
            Quantize(embed_dim=embed_dim, n_embed=codebook_size, forward_mode=codebook_mode,
                     do_kmeans_init=codebook_kmeans_init, codebook_normalize=(i == 0 and codebook_normalize),
                     sim_vq=codebook_sim_vq, commitment_weight=commitment_weight)
            for i in range(n_layers)])

        self.concat_embed_dims = [embed_dim * (i + 1) for i in range(n_layers)]
        self._stored_tag_class_counts = None
        self.tag_predictors = self._make_tag_predictors(hidden_dims[0], dropout_rate, use_batch_norm)
        self.tag_projectors = self._make_tag_projectors(hidden_dims[0], dropout_rate, use_batch_norm, codebook_normalize)

        self.encoder = MLP(input_dim=input_dim, hidden_dims=hidden_dims, out_dim=embed_dim, normalize=codebook_normalize)
        self.decoder = MLP(input_dim=embed_dim, hidden_dims=hidden_dims[-1::-1], out_dim=input_dim, normalize=True)

        self.reconstruction_loss = (CategoricalReconstructionLoss(n_cat_features) if n_cat_features != 0
                                    else ReconstructionLoss())
        self.tag_alignment_loss = TagAlignmentLoss(alignment_weight=tag_alignment_weight, temperature=alignment_temperature)
        self.tag_prediction_loss = TagPredictionLoss(use_focal_loss=use_focal_loss, focal_params=focal_loss_params,
                                                     class_counts=None)
        self.sem_id_uniqueness_loss = SemanticIdUniquenessLoss(margin=sem_id_uniqueness_margin,
                                                               weight=sem_id_uniqueness_weight)
        self.register_buffer("class_freq_counts", None)

    # ---- builders -----------------------------------------------------------------------------------------------
    def _make_tag_predictors(self, first_hidden: int, dropout_rate: float, use_batch_norm: bool) -> nn.ModuleList:
        return nn.ModuleList([
            TagPredictor(embed_dim=self.concat_embed_dims[i], num_classes=self.tag_class_counts[i],
                         hidden_dim=first_hidden // 2 * (i + 1), dropout_rate=dropout_rate,
                         use_batch_norm=use_batch_norm, layer_idx=i)
            for i in range(self.n_layers)])

    def _make_tag_projectors(self, first_hidden: int, dropout_rate: float, use_batch_norm: bool,
                             layer_norm_tail: bool) -> nn.ModuleList:
        return nn.ModuleList([
            nn.Sequential(nn.Linear(self.tag_embed_dim, first_hidden),
                          nn.BatchNorm1d(first_hidden) if use_batch_norm else nn.Identity(),
                          nn.ReLU(), nn.Dropout(dropout_rate),
                          nn.Linear(first_hidden, self.concat_embed_dims[i]),
                          nn.LayerNorm(self.concat_embed_dims[i]) if layer_norm_tail else nn.Identity())
            for i in range(self.n_layers)])

    # ---- small API ----------------------------------------------------------------------------------------------
    @cached_property
    def config(self) -> dict:
        return self._config

    @property
    def device(self) -> torch.device:
        return next(self.encoder.parameters()).device

    def encode(self, x: Tensor) -> Tensor:
        # fp16 items (a catalogue stored in half precision) go to the fused encoder as they are; everything else is fp32
        if x.dtype == torch.float16 and getattr(self.encoder, "inference_precision", None) == "fused" and self.encoder.fused_available(x):
            return self.encoder(x)
        return self.encoder(x.float())

    def decode(self, x: Tensor) -> Tensor:
        return self.decoder(x)

    def update_class_counts(self, class_counts_dict) -> None:
        for layer_idx, counts in class_counts_dict.items():
            if not isinstance(counts, Tensor):
                counts = torch.tensor(counts, device=self.device)
            self.register_buffer(f"class_freq_counts_{layer_idx}", counts)
        self.class_freq_layers = list(class_counts_dict.keys())

    def load_pretrained(self, path: str) -> None:
        """Load a reference-format checkpoint ({'model': state_dict, 'iter': ...}); tag heads are rebuilt when the
        checkpoint's class counts / projector tail differ from this model (reference h_rqvae.py:382-471)."""
        state = torch.load(path, map_location=self.device, weights_only=False)
        saved = state["model"]
        own = self.state_dict()

        counts_in_file, resized = [], False
        for i in range(self.n_layers):
            key = f"tag_predictors.{i}.classifier.7.weight"
            if key in saved and key in own and saved[key].shape[0] != own[key].shape[0]:
                counts_in_file.append(saved[key].shape[0])
                resized = True
            else:
                counts_in_file.append(self.tag_class_counts[i])
        cfg = self._config
        first_hidden = cfg.get("hidden_dims", [512, 256, 128])[0]
        if resized:
            print(f"Tag predictor mismatch detected. Adjusting number of classes from {self.tag_class_counts} to {counts_in_file}")
            self._stored_tag_class_counts = self.tag_class_counts
            self.tag_class_counts = counts_in_file
            self.tag_predictors = self._make_tag_predictors(first_hidden, cfg.get("dropout_rate", 0.2),
                                                            cfg.get("use_batch_norm", True)).to(self.device)
        extra_tail = any(f"tag_projectors.{i}.5.weight" in saved and f"tag_projectors.{i}.5.weight" not in own
                         for i in range(self.n_layers))
        if extra_tail:
            print("Tag projector mismatch detected. Adjusting structure to match the weight file.")
            self.tag_projectors = self._make_tag_projectors(first_hidden, cfg.get("dropout_rate", 0.2),
                                                            cfg.get("use_batch_norm", True), True).to(self.device)
        own = self.state_dict()
        usable = {k: v for k, v in saved.items() if k in own}
        if len(usable) < len(saved):
            print(f"Warning: keys skipped (absent from the current model): {sorted(set(saved) - set(usable))}")
        try:
            own.update(usable)
            self.load_state_dict(own)
            print(f"---Loaded HRQVAE Iter {state['iter']}---")
        except Exception as e:
            print(f"Standard loading failed, trying to load with strict=False: {e}")
            self.load_state_dict(saved, strict=False)
            print(f"---Loaded HRQVAE Iter {state['iter']} (strict=False)---")
        for layer in self.layers:
            layer.kmeans_initted = True  # a loaded codebook must not be overwritten by a lazy k-means

    # ---- the hot path -------------------------------------------------------------------------------------------
    def _can_fuse(self) -> bool:
        """All L levels in one launch: L2 distance, no pending k-means init, and STE / rotation trick -- or eval mode,
        whose semantics do not depend on the forward mode (emb_out = codebook[ids], quantize.py:146-148)."""
        from modules.quantize import QuantizeDistance
        return self.fuse_levels and all(
            (layer.fused or (not self.training and layer.distance_mode == QuantizeDistance.L2)) and not layer.needs_kmeans()
            for layer in self.layers)

    def effective_codebooks(self) -> Tensor:
        """[L, K, D] stack of out_proj(embedding.weight) (autograd-tracked)."""
        return torch.stack([layer.effective_codebook() for layer in self.layers])

    def quantize_all_levels(self, encoded_x: Tensor, gumbel_t: float = 0.001, want_residuals: bool = True):
        """All L levels -> (emb_out [L, N, D], residuals [L, N, D], ids [N, L], loss [N]).  One fused launch when
        possible, otherwise the level-by-level loop of the reference (first call with k-means init, Gumbel).
        `want_residuals=False` (the training step: HRqVae.forward never reads them) skips writing [L, N, D]."""
        if self._can_fuse():
            mode = self.layers[0].forward_mode.value if self.layers[0].fused else QuantizeForwardMode.STE.value
            emb, res, ids, loss, _ll = ops.rq_apply(encoded_x, self.effective_codebooks(), mode, self.training,
                                                    self.commitment_weight, algo=self.layers[0].algo,
                                                    want_residuals=want_residuals, want_level_loss=False)
            if self.training and mode == QuantizeForwardMode.ROTATION_TRICK.value and encoded_x.shape[0] == 1:
                pass  # shapes stay [L, 1, D]; the per-level API reproduces the reference's squeeze, the fused one does not
            return emb, res, ids, loss
        res = encoded_x
        embs, residuals, ids = [], [], []
        loss = torch.zeros((), device=encoded_x.device)
        for layer in self.layers:
            residuals.append(res)
            q = layer(res, temperature=gumbel_t)
            loss = loss + q.loss
            e = q.embeddings if q.embeddings.dim() == 2 else q.embeddings.unsqueeze(0)  # N == 1 rotation squeeze
            embs.append(e)
            ids.append(q.ids)
            res = res - e
        return torch.stack(embs), torch.stack(residuals), torch.stack(ids, dim=1), loss

    def get_semantic_ids(self, encoded_x: Tensor, tags_emb: Optional[Tensor] = None,
                         tags_indices: Optional[Tensor] = None, gumbel_t: float = 0.001,
                         _want_residuals: bool = True) -> HRqVaeOutput:
        dev = encoded_x.device
        emb, residuals, sem_ids, quantize_loss = self.quantize_all_levels(encoded_x, gumbel_t, want_residuals=_want_residuals)

        zero = lambda: torch.zeros((), device=dev)
        align_total, pred_total, acc_total = zero(), zero(), zero()
        align_by_layer, pred_by_layer, acc_by_layer = [], [], []
        have_tags = tags_emb is not None and tags_indices is not None
        if have_tags:
            for i in range(self.n_layers):
                concat = torch.cat(list(emb[: i + 1]), dim=-1)           # [N, (i+1) D]
                projected = self.tag_projectors[i](tags_emb[:, i])
                align = self.tag_alignment_loss(concat, projected, i).mean()
                pred, acc = self.tag_prediction_loss(self.tag_predictors[i](concat), tags_indices[:, i])
                align_total, pred_total, acc_total = align_total + align, pred_total + pred, acc_total + acc
                align_by_layer.append(align), pred_by_layer.append(pred), acc_by_layer.append(acc)
            align_total, pred_total, acc_total = (v / self.n_layers for v in (align_total, pred_total, acc_total))
        stack = lambda xs: torch.stack(xs) if xs else (None if have_tags else [])

        return HRqVaeOutput(
            embeddings=emb.permute(1, 2, 0),          # [N, D, L] like rearrange(embs, "b h d -> h d b")
            residuals=residuals.permute(1, 2, 0) if residuals is not None else None,
            sem_ids=sem_ids,                          # [N, L]
            quantize_loss=quantize_loss,
            tag_align_loss=align_total,
            tag_pred_loss=pred_total,
            tag_pred_accuracy=acc_total,
            tag_align_loss_by_layer=stack(align_by_layer),
            tag_pred_loss_by_layer=stack(pred_by_layer),
            tag_pred_accuracy_by_layer=stack(acc_by_layer),
        )

    def forward(self, batch: SeqBatch, gumbel_t: float = 1.0) -> HRqVaeComputedLosses:
        x = batch.x.float()
        tags_emb = getattr(batch, "tags_emb", None)
        tags_indices = getattr(batch, "tags_indices", None)
        if tags_emb is not None:
            tags_emb = tags_emb.float()

        encoded = self.encode(x)
        q = self.get_semantic_ids(encoded, tags_emb, tags_indices, gumbel_t, _want_residuals=False)  # (:604 reads, never uses them)

        x_hat = self.decode(q.embeddings.sum(dim=-1))
        # reference :610 -- with n_cat_feats == 0 the slices are [:-0] (empty) and [-0:] (everything): identity
        c = self.n_cat_feats
        x_hat = torch.cat([l2norm(x_hat[..., :-c]), x_hat[..., -c:]], dim=-1)
        reconstruction = self.reconstruction_loss(x_hat, x)

        ids_for_loss = q.sem_ids.transpose(0, 1) if self.uniqueness_as_reference else q.sem_ids
        uniqueness = self.sem_id_uniqueness_loss(ids_for_loss, encoded)

        loss = (reconstruction.mean() + q.quantize_loss.mean()
                + self.tag_alignment_weight * q.tag_align_loss
                + self.tag_prediction_weight * q.tag_pred_loss
                + self.sem_id_uniqueness_weight * uniqueness)

        with torch.no_grad():
            embs_norm = q.embeddings.norm(dim=1)                                      # [N, L]
            n_rows = q.sem_ids.shape[0]
            later_twins = ops.count_rows_with_later_twin(q.sem_ids)
            p_unique_ids = ((n_rows - later_twins) / n_rows).to(torch.float32)        # reference :645-648

        return HRqVaeComputedLosses(
            loss=loss, reconstruction_loss=reconstruction, rqvae_loss=q.quantize_loss,
            tag_align_loss=q.tag_align_loss, tag_pred_loss=q.tag_pred_loss, tag_pred_accuracy=q.tag_pred_accuracy,
            embs_norm=embs_norm, p_unique_ids=p_unique_ids,
            tag_align_loss_by_layer=q.tag_align_loss_by_layer, tag_pred_loss_by_layer=q.tag_pred_loss_by_layer,
            tag_pred_accuracy_by_layer=q.tag_pred_accuracy_by_layer, sem_id_uniqueness_loss=uniqueness)

    def _tag_heads_shape(self):
        """(d, first_hidden, class_counts, use_norm) when the heads have the architecture the fused kernels compute."""
        first_hidden, counts, norms = self.hidden_dims[0], [], []
        for i, tp in enumerate(self.tag_predictors):
            fe, cl = tp.feature_extractor, tp.classifier
            lns = [m for m in tp.modules() if isinstance(m, nn.LayerNorm)]
            if (tp.attention[0].in_features != self.embed_dim * (i + 1) or fe[0].out_features != first_hidden // 2 * (i + 1)
                    or tp.apply_norm != (i > 0) or any(m.eps != 1e-5 or not m.elementwise_affine for m in lns)):
                return None
            norms.append(isinstance(fe[1], nn.LayerNorm))
            counts.append(cl[-1].out_features)
        if len(set(norms)) != 1 or not ops.tag_heads_supported(self.n_layers, self.embed_dim, first_hidden, counts, norms[0]):
            return None
        return self.embed_dim, first_hidden, counts, norms[0]

    def _fused_tag_image(self, level_embeddings: Tensor):
        """The packed tag-head image when this call takes the fused path, else None.  Re-packed whenever a weight
        changed (version counters), like MLP._weight_image."""
        if self.tag_inference_precision not in ("torch", "fused"):
            raise ValueError(f"tag_inference_precision must be 'torch' or 'fused', got {self.tag_inference_precision!r}")
        if (self.tag_inference_precision != "fused" or not level_embeddings.is_cuda or torch.is_grad_enabled()
                or any(m.training for m in self.tag_predictors.modules())):
            return None
        shape = self._tag_heads_shape()
        if shape is None:
            return None
        params = [p for tp in self.tag_predictors for p in tp.parameters()]
        key = (tuple(shape[2]), shape[3], tuple((p.data_ptr(), p._version) for p in params))
        if self._tag_image is None or key != self._tag_image_key:
            self._tag_image, self._tag_image_key = ops.tag_heads_pack(params, *shape), key
        return self._tag_image

    def predict_tags_into(self, level_embeddings: Tensor, pred_out: Optional[Tensor],
                          conf_out: Optional[Tensor] = None) -> bool:
        """Fused path only: write the predicted tags of level_embeddings [L, N, D] into pred_out [N, L] int64 (any
        strides, e.g. the tag columns of an id table) and return True; False (nothing written) when the call does not
        take the fused path."""
        if pred_out is None:
            return False
        image = self._fused_tag_image(level_embeddings)
        if image is None:
            return False
        emb = level_embeddings.float()
        ops.tag_heads_forward(emb if emb.stride(-1) == 1 else emb.contiguous(), image, pred_out, conf_out)
        return True

    def predict_tags(self, x: Tensor, gumbel_t: float = 0.001, encoded: Optional[Tensor] = None,
                     level_embeddings: Optional[Tensor] = None) -> Dict[str, Tensor]:
        """Tag ids + confidences per level for x [B, F] or [B, S, F] (reference h_rqvae.py:674-738).  Passing
        `level_embeddings` [L, N, D] from an earlier `quantize_all_levels` call skips the second encode + RQ pass the
        reference's tokenizer pays per item (SURVEY.md section 8f rank 1)."""
        shape = x.shape
        seq = len(shape) == 3
        if seq:
            x = x.reshape(-1, shape[-1])
        if level_embeddings is None:
            enc = self.encode(x) if encoded is None else encoded
            level_embeddings, _res, _ids, _loss = self.quantize_all_levels(enc, gumbel_t)
        if self._fused_tag_image(level_embeddings) is not None:
            n = level_embeddings.shape[1]
            pred = torch.empty((n, self.n_layers), dtype=torch.int64, device=level_embeddings.device)
            conf = torch.empty((n, self.n_layers), dtype=torch.float32, device=level_embeddings.device)
            self.predict_tags_into(level_embeddings, pred, conf)
            if seq:
                pred, conf = pred.reshape(shape[0], shape[1], -1), conf.reshape(shape[0], shape[1], -1)
            return {"predictions": pred, "confidences": conf}
        preds, confs = [], []
        for i in range(self.n_layers):
            concat = torch.cat(list(level_embeddings[: i + 1]), dim=-1)
            conf, pred = torch.softmax(self.tag_predictors[i](concat), dim=-1).max(dim=-1)
            preds.append(pred), confs.append(conf)
        if seq:
            preds = [p.reshape(shape[0], shape[1]) for p in preds]
            confs = [c.reshape(shape[0], shape[1]) for c in confs]
        return {"predictions": torch.stack(preds, dim=-1), "confidences": torch.stack(confs, dim=-1)}
