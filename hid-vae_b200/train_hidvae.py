"""gin-configurable HiD-VAE (stage 1) trainer with the parameter names of the reference's train_hidvae.py:65-135,
so `python train_hidvae.py configs/h_rqvae_amazon.gin` keeps working with the reference's own .gin files.

    python train_hidvae.py configs/h_rqvae_amazon.gin
    torchrun --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 train_hidvae.py configs/h_rqvae_kuairand.gin

What is the same: the model, AdamW (optionally with the per-component parameter groups), cosine / step LR schedule,
gradient accumulation, iteration-0 k-means codebook init on min(20000, N) items, evaluation every `eval_every`
iterations (eval losses, corpus semantic ids, entropy / codebook usage / repetition rate) and the checkpoint gate
(eval tag accuracy > 0.60 and id repetition rate < threshold) with the reference's checkpoint keys.

What is B200-native: the residual quantiser runs on the fused sm_100a kernels; data parallelism is one process per
GPU over torch.distributed/NCCL with ONE flat-buffer gradient all-reduce per step instead of Accelerate/DDP buckets
and two barriers (train_hidvae.py:709, 760, 768); k-means init is a dedicated encode -> per-level k-means pass whose
centroids are identical on every rank; losses are accumulated on the device and read back only when a log line is
printed (the reference issues six .cpu().item() syncs per iteration, :711-717); the catalogue lives in HBM.
"""
import logging
import os
import sys
import time
from datetime import datetime

import numpy as np
import torch
from torch.optim import AdamW, lr_scheduler

HERE = os.path.dirname(os.path.abspath(__file__))
if HERE not in sys.path:
    sys.path.insert(0, HERE)

from data.tags_processed import ItemData, RecDataset  # noqa: E402
from hidvae_b200 import dist as hv_dist  # noqa: E402
from hidvae_b200 import gin_lite  # noqa: E402
from hidvae_b200.graph_step import GraphedTrainStep, step_statistics  # noqa: E402
from modules.h_rqvae import HRqVae  # noqa: E402
from modules.quantize import QuantizeForwardMode  # noqa: E402
from modules.tokenizer.h_semids import HSemanticIdTokenizer  # noqa: E402
from modules.utils import parse_config  # noqa: E402


def calculate_repetition_rate(item_ids: torch.Tensor):
    """1 - (#distinct id rows / #rows) (reference train_hidvae.py:38-63)."""
    total = item_ids.shape[0]
    if total == 0:
        return 0.0, 0, 0
    unique = torch.unique(item_ids, dim=0).shape[0]
    return 1.0 - unique / total, unique, total


def tag_class_statistics(dataset: ItemData, n_layers: int, tag_class_counts, rare_tag_threshold: int, device):
    """Per-level class frequencies for the focal-loss class weights (reference :359-491, minus the rare-tag remap
    of real vocabularies, which needs the raw tag strings)."""
    out = {}
    if not getattr(dataset, "has_tags", False):
        return out
    for i in range(n_layers):
        idx = dataset.tags_indices[:, i]
        out[i] = torch.bincount(idx[idx >= 0], minlength=tag_class_counts[i]).to(device)
    return out


@torch.no_grad()
def init_codebooks(model: HRqVae, x: torch.Tensor, process_group=None) -> None:
    """Iteration-0 codebook init.  The reference triggers the lazy k-means of every level with a whole training-mode
    model forward on up to 20000 items (train_hidvae.py:692-694), paying tag heads and [B, B] temporaries for
    nothing; here: encode, then level by level k-means on the level's input and the training-mode residual update."""
    was_training = model.training
    model.train()
    for layer in model.layers:
        layer.kmeans_process_group = process_group
    model.get_semantic_ids(model.encode(x))      # per-level path: every Quantize runs its k-means on first use
    model.train(was_training)


@gin_lite.configurable
def train(
    iterations=50000,
    batch_size=64,
    learning_rate=0.0001,
    weight_decay=0.01,
    dataset_folder="dataset/ml-1m",
    dataset=RecDataset.ML_1M,
    pretrained_hrqvae_path=None,
    save_dir_root="out/",
    use_kmeans_init=True,
    split_batches=True,
    amp=False,
    do_eval=True,
    force_dataset_process=False,
    mixed_precision_type="fp16",
    gradient_accumulate_every=1,
    save_model_every=1000,
    eval_every=5000,
    commitment_weight=0.25,
    tag_alignment_weight=0.5,
    tag_prediction_weight=0.5,
    vae_n_cat_feats=18,
    vae_input_dim=768,
    vae_embed_dim=128,
    vae_hidden_dims=[512, 256],
    vae_codebook_size=512,
    vae_codebook_normalize=False,
    vae_codebook_mode=QuantizeForwardMode.GUMBEL_SOFTMAX,
    vae_sim_vq=False,
    vae_n_layers=3,
    dataset_split="beauty",
    tag_class_counts=None,
    tag_embed_dim=768,
    use_focal_loss=True,
    focal_loss_gamma_base=2.0,
    focal_loss_alpha_base=0.25,
    rare_tag_threshold=30,
    dropout_rate=0.3,
    use_batch_norm=True,
    alignment_temperature=0.1,
    predictor_weight_decay=0.02,
    layer_specific_lr=False,
    use_label_smoothing=True,
    label_smoothing_alpha=0.1,
    use_mixup=True,
    mixup_alpha=0.2,
    eval_tta=True,
    eval_temperature=0.8,
    ensemble_predictions=True,
    use_lr_scheduler=True,
    lr_scheduler_type="cosine",
    lr_scheduler_T_max=400000,
    lr_scheduler_eta_min=1e-7,
    lr_scheduler_step_size=100000,
    lr_scheduler_gamma=0.5,
    lr_scheduler_factor=0.5,
    lr_scheduler_patience=10,
    sem_id_uniqueness_weight=0.5,
    sem_id_uniqueness_margin=0.5,
    id_repetition_threshold=0.03,
    use_concatenated_ids: bool = True,
    use_interleaved_ids: bool = False,
    # -- additions (not in the reference): all optional ---------------------------------------------------------
    log_every=100,
    synthetic_items=None,      # opt in to a seeded synthetic catalogue of this many items
    synthetic_data=None,       # True: opt in to the synthetic catalogue at the dataset's own size; a missing
                               # `<dataset_folder>/processed/items.pt` raises unless one of the two is given
    seed=0,
    uniqueness_as_reference=True,
    use_cuda_graph=False,      # replay the micro-step (gather + forward + backward) and the AdamW step as CUDA graphs
                               # (hidvae_b200/graph_step.py); not with fp16 loss scaling
    tag_precision="torch",     # tag heads of the eval catalogue pass: "torch" (the PyTorch heads) or "fused"
                               # (the tcgen05 kernels of csrc/tag_heads.cu, HRqVae.tag_inference_precision)
):
    rank, world, local = hv_dist.init_from_env()
    is_main = rank == 0
    assert torch.cuda.is_available(), "train_hidvae.py needs a CUDA device (hidvae_b200 has no CPU fallback)"
    # The reference trains with TF32 matmuls: it sets torch.set_float32_matmul_precision('high') when modules/h_rqvae.py is
    # imported (:21).  Here the setting is scoped to the training run instead of being an import side effect.
    matmul_precision_before = torch.get_float32_matmul_precision()
    torch.set_float32_matmul_precision("high")
    try:
        torch.cuda.set_device(local)
        device = torch.device("cuda", local)
        torch.manual_seed(seed + rank)
        np.random.seed(seed)                 # k-means initial rows are drawn on rank 0 from NumPy's global RNG

        save_dir = os.path.join(save_dir_root, f"hrqvae_{dataset.name}_{datetime.now().strftime('%Y%m%d_%H%M%S')}")
        logger = logging.getLogger("hrqvae_training")
        if is_main and not logger.handlers:
            os.makedirs(os.path.join(save_dir, "log"), exist_ok=True)
            logging.basicConfig(level=logging.INFO, format="%(asctime)s - %(levelname)s - %(message)s",
                                handlers=[logging.FileHandler(os.path.join(save_dir, "log", "hrqvae_training.log")),
                                          logging.StreamHandler()])
        if is_main:
            logger.info("Training parameters: %s", {k: v for k, v in locals().items() if k not in ("logger",)})

        data_kw = dict(root=dataset_folder, dataset=dataset, force_process=force_dataset_process, n_items=synthetic_items,
                       input_dim=vae_input_dim, tag_embed_dim=tag_embed_dim, tag_class_counts=tag_class_counts, device=device,
                       synthetic=synthetic_data)
        train_dataset = ItemData(train_test_split="train" if do_eval else "all", **data_kw)
        eval_dataset = ItemData(train_test_split="eval", **data_kw) if do_eval else None
        index_dataset = ItemData(train_test_split="all", **data_kw) if do_eval else train_dataset
        n_train = len(train_dataset)
        if is_main and train_dataset.synthetic:
            logger.warning("=" * 100)
            logger.warning("TRAINING ON A SEEDED SYNTHETIC CATALOGUE (%d items): no processed dataset was loaded from %s. "
                           "Losses, accuracies and checkpoints of this run say nothing about the real data.", n_train, dataset_folder)
            logger.warning("=" * 100)

        has_tags = getattr(train_dataset, "has_tags", False)
        if not has_tags:
            logger.warning("Dataset does not contain tag information. Disabling tag alignment and prediction.")
            tag_alignment_weight = tag_prediction_weight = 0.0
        if tag_class_counts is None and has_tags:
            tag_class_counts = [int(train_dataset.tags_indices[:, i].max()) + 1 for i in range(vae_n_layers)]

        focal_loss_params = {"gamma": focal_loss_gamma_base, "alpha": focal_loss_alpha_base} if use_focal_loss else None
        model = HRqVae(
            input_dim=vae_input_dim, embed_dim=vae_embed_dim, hidden_dims=vae_hidden_dims, codebook_size=vae_codebook_size,
            codebook_kmeans_init=use_kmeans_init and pretrained_hrqvae_path is None, codebook_normalize=vae_codebook_normalize,
            codebook_sim_vq=vae_sim_vq, codebook_mode=vae_codebook_mode, n_layers=vae_n_layers, n_cat_features=vae_n_cat_feats,
            commitment_weight=commitment_weight, tag_alignment_weight=tag_alignment_weight,
            tag_prediction_weight=tag_prediction_weight, tag_class_counts=tag_class_counts, tag_embed_dim=tag_embed_dim,
            use_focal_loss=use_focal_loss, focal_loss_params=focal_loss_params, dropout_rate=dropout_rate,
            use_batch_norm=use_batch_norm, alignment_temperature=alignment_temperature,
            sem_id_uniqueness_weight=sem_id_uniqueness_weight, sem_id_uniqueness_margin=sem_id_uniqueness_margin).to(device)
        model.uniqueness_as_reference = uniqueness_as_reference
        if use_focal_loss and has_tags:
            model.update_class_counts(tag_class_statistics(train_dataset, vae_n_layers, model.tag_class_counts,
                                                           rare_tag_threshold, device))
        tpl = model.tag_prediction_loss
        tpl.use_label_smoothing, tpl.label_smoothing_alpha = use_label_smoothing, label_smoothing_alpha
        tpl.use_mixup, tpl.mixup_alpha = use_mixup, mixup_alpha

        if layer_specific_lr:
            groups = [dict(params=list(model.encoder.parameters()) + list(model.decoder.parameters()), lr=learning_rate,
                           weight_decay=weight_decay),
                      dict(params=[p for layer in model.layers for p in layer.parameters()], lr=learning_rate,
                           weight_decay=weight_decay)]
            for i in range(vae_n_layers):
                lr_i = learning_rate * (1 + 0.1 * i)
                wd_i = predictor_weight_decay / (1 + 0.2 * i) if predictor_weight_decay > 0 else predictor_weight_decay
                groups.append(dict(params=list(model.tag_predictors[i].parameters()), lr=lr_i, weight_decay=wd_i))
                groups.append(dict(params=list(model.tag_projectors[i].parameters()), lr=lr_i, weight_decay=wd_i))
            optimizer = AdamW(groups, capturable=bool(use_cuda_graph), fused=True)
        else:
            # fused=True: one multi-tensor kernel per step instead of ~a dozen foreach passes (1.3 ms -> 0.05 ms at 7.2 M parameters)
            optimizer = AdamW(params=model.parameters(), lr=learning_rate, weight_decay=weight_decay, capturable=bool(use_cuda_graph),
                              fused=True)
        if use_cuda_graph:
            if bool(amp) and mixed_precision_type == "fp16":
                raise ValueError("train.use_cuda_graph: fp16 loss scaling reads its inf check back to the host; use bf16 or amp=False")
            for g_ in optimizer.param_groups:      # the graph reads the learning rate from device memory: the scheduler updates it in place
                g_["lr"] = torch.tensor(float(g_["lr"]), device=device)

        start_iter = 0
        if pretrained_hrqvae_path is not None:
            model.load_pretrained(pretrained_hrqvae_path)
            state = torch.load(pretrained_hrqvae_path, map_location=device, weights_only=False)
            optimizer.load_state_dict(state["optimizer"])
            start_iter = state["iter"] + 1

        if not has_tags:
            # no tag supervision: the tag heads receive no gradient.  The reference's optimizer skips parameters whose grad is
            # None; freezing them keeps them out of the flat gradient buffer, so AdamW applies no weight decay to them either.
            for p in list(model.tag_predictors.parameters()) + list(model.tag_projectors.parameters()):
                p.requires_grad_(False)
        hv_dist.broadcast_parameters(model)                       # what DDP does in accelerator.prepare (:630)
        grads = hv_dist.FlatGradAllReduce(model.parameters())     # one flat buffer, one collective per step
        # Batch-size semantics: every rank draws `batch_size` items per micro-step (global batch = world * batch_size), which
        # is what the reference does in effect -- its dataloader is wrapped in cycle() before accelerator.prepare, so
        # `split_batches` cannot shard it (SURVEY.md section 2.3).  `split_batches` is accepted and ignored for that reason.
        # fp16 autocast needs loss scaling (Accelerate(mixed_precision="fp16") applies a GradScaler, train_hidvae.py:186-189)
        use_fp16 = bool(amp) and mixed_precision_type == "fp16"
        scaler = torch.amp.GradScaler("cuda", enabled=use_fp16)

        scheduler = None
        if use_lr_scheduler:
            last = start_iter - 1 if start_iter > 0 else -1
            if last >= 0:
                for g in optimizer.param_groups:
                    g.setdefault("initial_lr", g["lr"])
            if lr_scheduler_type == "cosine":
                scheduler = lr_scheduler.CosineAnnealingLR(optimizer, T_max=lr_scheduler_T_max, eta_min=lr_scheduler_eta_min,
                                                           last_epoch=last)
            elif lr_scheduler_type == "step":
                scheduler = lr_scheduler.StepLR(optimizer, step_size=lr_scheduler_step_size, gamma=lr_scheduler_gamma,
                                                last_epoch=last)
            elif is_main:
                logger.warning(f"Unsupported learning rate scheduler type: {lr_scheduler_type}. Not using a scheduler.")

        tokenizer = HSemanticIdTokenizer(
            input_dim=vae_input_dim, output_dim=vae_embed_dim, hidden_dims=vae_hidden_dims, codebook_size=vae_codebook_size,
            n_layers=vae_n_layers, n_cat_feats=vae_n_cat_feats, hrqvae_weights_path=None,
            hrqvae_codebook_normalize=vae_codebook_normalize, hrqvae_sim_vq=vae_sim_vq,
            tag_alignment_weight=tag_alignment_weight, tag_prediction_weight=tag_prediction_weight,
            tag_class_counts=model.tag_class_counts, tag_embed_dim=tag_embed_dim,
            use_concatenated_ids=use_concatenated_ids, use_interleaved_ids=use_interleaved_ids,
            commitment_weight=commitment_weight, tag_precision=tag_precision)
        tokenizer.hrq_vae = model
        model.tag_inference_precision = tag_precision

        # running sums of the logged quantities live on the device; .tolist() happens only when a line is printed
        names = ["loss", "reconstruction", "rqvae", "tag_align", "tag_pred", "tag_acc", "p_unique"]
        acc = torch.zeros(len(names), device=device)
        acc_n = 0
        gen = torch.Generator(device=device).manual_seed(seed * 1000 + rank)   # every rank draws its own batches (:213,233)
        t = 0.2                                                                # hard-coded in the reference (:690)
        history = []
        t_start = time.time()
        best_eval_accuracy = 0.0

        graphed = None
        for it in range(start_iter, start_iter + 1 + iterations):
            model.train()
            if it == 0 and use_kmeans_init and pretrained_hrqvae_path is None:
                n_init = min(20000, n_train)                          # (train_hidvae.py:693); every rank contributes its share
                lo_i, hi_i = hv_dist.shard_range(n_init, rank, world)
                init_codebooks(model, train_dataset[torch.arange(lo_i, hi_i, device=device)].x.float(),
                               process_group=torch.distributed.group.WORLD if world > 1 else None)
                if is_main:
                    logger.info("K-means initialization complete")

            if use_cuda_graph and graphed is None:
                # captured after the k-means init (it runs inside the first forward otherwise) on this rank's own sampler
                graphed = GraphedTrainStep(model, optimizer, grads, train_dataset.__getitem__, batch_size, n_train, gumbel_t=t,
                                           loss_divisor=gradient_accumulate_every,
                                           autocast_dtype=torch.bfloat16 if bool(amp) else None, generator=gen)
            grads.zero()
            if graphed is not None:
                for _ in range(gradient_accumulate_every):
                    stats = graphed.micro_step()
                grads.all_reduce()
                graphed.optimizer_step()
                norms_dev = graphed.emb_norms
            else:
                out = None
                for _ in range(gradient_accumulate_every):
                    batch = train_dataset[torch.randint(0, n_train, (batch_size,), device=device, generator=gen)]
                    with torch.autocast("cuda", dtype=torch.float16 if mixed_precision_type == "fp16" else torch.bfloat16, enabled=bool(amp)):
                        out = model(batch, gumbel_t=t)
                    grads.backward(scaler.scale(out.loss / gradient_accumulate_every))
                grads.all_reduce()                # (scaled) gradients first: every rank then sees the same inf / nan verdict
                scaler.unscale_(optimizer)
                scaler.step(optimizer)
                scaler.update()
                with torch.no_grad():
                    stats = step_statistics(out)
                norms_dev = out.embs_norm.mean(dim=0)
            if scheduler is not None:
                scheduler.step()

            acc += stats
            acc_n += 1
            if is_main and it % log_every == 0:
                means = (acc / acc_n).tolist()
                acc.zero_()
                acc_n = 0
                norms = norms_dev.tolist()
                rate = (it - start_iter + 1) * batch_size * gradient_accumulate_every * world / max(time.time() - t_start, 1e-9)
                history.append(dict(iter=it, **dict(zip(names, means))))
                logger.info("Iteration %d - " % it + ", ".join(f"{n}: {v:.4f}" for n, v in zip(names, means))
                            + f", emb norms: {[round(v, 4) for v in norms]}, lr: {[float(g['lr']) for g in optimizer.param_groups][:2]}, "
                            + f"items/s: {rate:.0f}")

            if do_eval and ((it + 1) % eval_every == 0 or it + 1 == iterations):
                hv_dist.broadcast_buffers(model)   # BatchNorm running statistics: rank 0's, as DDP broadcasts buffers
                ev = evaluate(model, tokenizer, eval_dataset, index_dataset, batch_size, t, vae_n_layers, vae_codebook_size,
                              rank, world)
                if is_main:
                    logger.info("Evaluation %d - " % (it + 1) + ", ".join(f"{k}: {v:.4f}" for k, v in ev.items()))
                    ok = ev["tag_acc"] > 0.60 and ev["sem_id_repetition_rate"] < id_repetition_threshold
                    if ok:
                        os.makedirs(save_dir, exist_ok=True)
                        path = os.path.join(save_dir, "hrqvae_model_ACC%.4f_RQLOSS%.4f_DUPR%.4f_%s.pt" % (
                            ev["tag_acc"], ev["rqvae"], ev["sem_id_repetition_rate"], datetime.now().strftime("%Y%m%d_%H%M%S")))
                        torch.save({"iter": it + 1, "model": model.state_dict(), "model_config": model.config,
                                    "optimizer": optimizer.state_dict(), "accuracy": ev["tag_acc"], "rqvae_loss": ev["rqvae"],
                                    "sem_id_repetition_rate": ev["sem_id_repetition_rate"]}, path)
                        logger.info(f"Model saved to: {path}")
                        best_eval_accuracy = max(best_eval_accuracy, ev["tag_acc"])
                    else:
                        logger.info("Checkpoint gate not met (accuracy %.4f / 0.60, id repetition %.4f / %.4f): not saving"
                                    % (ev["tag_acc"], ev["sem_id_repetition_rate"], id_repetition_threshold))
                history.append(dict(iter=it + 1, eval=ev))
        return dict(model=model, tokenizer=tokenizer, history=history, save_dir=save_dir)
    finally:
        torch.set_float32_matmul_precision(matmul_precision_before)


@torch.no_grad()
def evaluate(model, tokenizer, eval_dataset, index_dataset, batch_size, t, n_layers, codebook_size, rank=0, world=1):
    """Eval losses over the eval split + corpus id statistics (reference train_hidvae.py:810-1142)."""
    model.eval()
    dev = model.device
    sums, n_batches = torch.zeros(6, device=dev), 0
    for lo in range(0, len(eval_dataset), max(batch_size, 1024)):
        out = model(eval_dataset[lo: lo + max(batch_size, 1024)], gumbel_t=t)
        sums += torch.stack([out.loss, out.reconstruction_loss.mean(), out.rqvae_loss.mean(), out.tag_align_loss.mean(),
                             out.tag_pred_loss.mean(), out.tag_pred_accuracy.mean()])
        n_batches += 1
    means = (sums / max(n_batches, 1)).tolist()
    tokenizer.reset()
    tokenizer.hrq_vae = model
    if world > 1:   # bulk assignment shards by items; one gather at the end (SURVEY.md section 8e)
        tokenizer.precompute_corpus_ids(index_dataset, shard=(rank, world))
        corpus_ids = tokenizer.gather_shards()
    else:
        corpus_ids = tokenizer.precompute_corpus_ids(index_dataset)
    res = dict(zip(["loss", "reconstruction", "rqvae", "tag_align", "tag_pred", "tag_acc"], means))
    _, counts = torch.unique(corpus_ids[:, n_layers - 1], return_counts=True)
    p = counts / corpus_ids.shape[0]
    res["rqvae_entropy"] = float(-(p * torch.log(p)).sum())
    res["max_id_duplicates"] = float(corpus_ids[:, -1].max() / corpus_ids.shape[0])
    for cid in range(n_layers):
        res[f"codebook_usage_{cid}"] = torch.unique(corpus_ids[:, cid]).numel() / codebook_size
    res["sem_id_repetition_rate"], _, _ = calculate_repetition_rate(corpus_ids[:, :n_layers])
    return res


if __name__ == "__main__":
    parse_config()
    train()
    if torch.distributed.is_initialized():
        torch.distributed.destroy_process_group()
