"""GPU tests of the drop-in module API (modules/quantize.py, modules/h_rqvae.py, init/kmeans.py,
modules/tokenizer/h_semids.py, train_hidvae.py) against fixtures recorded from the real reference.

The strongest drop-in check: the REFERENCE's state_dict is loaded into this repo's HRqVae and every field of
`HRqVaeComputedLosses` must match what the reference computed with those weights (tests/golden/hrqvae_forward.npz),
in eval mode and in (dropout-free, mixup-free) training mode, including gradients.
"""
import numpy as np
import pytest
import torch

from helpers import npz, t, unit_rows
from oracle import rq as O

pytestmark = pytest.mark.gpu

VAL = dict(rtol=1e-5, atol=1e-6)


@pytest.fixture(scope="module")
def mods():
    import types
    from data.schemas import TaggedSeqBatch
    from init.kmeans import Kmeans, kmeans_init_
    from modules.h_rqvae import HRqVae
    from modules.quantize import Quantize, QuantizeDistance, QuantizeForwardMode
    from modules.tokenizer.h_semids import HSemanticIdTokenizer
    return types.SimpleNamespace(TaggedSeqBatch=TaggedSeqBatch, Kmeans=Kmeans, kmeans_init_=kmeans_init_, HRqVae=HRqVae,
                                 Quantize=Quantize, QuantizeDistance=QuantizeDistance,
                                 QuantizeForwardMode=QuantizeForwardMode, HSemanticIdTokenizer=HSemanticIdTokenizer)


def _mode(mods, name):
    return {"ste": mods.QuantizeForwardMode.STE, "rot": mods.QuantizeForwardMode.ROTATION_TRICK}[name]


@pytest.mark.parametrize("mname", ["ste", "rot"])
@pytest.mark.parametrize("normalize", [0, 1])
@pytest.mark.parametrize("training", [0, 1])
def test_quantize_module_matches_reference(mods, golden_dir, mname, normalize, training):
    """`Quantize(...).forward(x, temperature)` -> QuantizeOutput, and autograd to x and embedding.weight."""
    g = npz(golden_dir, "quantize_levels.npz")
    tag = f"{mname}_norm{normalize}_train{training}"
    layer = mods.Quantize(32, 64, do_kmeans_init=False, codebook_normalize=bool(normalize),
                          commitment_weight=float(g[f"{tag}/beta"]), forward_mode=_mode(mods, mname)).cuda()
    with torch.no_grad():
        layer.embedding.weight.copy_(t(g[f"{tag}/weight"]))
    layer.train(bool(training))
    x = t(g[f"{tag}/x"]).cuda().requires_grad_(True)
    out = layer(x, temperature=0.2)
    assert torch.equal(out.ids.cpu(), t(g[f"{tag}/ids"]))
    torch.testing.assert_close(out.embeddings.cpu(), t(g[f"{tag}/emb_out"]), **VAL)
    torch.testing.assert_close(out.loss.cpu(), t(g[f"{tag}/loss"]), **VAL)
    ((out.embeddings * t(g[f"{tag}/g_emb"]).cuda()).sum() + (out.loss * t(g[f"{tag}/g_loss"]).cuda()).sum()).backward()
    torch.testing.assert_close(x.grad.cpu(), t(g[f"{tag}/grad_x"]), rtol=2e-5, atol=2e-6)
    torch.testing.assert_close(layer.embedding.weight.grad.cpu(), t(g[f"{tag}/grad_weight"]), rtol=1e-4, atol=1e-5)


def test_quantize_gumbel_and_errors(mods, golden_dir):
    """GUMBEL_SOFTMAX through the module (fused hv_gumbel_forward in training, the STE kernel in eval): ids equal the
    reference recording in both modes; CPU input is refused.  Values / gradients: tests/test_gpu_gumbel.py."""
    g = npz(golden_dir, "quantize_levels.npz")
    layer = mods.Quantize(32, 64, do_kmeans_init=False, commitment_weight=0.25,
                          forward_mode=mods.QuantizeForwardMode.GUMBEL_SOFTMAX).cuda()
    with torch.no_grad():
        layer.embedding.weight.copy_(t(g["gumbel/weight"]))
    layer.train(True)
    out = layer(t(g["gumbel/x"]).cuda(), temperature=0.2)
    assert torch.equal(out.ids.cpu(), t(g["gumbel/ids"]))
    assert out.embeddings.shape == (16, 32) and torch.isfinite(out.loss).all()
    layer.eval()
    out = layer(t(g["gumbel/x"]).cuda(), temperature=0.2)      # eval: fused kernel, mode-independent
    assert torch.equal(out.ids.cpu(), t(g["gumbel/ids"]))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        layer(t(g["gumbel/x"]), temperature=0.2)
    with pytest.raises(AssertionError):
        layer(torch.zeros(4, 31, device="cuda"), temperature=0.2)


def _load_reference_model(mods, g, tag, mname):
    model = mods.HRqVae(input_dim=64, embed_dim=32, hidden_dims=[48, 40], codebook_size=64, codebook_kmeans_init=False,
                        codebook_normalize=True, codebook_mode=_mode(mods, mname), n_layers=3, commitment_weight=0.4,
                        n_cat_features=0, tag_alignment_weight=0.15, tag_prediction_weight=0.55,
                        tag_class_counts=[5, 7, 9], tag_embed_dim=16, use_focal_loss=True,
                        focal_loss_params={"gamma": 2.7, "alpha": 0.24}, dropout_rate=0.0,
                        sem_id_uniqueness_weight=1.5, sem_id_uniqueness_margin=0.0)
    model.tag_prediction_loss.use_mixup = False
    for m in model.modules():               # same as the recording run: no dropout noise in the training-mode case
        if isinstance(m, torch.nn.Dropout):
            m.p = 0.0
    # weights shared by every case are stored once under state/; <tag>/state/ holds what the case's own forward changed
    state = {k[len("state/"):]: t(g[k]) for k in g.files if k.startswith("state/")}
    prefix = f"{tag}/state/"
    state.update({k[len(prefix):]: t(g[k]) for k in g.files if k.startswith(prefix)})
    missing, unexpected = model.load_state_dict(state, strict=True), None   # the reference's keys, unchanged
    return model.cuda()


@pytest.mark.parametrize("mname", ["ste", "rot"])
@pytest.mark.parametrize("training", [0, 1])
def test_hrqvae_forward_with_reference_weights(mods, golden_dir, mname, training):
    g = npz(golden_dir, "hrqvae_forward.npz")
    tag = f"{mname}_train{training}"
    model = _load_reference_model(mods, g, tag, mname)
    model.train(bool(training))
    batch = mods.TaggedSeqBatch(None, None, None, t(g["x"]).cuda(), None, None, t(g["tags_emb"]).cuda(),
                                t(g["tags_indices"]).cuda())
    out = model(batch, gumbel_t=0.2)
    tol = dict(rtol=2e-4, atol=2e-5)  # encoder/decoder GEMMs run on cuBLAS (TF32 off) vs the reference's CPU sgemm
    for name in ("reconstruction_loss", "rqvae_loss", "embs_norm"):
        torch.testing.assert_close(getattr(out, name).cpu(), t(g[f"{tag}/{name}"]), **tol)
    for name in ("loss", "tag_align_loss", "tag_pred_loss", "tag_pred_accuracy", "p_unique_ids", "sem_id_uniqueness_loss"):
        torch.testing.assert_close(getattr(out, name).detach().cpu().float().reshape(()), t(g[f"{tag}/{name}"]).float().reshape(()), **tol)
    torch.testing.assert_close(out.tag_pred_loss_by_layer.detach().cpu(), t(g[f"{tag}/tag_pred_loss_by_layer"]), **tol)
    if training:
        out.loss.backward()
        params = dict(model.named_parameters())
        for key in ("encoder.mlp.0.weight", "decoder.mlp.4.weight", "layers.0.embedding.weight", "layers.2.embedding.weight",
                    "tag_predictors.1.classifier.7.weight", "tag_projectors.0.0.weight"):
            torch.testing.assert_close(params[key].grad.cpu(), t(g[f"{tag}/grad/{key}"]), rtol=2e-3, atol=2e-5)
    # eval-mode ids and tag predictions (what the tokenizer caches)
    model.eval()
    with torch.no_grad():
        x = batch.x
        q = model.get_semantic_ids(model.encode(x))
        assert q.sem_ids.shape == (96, 3) and q.embeddings.shape == (96, 32, 3) and q.residuals.shape == (96, 32, 3)
        assert torch.equal(q.sem_ids.cpu(), t(g[f"{tag}/eval_sem_ids"]))
        assert torch.equal(model.predict_tags(x)["predictions"].cpu(), t(g[f"{tag}/eval_tag_predictions"]))


def test_fused_levels_equal_level_by_level(mods):
    """One fused launch for all levels == the reference's per-level loop through `Quantize.forward`."""
    torch.manual_seed(3)
    model = mods.HRqVae(input_dim=64, embed_dim=32, hidden_dims=[48], codebook_size=256, codebook_kmeans_init=False,
                        codebook_normalize=True, codebook_mode=mods.QuantizeForwardMode.ROTATION_TRICK, n_layers=3,
                        commitment_weight=0.4, n_cat_features=0, tag_class_counts=[5, 7, 9], tag_embed_dim=16).cuda()
    with torch.no_grad():
        model.layers[1].embedding.weight.mul_(0.3).sub_(0.15)
        model.layers[2].embedding.weight.mul_(0.12).sub_(0.06)
    enc = unit_rows(700, 32, 5).cuda()
    res = {}
    for fuse in (True, False):
        model.fuse_levels = fuse
        e = enc.clone().requires_grad_(True)
        q = model.get_semantic_ids(e)
        (q.embeddings.sum() + q.quantize_loss.sum()).backward()
        res[fuse] = (q, e.grad, [l.embedding.weight.grad.clone() for l in model.layers])
        model.zero_grad()
    assert torch.equal(res[True][0].sem_ids, res[False][0].sem_ids)
    torch.testing.assert_close(res[True][0].embeddings, res[False][0].embeddings, **VAL)
    torch.testing.assert_close(res[True][0].quantize_loss, res[False][0].quantize_loss, **VAL)
    torch.testing.assert_close(res[True][1], res[False][1], rtol=2e-5, atol=2e-6)
    for a, b in zip(res[True][2], res[False][2]):
        torch.testing.assert_close(a, b, rtol=1e-4, atol=1e-5)


@pytest.mark.parametrize("name", ["blobs", "unit32"])
def test_kmeans_class_matches_reference(mods, golden_dir, name):
    """`Kmeans(k).run(x)` with NumPy's global RNG seeded like the recording run (init/kmeans.py:38)."""
    g = npz(golden_dir, "kmeans.npz")
    x = t(g[f"{name}/x"])
    k = g[f"{name}/init_idx"].shape[0]
    seed = {"blobs": 4, "unit32": 7}[name]
    np.random.seed(seed)
    torch.manual_seed(seed)
    out = mods.Kmeans(k=k).run(x.cuda())
    assert torch.equal(out.assignment.cpu(), t(g[f"{name}/assignment"]))
    torch.testing.assert_close(out.centroids.cpu(), t(g[f"{name}/centroids"]), rtol=1e-5, atol=1e-6)
    with pytest.raises(ValueError):       # fewer rows than clusters: np.random.choice raises, like the reference
        mods.Kmeans(k=64).run(x[:10].cuda())
    weight = torch.empty(k, x.shape[1], device="cuda")
    np.random.seed(seed)
    mods.kmeans_init_(weight, x.cuda())
    torch.testing.assert_close(weight.cpu(), t(g[f"{name}/centroids"]), rtol=1e-5, atol=1e-6)


def test_kmeans_reseeds_empty_clusters(mods):
    """Duplicate points force empty clusters (exact distance ties go to the lowest index): every Lloyd iteration
    re-seeds them from data rows (init/kmeans.py:54-56); the run must end at max_iters with sane centroids."""
    np.random.seed(1)
    torch.manual_seed(1)
    x = torch.cat([torch.zeros(50, 8), torch.ones(50, 8), 2 * torch.ones(3, 8)]).cuda()
    out = mods.Kmeans(k=6, max_iters=50).run(x)
    assert out.centroids.shape == (6, 8) and torch.isfinite(out.centroids).all()
    assert float(out.centroids.min()) >= 0.0 and float(out.centroids.max()) <= 2.0
    assert out.assignment.shape == (103,) and int(out.assignment.max()) < 6


def test_lazy_kmeans_init_in_model(mods):
    """First training-mode call runs k-means level by level on that level's input (quantize.py:103-104)."""
    np.random.seed(0)
    torch.manual_seed(0)
    model = mods.HRqVae(input_dim=64, embed_dim=16, hidden_dims=[32], codebook_size=32, codebook_kmeans_init=True,
                        codebook_normalize=True, codebook_mode=mods.QuantizeForwardMode.STE, n_layers=2,
                        n_cat_features=0, tag_class_counts=[3, 4], tag_embed_dim=8).cuda()
    x = unit_rows(2000, 64, 8).cuda()
    model.train()
    with torch.no_grad():
        q = model.get_semantic_ids(model.encode(x))
    assert all(l.kmeans_initted for l in model.layers) and model._can_fuse()
    # after k-means every code of level 0 is used and the loss is far below that of the uniform(0,1) init
    assert torch.unique(q.sem_ids[:, 0]).numel() == 32
    fresh = mods.HRqVae(input_dim=64, embed_dim=16, hidden_dims=[32], codebook_size=32, codebook_kmeans_init=False,
                        codebook_normalize=True, codebook_mode=mods.QuantizeForwardMode.STE, n_layers=2,
                        n_cat_features=0, tag_class_counts=[3, 4], tag_embed_dim=8).cuda()
    fresh.encoder.load_state_dict(model.encoder.state_dict())
    with torch.no_grad():
        q0 = fresh.get_semantic_ids(fresh.encode(x))
    assert float(q.quantize_loss.mean()) < 0.5 * float(q0.quantize_loss.mean())   # k-means beats the uniform(0,1) init


def test_tokenizer_precompute_corpus_ids(mods, golden_dir):
    g = npz(golden_dir, "hrqvae_forward.npz")
    tag = "rot_train0"
    model = _load_reference_model(mods, g, tag, "rot")
    x = t(g["x"]).cuda()
    for kw, width in ((dict(use_concatenated_ids=True), 6), (dict(use_interleaved_ids=True), 6), (dict(), 3)):
        tok = mods.HSemanticIdTokenizer(input_dim=64, output_dim=32, hidden_dims=[48, 40], codebook_size=64, n_layers=3,
                                        n_cat_feats=0, hrqvae_codebook_normalize=True, tag_class_counts=[5, 7, 9],
                                        tag_embed_dim=16, chunk_items=40, **kw)
        tok.hrq_vae = model
        ids = tok.precompute_corpus_ids(x)
        assert ids.shape == (96, width) and tok.sem_ids_dim == width
        sem, tags = t(g[f"{tag}/eval_sem_ids"]), t(g[f"{tag}/eval_tag_predictions"])
        if "use_concatenated_ids" in kw:
            expect = torch.cat([sem, tags], dim=1)
        elif "use_interleaved_ids" in kw:
            expect = torch.stack([sem, tags], dim=2).reshape(96, 6)
        else:
            expect = sem
        assert torch.equal(ids.cpu(), expect)
    # sharded assignment: two ranks' contiguous shards concatenate to the unsharded table
    tok.reset()
    a = tok.precompute_corpus_ids(x, shard=(0, 2)).clone()
    b = tok.precompute_corpus_ids(x, shard=(1, 2)).clone()
    assert torch.equal(torch.cat([a, b]).cpu(), sem)
    # prefix lookups against the cache
    tok.cached_ids = torch.cat([a, b])
    present = tok.exists_prefix(sem[:10, :2].cuda())
    assert bool(present.all())
    absent = tok.exists_prefix(torch.full((4, 3), 63, dtype=torch.int64, device="cuda"))
    ref = (torch.full((4, 3), 63)[:, None, :] == sem[None]).all(-1).any(-1)
    assert torch.equal(absent.cpu(), ref)


def test_trainer_smoke(mods, tmp_path):
    """A short gin-configured run of train_hidvae.train on a synthetic catalogue: k-means init, accumulation,
    evaluation with corpus-id statistics; losses must be finite and the RQ loss must fall."""
    from hidvae_b200 import gin_lite
    import train_hidvae
    gin_lite.clear_config()
    gin_lite.parse_config("""
import modules.quantize
train.iterations = 60
train.batch_size = 128
train.gradient_accumulate_every = 2
train.vae_input_dim = 768
train.vae_n_cat_feats = 0
train.vae_hidden_dims = [128, 64]
train.vae_embed_dim = 32
train.vae_codebook_size = 64
train.vae_codebook_normalize = True
train.vae_n_layers = 3
train.vae_codebook_mode = %modules.quantize.QuantizeForwardMode.ROTATION_TRICK
train.dataset = %data.tags_processed.RecDataset.AMAZON
train.commitment_weight = 0.4
train.tag_class_counts = [8, 16, 32]
train.tag_embed_dim = 768
train.layer_specific_lr = True
train.learning_rate = 0.001
train.eval_every = 30
train.use_kmeans_init = True
train.synthetic_items = 3000
train.log_every = 10
""")
    res = train_hidvae.train(save_dir_root=str(tmp_path), dataset_folder="")
    logs = [h for h in res["history"] if "eval" not in h]
    evals = [h["eval"] for h in res["history"] if "eval" in h]
    assert len(logs) >= 6 and len(evals) == 2
    assert all(np.isfinite(h["loss"]) for h in logs)
    assert logs[-1]["rqvae"] < logs[0]["rqvae"] * 1.05
    assert 0.0 <= evals[-1]["sem_id_repetition_rate"] <= 1.0 and evals[-1]["codebook_usage_0"] > 0.3
    gin_lite.clear_config()


def test_trainer_fp16_amp_uses_loss_scaling_and_refuses_silent_synthetic_data(mods, tmp_path):
    """amp=True with the reference's default mixed_precision_type='fp16' (Accelerate applies a GradScaler there): the
    encoder must receive non-zero, finite gradients and the run must stay finite.  And a missing processed catalogue
    must raise unless synthetic data is asked for."""
    from hidvae_b200 import gin_lite
    import train_hidvae
    base = """
import modules.quantize
train.iterations = 8
train.batch_size = 128
train.vae_input_dim = 768
train.vae_n_cat_feats = 0
train.vae_hidden_dims = [128, 64]
train.vae_embed_dim = 32
train.vae_codebook_size = 64
train.vae_codebook_normalize = True
train.vae_codebook_mode = %modules.quantize.QuantizeForwardMode.ROTATION_TRICK
train.dataset = %data.tags_processed.RecDataset.AMAZON
train.tag_class_counts = [8, 16, 32]
train.use_kmeans_init = False
train.do_eval = False
train.log_every = 2
train.amp = True
train.mixed_precision_type = "fp16"
"""
    gin_lite.clear_config()
    gin_lite.parse_config(base)
    with pytest.raises(FileNotFoundError):
        train_hidvae.train(save_dir_root=str(tmp_path), dataset_folder=str(tmp_path / "nothing_here"))
    gin_lite.clear_config()
    gin_lite.parse_config(base + "train.synthetic_data = True\ntrain.synthetic_items = 2000\n")
    before = None
    res = train_hidvae.train(save_dir_root=str(tmp_path), dataset_folder="")
    logs = [h for h in res["history"] if "eval" not in h]
    assert logs and all(np.isfinite(h["loss"]) for h in logs)
    enc_w = res["model"].encoder.mlp[0].weight
    assert enc_w.grad is not None and bool(torch.isfinite(enc_w.grad).all()) and float(enc_w.grad.abs().max()) > 0.0
    gin_lite.clear_config()


def test_tag_prediction_loss_masked_form_equals_row_compaction(mods):
    """TagPredictionLoss averages over the rows with a valid target without compacting them (no host synchronisation,
    fixed shapes).  Against the reference's formulation -- boolean-mask the rows first, then plain means
    (modules/loss.py:232-321) -- for both loss families, with and without class weights; all targets invalid gives 0."""
    from modules.loss import TagPredictionLoss
    import torch.nn.functional as F
    g = torch.Generator().manual_seed(5)
    n, c = 257, 140
    logits = torch.randn(n, c, generator=g).cuda().requires_grad_(True)
    targets = torch.randint(0, c, (n,), generator=g)
    targets[::7] = -1
    targets = targets.cuda()
    keep = targets >= 0
    for focal, counts in ((False, None), (True, None), (True, {1: torch.randint(1, 50, (c,), generator=g).cuda()})):
        crit = TagPredictionLoss(use_focal_loss=focal, focal_params={"gamma": 2.2, "alpha": 0.3}, class_counts=counts)
        crit.use_mixup = False
        loss, acc = crit(logits, targets, layer_idx=1)
        # reference formulation on the compacted rows (every helper returns one value per row)
        lk, tk = logits[keep], targets[keep]
        if not focal:
            s = min(0.25, 0.05 + 0.06 * 1)
            probs = F.softmax(lk, dim=-1)
            ref = F.cross_entropy(lk, tk, label_smoothing=s) + 0.05 * F.kl_div(torch.log(probs + 1e-8), torch.full_like(probs, 1.0 / c),
                                                                                 reduction="batchmean")
        elif counts is None:
            ref = crit._focal_loss_with_smoothing(lk, tk, 2.2 * 1.35, max(0.08, 0.3 - 0.06)).mean()
        else:
            ref = crit._focal_loss_with_weights_and_smoothing(lk, tk, 2.2 * 1.35, crit._class_weights(1, lk.device)).mean()
        torch.testing.assert_close(loss, ref, rtol=1e-5, atol=1e-6)
        torch.testing.assert_close(acc, (lk.argmax(-1) == tk).float().mean(), rtol=0, atol=1e-6)
        (gl,) = torch.autograd.grad(loss, logits, retain_graph=True)
        (gr,) = torch.autograd.grad(ref, logits)
        torch.testing.assert_close(gl, gr, rtol=1e-4, atol=1e-7)
        assert float(gl[~keep].abs().max()) == 0.0                 # dropped rows receive no gradient
    none_valid = torch.full((n,), -1, device="cuda")
    loss0, acc0 = crit(logits, none_valid)
    assert float(loss0) == 0.0 and float(acc0) == 0.0
    # mixup: partners are drawn among the kept rows only, so the loss stays finite and dropped rows stay gradient-free
    crit.use_mixup = True
    torch.manual_seed(1)
    loss_m, _ = crit(logits, targets, layer_idx=1)
    (gm,) = torch.autograd.grad(loss_m, logits)
    assert bool(torch.isfinite(loss_m)) and float(gm[~keep].abs().max()) == 0.0 and float(gm[keep].abs().max()) > 0.0


def _small_tagged_model(mods):
    torch.manual_seed(0)
    np.random.seed(0)
    m = mods.HRqVae(input_dim=64, embed_dim=32, hidden_dims=[48], codebook_size=64, codebook_kmeans_init=False,
                    codebook_normalize=True, codebook_mode=mods.QuantizeForwardMode.ROTATION_TRICK, n_layers=3, n_cat_features=0,
                    commitment_weight=0.4, tag_class_counts=[5, 9, 17], tag_embed_dim=24, dropout_rate=0.0,
                    sem_id_uniqueness_weight=0.5, sem_id_uniqueness_margin=0.2).cuda().train()
    m.tag_prediction_loss.use_mixup = False
    for mod in m.modules():
        if isinstance(mod, torch.nn.Dropout):
            mod.p = 0.0
    return m


def test_graphed_train_step_equals_eager_steps(mods):
    """hidvae_b200.graph_step.GraphedTrainStep (gather + forward + backward as one CUDA graph, AdamW as another) against
    the same number of eager steps on the same index draws: parameters agree to summation-order noise, statistics too."""
    from data.schemas import TaggedSeqBatch
    from hidvae_b200 import dist as hv_dist
    from hidvae_b200.graph_step import GraphedTrainStep, step_statistics
    n, bs, steps, warm = 4096, 256, 6, 3
    g = torch.Generator().manual_seed(3)
    x = unit_rows(n, 64, 1).cuda()
    tags_emb = torch.randn(n, 3, 24, generator=g).cuda()
    tags_idx = torch.stack([torch.randint(0, c, (n,), generator=g) for c in (5, 9, 17)], dim=1)
    tags_idx[::9, 2] = -1
    tags_idx = tags_idx.cuda()
    fetch = lambda idx: TaggedSeqBatch(None, None, None, x[idx], None, None, tags_emb[idx], tags_idx[idx])
    results = []
    for graphed in (False, True):
        model = _small_tagged_model(mods)
        grads = hv_dist.FlatGradAllReduce(model.parameters())
        opt = torch.optim.AdamW(model.parameters(), lr=torch.tensor(1e-3, device="cuda"), weight_decay=0.01, capturable=True)
        gen = torch.Generator(device="cuda").manual_seed(11)
        stats = None
        if graphed:
            step = GraphedTrainStep(model, opt, grads, fetch, bs, n, gumbel_t=0.2, generator=gen, warmup=warm)
            for _ in range(steps):
                stats = step().clone()
        else:
            for _ in range(warm + steps):
                idx = torch.randint(0, n, (bs,), device="cuda", generator=gen)
                grads.zero()
                out = model(fetch(idx), gumbel_t=0.2)
                out.loss.backward()
                opt.step()
                stats = step_statistics(out)
        results.append((torch.cat([p.detach().flatten() for p in model.parameters()]), stats))
    (p_e, s_e), (p_g, s_g) = results
    torch.testing.assert_close(s_g, s_e, rtol=2e-3, atol=2e-4)
    assert float((p_g - p_e).abs().max()) < 5e-4                  # nine Adam steps of 1e-3 each: the two runs stay together
    with pytest.raises(ValueError, match="capturable"):
        GraphedTrainStep(model, torch.optim.AdamW(model.parameters(), lr=1e-3), grads, fetch, bs, n)


def test_trainer_with_cuda_graph(mods, tmp_path):
    """train_hidvae.train(use_cuda_graph=True): k-means init, then graph replays with the cosine schedule writing the
    learning rate in place; the RQ loss must fall as in the eager run, evaluation runs between replays."""
    from hidvae_b200 import gin_lite
    import train_hidvae
    gin_lite.clear_config()
    gin_lite.parse_config("""
import modules.quantize
train.iterations = 60
train.batch_size = 128
train.gradient_accumulate_every = 2
train.vae_input_dim = 768
train.vae_n_cat_feats = 0
train.vae_hidden_dims = [128, 64]
train.vae_embed_dim = 32
train.vae_codebook_size = 64
train.vae_codebook_normalize = True
train.vae_n_layers = 3
train.vae_codebook_mode = %modules.quantize.QuantizeForwardMode.ROTATION_TRICK
train.dataset = %data.tags_processed.RecDataset.AMAZON
train.commitment_weight = 0.4
train.tag_class_counts = [8, 16, 32]
train.tag_embed_dim = 768
train.layer_specific_lr = True
train.learning_rate = 0.001
train.lr_scheduler_T_max = 60
train.eval_every = 30
train.use_kmeans_init = True
train.synthetic_items = 3000
train.log_every = 10
train.use_cuda_graph = True
""")
    res = train_hidvae.train(save_dir_root=str(tmp_path), dataset_folder="")
    logs = [h for h in res["history"] if "eval" not in h]
    evals = [h["eval"] for h in res["history"] if "eval" in h]
    assert len(logs) >= 6 and len(evals) == 2
    assert all(np.isfinite(h["loss"]) for h in logs)
    assert logs[-1]["rqvae"] < logs[0]["rqvae"] * 1.05
    assert 0.0 <= evals[-1]["sem_id_repetition_rate"] <= 1.0 and evals[-1]["codebook_usage_0"] > 0.3
    gin_lite.clear_config()
    gin_lite.parse_config("train.use_cuda_graph = True\ntrain.amp = True\ntrain.synthetic_items = 500\ntrain.dataset = %data.tags_processed.RecDataset.AMAZON\n")
    with pytest.raises(ValueError, match="fp16"):
        train_hidvae.train(save_dir_root=str(tmp_path), dataset_folder="")
    gin_lite.clear_config()
