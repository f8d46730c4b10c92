"""TEST INFRASTRUCTURE ONLY -- writes tests/golden/*.npz by running the REAL reference (authoring container).

    python oracle/make_golden.py            # needs /root/reference; re-creates every fixture

The reference ships no golden vectors (SURVEY.md section 4), so these fixtures -- outputs of the reference's own
`Quantize`, `HRqVae.get_semantic_ids`, `SemanticIdUniquenessLoss`, `Kmeans` on seeded synthetic inputs
(SURVEY.md section 8d) -- are what pins the oracle, and through it the CUDA path.  The fixtures travel to the GPU
box; the reference does not.
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle.reference_shim import load_reference  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")


def _np(t):
    return t.detach().cpu().numpy()


def unit_rows(n, d, gen):
    return torch.nn.functional.normalize(torch.randn(n, d, generator=gen), dim=-1)


def make_quantize_cases(ref):
    """Single `Quantize.forward` (modules/quantize.py:100-154): value + autograd gradients."""
    Q = ref.quantize
    modes = {"ste": Q.QuantizeForwardMode.STE, "rot": Q.QuantizeForwardMode.ROTATION_TRICK}
    out = {}
    for mname, mode in modes.items():
        for normalize in (False, True):
            for training in (True, False):
                gen = torch.Generator().manual_seed(11)
                n, d, k, beta = 48, 32, 64, 0.4
                layer = Q.Quantize(d, k, do_kmeans_init=False, codebook_normalize=normalize,
                                   commitment_weight=beta, forward_mode=mode)
                with torch.no_grad():
                    layer.embedding.weight.copy_(torch.rand(k, d, generator=gen))
                layer.train(training)
                x = (unit_rows(n, d, gen) * (0.5 + torch.rand(n, 1, generator=gen))).requires_grad_(True)
                g_emb = torch.randn(n, d, generator=gen)
                g_loss = torch.randn(n, generator=gen)
                res = layer(x, temperature=0.2)
                ((res.embeddings * g_emb).sum() + (res.loss * g_loss).sum()).backward()
                tag = f"{mname}_norm{int(normalize)}_train{int(training)}"
                out.update({
                    f"{tag}/x": _np(x), f"{tag}/weight": _np(layer.embedding.weight),
                    f"{tag}/g_emb": _np(g_emb), f"{tag}/g_loss": _np(g_loss),
                    f"{tag}/emb_out": _np(res.embeddings), f"{tag}/ids": _np(res.ids),
                    f"{tag}/loss": _np(res.loss), f"{tag}/grad_x": _np(x.grad),
                    f"{tag}/grad_weight": _np(layer.embedding.weight.grad),
                    f"{tag}/beta": np.float32(beta),
                })
    # Gumbel-softmax with the uniform noise recorded (distributions/gumbel.py:8-18 draws torch.rand)
    gen = torch.Generator().manual_seed(5)
    n, d, k = 16, 32, 64
    layer = Q.Quantize(d, k, do_kmeans_init=False, commitment_weight=0.25,
                       forward_mode=Q.QuantizeForwardMode.GUMBEL_SOFTMAX)
    with torch.no_grad():
        layer.embedding.weight.copy_(torch.rand(k, d, generator=gen))
    layer.train(True)
    x = unit_rows(n, d, gen)
    torch.manual_seed(123)
    uniform = torch.rand((n, k))
    torch.manual_seed(123)
    res = layer(x, temperature=0.2)
    out.update({"gumbel/x": _np(x), "gumbel/weight": _np(layer.embedding.weight), "gumbel/uniform": _np(uniform),
                "gumbel/emb_out": _np(res.embeddings), "gumbel/ids": _np(res.ids), "gumbel/loss": _np(res.loss)})
    np.savez_compressed(os.path.join(OUT, "quantize_levels.npz"), **out)


def make_rq_cases(ref):
    """`HRqVae.get_semantic_ids` without tags (modules/h_rqvae.py:481-583), C1 shape: D=32 K=256 L=3."""
    Q = ref.quantize
    H = ref.h_rqvae
    modes = {"ste": Q.QuantizeForwardMode.STE, "rot": Q.QuantizeForwardMode.ROTATION_TRICK}
    out = {}
    for mname, mode in modes.items():
        for training in (True, False):
            gen = torch.Generator().manual_seed(3)
            n, d, k, L, beta = 64, 32, 256, 3, 0.4
            model = H.HRqVae(input_dim=48, embed_dim=d, hidden_dims=[40], codebook_size=k,
                             codebook_kmeans_init=False, codebook_normalize=True, codebook_mode=mode,
                             n_layers=L, commitment_weight=beta, n_cat_features=0,
                             tag_class_counts=[5, 7, 9], tag_embed_dim=16)
            with torch.no_grad():
                for layer in model.layers:
                    layer.embedding.weight.copy_(torch.rand(k, d, generator=gen))
                # make later levels comparable in scale to the residuals so every level is exercised
                model.layers[1].embedding.weight.mul_(0.25).sub_(0.125)
                model.layers[2].embedding.weight.mul_(0.1).sub_(0.05)
            model.train(training)
            enc = unit_rows(n, d, gen).requires_grad_(True)
            g_emb = torch.randn(n, d, L, generator=gen)
            g_loss = torch.randn(n, generator=gen)
            res = model.get_semantic_ids(enc)
            ((res.embeddings * g_emb).sum() + (res.quantize_loss * g_loss).sum()).backward()
            tag = f"{mname}_train{int(training)}"
            out.update({
                f"{tag}/enc": _np(enc), f"{tag}/g_emb": _np(g_emb), f"{tag}/g_loss": _np(g_loss),
                f"{tag}/weights": np.stack([_np(l.embedding.weight) for l in model.layers]),
                f"{tag}/embeddings": _np(res.embeddings), f"{tag}/residuals": _np(res.residuals),
                f"{tag}/sem_ids": _np(res.sem_ids), f"{tag}/quantize_loss": _np(res.quantize_loss),
                f"{tag}/grad_enc": _np(enc.grad),
                f"{tag}/grad_weights": np.stack([_np(l.embedding.weight.grad) for l in model.layers]),
                f"{tag}/beta": np.float32(beta),
            })
    np.savez_compressed(os.path.join(OUT, "rq_c1.npz"), **out)


def make_uniqueness_cases(ref):
    """`SemanticIdUniquenessLoss` (modules/h_rqvae.py:25-105) and p_unique_ids (:645-648)."""
    H = ref.h_rqvae
    from einops import rearrange
    gen = torch.Generator().manual_seed(9)
    out = {}
    for name, (b, L, k, margin, weight) in {"dups": (96, 3, 3, 0.0, 1.5), "margin": (64, 3, 2, 0.5, 0.5),
                                           "nodup": (40, 3, 256, 0.0, 1.5)}.items():
        ids = torch.randint(0, k, (b, L), generator=gen)
        if name == "nodup":
            ids[:, 0] = torch.arange(b)
        feats = torch.randn(b, 32, generator=gen).requires_grad_(True)
        loss_fn = H.SemanticIdUniquenessLoss(margin=margin, weight=weight)
        loss = loss_fn(ids, feats)
        if loss.requires_grad:
            loss.backward()
            grad = _np(feats.grad)
        else:
            grad = np.zeros((b, 32), np.float32)
        as_wired = loss_fn(ids.transpose(0, 1), feats.detach())  # what HRqVae.forward actually calls (:630-631)
        p_unique = (~torch.triu((rearrange(ids, "b d -> b 1 d") == rearrange(ids, "b d -> 1 b d")).all(axis=-1),
                                diagonal=1)).all(axis=1).sum() / ids.shape[0]
        out.update({f"{name}/ids": _np(ids), f"{name}/feats": _np(feats), f"{name}/loss": _np(loss),
                    f"{name}/grad_feats": grad, f"{name}/loss_as_wired": _np(as_wired),
                    f"{name}/p_unique": _np(p_unique), f"{name}/margin": np.float32(margin),
                    f"{name}/weight": np.float32(weight)})
    np.savez_compressed(os.path.join(OUT, "uniqueness.npz"), **out)


def make_kmeans_cases(ref):
    """`Kmeans(k).run(x)` (init/kmeans.py:63-77) with the NumPy-global-RNG initial rows recorded."""
    K = ref.kmeans
    out = {}
    for name, (n, d, k, seed) in {"blobs": (600, 8, 12, 4), "unit32": (2000, 32, 64, 7)}.items():
        gen = torch.Generator().manual_seed(seed)
        if name == "blobs":
            centers = torch.randn(k, d, generator=gen) * 4
            x = centers[torch.randint(0, k, (n,), generator=gen)] + 0.3 * torch.randn(n, d, generator=gen)
        else:
            x = unit_rows(n, d, gen)
        np.random.seed(seed)
        init_idx = np.random.choice(n, k, replace=False)
        np.random.seed(seed)
        torch.manual_seed(seed)
        import io, contextlib
        with contextlib.redirect_stdout(io.StringIO()):
            res = K.Kmeans(k=k).run(x)
        out.update({f"{name}/x": _np(x), f"{name}/init_idx": init_idx.astype(np.int64),
                    f"{name}/centroids": _np(res.centroids), f"{name}/assignment": _np(res.assignment)})
    np.savez_compressed(os.path.join(OUT, "kmeans.npz"), **out)


def make_hrqvae_forward_cases(ref):
    """Whole `HRqVae.forward` of the reference (modules/h_rqvae.py:585-672) with tags, plus its state_dict, so the
    drop-in module can be loaded with the reference's weights and compared output by output.  Dropout is 0 and mixup
    is off so that the training-mode case is deterministic."""
    Q, H, S = ref.quantize, ref.h_rqvae, ref.schemas
    out = {}
    for mname, mode in {"ste": Q.QuantizeForwardMode.STE, "rot": Q.QuantizeForwardMode.ROTATION_TRICK}.items():
        for training in (True, False):
            torch.manual_seed(17)
            gen = torch.Generator().manual_seed(17)
            n, din, d, k, L, tdim = 96, 64, 32, 64, 3, 16
            counts = [5, 7, 9]
            model = H.HRqVae(input_dim=din, embed_dim=d, hidden_dims=[48, 40], codebook_size=k,
                             codebook_kmeans_init=False, codebook_normalize=True, codebook_mode=mode, n_layers=L,
                             commitment_weight=0.4, n_cat_features=0, tag_alignment_weight=0.15,
                             tag_prediction_weight=0.55, tag_class_counts=counts, tag_embed_dim=tdim,
                             use_focal_loss=True, focal_loss_params={"gamma": 2.7, "alpha": 0.24}, dropout_rate=0.0,
                             sem_id_uniqueness_weight=1.5, sem_id_uniqueness_margin=0.0)
            model.tag_prediction_loss.use_mixup = False
            for m in model.modules():       # TagPredictor adds 0.075 * layer_idx of dropout even at dropout_rate 0
                if isinstance(m, torch.nn.Dropout):
                    m.p = 0.0
            with torch.no_grad():
                model.layers[1].embedding.weight.mul_(0.3).sub_(0.15)
                model.layers[2].embedding.weight.mul_(0.12).sub_(0.06)
            model.train(training)
            x = unit_rows(n, din, gen)
            tags_emb = torch.randn(n, L, tdim, generator=gen)
            tags_idx = torch.stack([torch.randint(0, c, (n,), generator=gen) for c in counts], dim=1)
            tags_idx[::11, 1] = -1
            batch = S.TaggedSeqBatch(None, None, None, x, None, None, tags_emb, tags_idx)
            res = model(batch, gumbel_t=0.2)
            tag = f"{mname}_train{int(training)}"
            if training:
                res.loss.backward()
                for key in ("encoder.mlp.0.weight", "decoder.mlp.4.weight", "layers.0.embedding.weight",
                            "layers.2.embedding.weight", "tag_predictors.1.classifier.7.weight", "tag_projectors.0.0.weight"):
                    out[f"{tag}/grad/{key}"] = _np(dict(model.named_parameters())[key].grad)
            for key, val in model.state_dict().items():
                out[f"{tag}/state/{key}"] = _np(val)
            out.update({f"{tag}/x": _np(x), f"{tag}/tags_emb": _np(tags_emb), f"{tag}/tags_indices": _np(tags_idx),
                        f"{tag}/loss": _np(res.loss), f"{tag}/reconstruction_loss": _np(res.reconstruction_loss),
                        f"{tag}/rqvae_loss": _np(res.rqvae_loss), f"{tag}/tag_align_loss": _np(res.tag_align_loss),
                        f"{tag}/tag_pred_loss": _np(res.tag_pred_loss), f"{tag}/tag_pred_accuracy": _np(res.tag_pred_accuracy),
                        f"{tag}/embs_norm": _np(res.embs_norm), f"{tag}/p_unique_ids": _np(res.p_unique_ids),
                        f"{tag}/sem_id_uniqueness_loss": _np(res.sem_id_uniqueness_loss),
                        f"{tag}/tag_pred_loss_by_layer": _np(res.tag_pred_loss_by_layer)})
            with torch.no_grad():
                model.eval()
                q = model.get_semantic_ids(model.encode(x))
                out[f"{tag}/eval_sem_ids"] = _np(q.sem_ids)
                out[f"{tag}/eval_tag_predictions"] = _np(model.predict_tags(x)["predictions"])
    tags = [f"{m}_train{int(tr)}" for m in ("ste", "rot") for tr in (True, False)]
    _store_shared_once(out, tags, lambda name: name.startswith("state/") or name in ("x", "tags_emb", "tags_indices"))
    np.savez_compressed(os.path.join(OUT, "hrqvae_forward.npz"), **out)


def _store_shared_once(out, tags, eligible):
    """Every case starts from the same seed, so weights and inputs repeat across cases: an eligible `<tag>/<name>`
    that is identical under every tag is stored once as `<name>` (keeps the fixture small).  What differs, such as
    the BatchNorm statistics a training-mode forward updates, stays under its tag."""
    for name in [k[len(tags[0]) + 1:] for k in out if k.startswith(tags[0] + "/")]:
        if not eligible(name):
            continue
        vals = [out[f"{tag}/{name}"] for tag in tags]
        if all(v.dtype == vals[0].dtype and np.array_equal(v, vals[0]) for v in vals[1:]):
            out[name] = vals[0]
            for tag in tags:
                del out[f"{tag}/{name}"]


def make_tokenizer_cases(ref):
    """Cached-id consumers of the reference tokenizer (modules/tokenizer/h_semids.py:197-258 and the cached branch of
    `forward`, :366-402): rows of `cached_ids` gathered per sequence position, masked positions set to -1, token type
    ids, `exists_prefix`.  `cached_ids` is synthetic (the methods only index it); prefix batches are multiples of the
    reference's BATCH_SIZE = 16, the only sizes its batching loop (`ceil(n // 16)`) covers completely."""
    from oracle.reference_shim import load_reference_tokenizer
    T = load_reference_tokenizer()
    S = ref.schemas
    out = {}
    for name, kw, width in (("plain", {}, 3), ("concat", dict(use_concatenated_ids=True, tag_class_counts=[5, 7, 9]), 6),
                            ("interleaved", dict(use_interleaved_ids=True, tag_class_counts=[5, 7, 9]), 6)):
        torch.manual_seed(3)
        gen = torch.Generator().manual_seed(31)
        tok = T.HSemanticIdTokenizer(input_dim=24, output_dim=8, hidden_dims=[16], codebook_size=16, n_layers=3,
                                     n_cat_feats=0, tag_embed_dim=8, **kw)
        n_items, b, n = 50, 6, 5
        tok.cached_ids = torch.randint(0, 16, (n_items, width), generator=gen)
        ids = torch.randint(0, n_items, (b, n), generator=gen)
        ids_fut = torch.randint(0, n_items, (b, 1), generator=gen)
        seq_mask = torch.rand(b, n, generator=gen) > 0.3
        batch = S.SeqBatch(user_ids=torch.arange(b), ids=ids, ids_fut=ids_fut, x=torch.zeros(b, n, 24),
                           x_fut=torch.zeros(b, 24), seq_mask=seq_mask)
        res = tok(batch)
        prefixes = torch.cat([tok.cached_ids[torch.randint(0, n_items, (24,), generator=gen), :2],
                              torch.randint(0, 16, (24, 2), generator=gen)])           # 48 = 3 x BATCH_SIZE rows
        full = torch.cat([tok.cached_ids[:8], torch.randint(0, 16, (8, width), generator=gen)])   # 16 rows, full width
        out.update({f"{name}/cached_ids": _np(tok.cached_ids), f"{name}/ids": _np(ids), f"{name}/ids_fut": _np(ids_fut),
                    f"{name}/seq_mask": _np(seq_mask), f"{name}/sem_ids": _np(res.sem_ids), f"{name}/sem_ids_fut": _np(res.sem_ids_fut),
                    f"{name}/out_seq_mask": _np(res.seq_mask), f"{name}/token_type_ids": _np(res.token_type_ids),
                    f"{name}/token_type_ids_fut": _np(res.token_type_ids_fut),
                    f"{name}/from_cached": _np(tok._tokenize_seq_batch_from_cached(ids)),
                    f"{name}/prefixes": _np(prefixes), f"{name}/prefix_hits": _np(tok.exists_prefix(prefixes)),
                    f"{name}/full_rows": _np(full), f"{name}/full_hits": _np(tok.exists_prefix(full)),
                    f"{name}/sem_ids_dim": np.asarray(tok.sem_ids_dim)})
    np.savez_compressed(os.path.join(OUT, "tokenizer_cached.npz"), **out)


def make_encoder_cases(ref):
    """The reference's own `MLP` (modules/encoder.py) at the gin shape 768 -> 512 -> 256 -> 128 -> 32, with and without
    the L2-norm tail, on seeded unit-norm rows.  The weights come from oracle.encoder.seeded_weights(dims, seed) so the
    fixture carries the seed, not the matrices."""
    import modules.encoder as ref_encoder
    from oracle import encoder as OE
    dims, seed = [768, 512, 256, 128, 32], 2024
    weights = OE.seeded_weights(dims, seed)
    gen = torch.Generator().manual_seed(77)
    x = unit_rows(48, dims[0], gen)
    out = {"dims": np.asarray(dims), "seed": np.asarray(seed), "x": _np(x)}
    for normalize in (False, True):
        mlp = ref_encoder.MLP(input_dim=dims[0], hidden_dims=dims[1:-1], out_dim=dims[-1], normalize=normalize).eval()
        linears = [m for m in mlp.mlp if isinstance(m, torch.nn.Linear)]
        with torch.no_grad():
            for lin, w in zip(linears, weights):
                lin.weight.copy_(w)
            out[f"z_norm{int(normalize)}"] = _np(mlp(x))
    np.savez_compressed(os.path.join(OUT, "encoder.npz"), **out)


def main():
    os.makedirs(OUT, exist_ok=True)
    torch.set_num_threads(1)  # fixed reduction order for the recorded values
    ref = load_reference()
    make_quantize_cases(ref)
    make_rq_cases(ref)
    make_uniqueness_cases(ref)
    make_kmeans_cases(ref)
    make_encoder_cases(ref)
    import io, contextlib
    with contextlib.redirect_stdout(io.StringIO()):
        make_hrqvae_forward_cases(ref)
        make_tokenizer_cases(ref)
    for f in sorted(os.listdir(OUT)):
        print(f, os.path.getsize(os.path.join(OUT, f)))


if __name__ == "__main__":
    main()
