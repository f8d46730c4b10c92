"""GPU parity of the fused Gumbel-softmax level (hv_gumbel_forward / hv_gumbel_backward, csrc/gumbel.cu) against the
reference recording (tests/golden/quantize_levels.npz: gumbel/*) and the CPU oracle with the SAME uniforms
(modules/quantize.py:108-130,144; distributions/gumbel.py:8-18).

Bars: ids bit-exact (the seeded inputs hold no near-tie), emb_out / loss rtol 1e-5 + atol 1e-6, g_x rtol 1e-4 + atol 1e-6,
codebook gradient rtol 1e-4 + atol 1e-5 x its scale (sums over rows in another order than the oracle's matmul)."""
import numpy as np
import pytest
import torch

from helpers import npz, ops, t, unit_rows
from oracle import rq as O

pytestmark = pytest.mark.gpu


def test_gumbel_golden_recorded_noise(ops, golden_dir):
    g = npz(golden_dir, "quantize_levels.npz")
    x, w, u = t(g["gumbel/x"]).cuda(), t(g["gumbel/weight"]).cuda(), t(g["gumbel/uniform"]).cuda()
    emb, ids, loss = ops.gumbel_apply(x, w, 0.2, 0.25, uniforms=u)
    assert torch.equal(ids.cpu(), t(g["gumbel/ids"]))
    torch.testing.assert_close(emb.cpu(), t(g["gumbel/emb_out"]), rtol=1e-5, atol=1e-6)
    torch.testing.assert_close(loss.cpu(), t(g["gumbel/loss"]), rtol=1e-5, atol=1e-6)


@pytest.mark.parametrize("temperature", [0.2, 1.0, 0.05])
@pytest.mark.parametrize("shape", [(1000, 32, 256), (513, 64, 200), (77, 16, 32), (1, 32, 7)], ids=lambda s: "n%d_d%d_k%d" % s)
def test_gumbel_forward_backward_vs_oracle(ops, shape, temperature):
    n, d, k = shape
    beta = 0.4
    gen = torch.Generator().manual_seed(11 + n)
    x = unit_rows(n, d, seed=5)
    cb = torch.nn.functional.normalize(torch.rand(k, d, generator=gen), dim=-1)
    u = torch.rand(n, k, generator=gen)
    g_emb = torch.randn(n, d, generator=gen) * 0.1
    g_loss = torch.rand(n, generator=gen) / n
    # oracle (autograd on the reference formulas)
    x_o, cb_o = x.clone().requires_grad_(True), cb.clone().requires_grad_(True)
    ref = O.quantize_level(x_o, cb_o, O.MODE_GUMBEL_SOFTMAX, beta, True, temperature, uniform=u)
    ((ref.embeddings * g_emb).sum() + (ref.loss * g_loss).sum()).backward()
    # GPU
    x_d, cb_d = x.cuda().requires_grad_(True), cb.cuda().requires_grad_(True)
    emb, ids, loss = ops.gumbel_apply(x_d, cb_d, temperature, beta, uniforms=u.cuda())
    ((emb * g_emb.cuda()).sum() + (loss * g_loss.cuda()).sum()).backward()
    assert torch.equal(ids.cpu(), ref.ids)
    tol = 1e-5 if temperature >= 0.2 else 1e-4        # logits are dist / T: fp32 round-off of dist is amplified by 1 / T
    torch.testing.assert_close(emb.detach().cpu(), ref.embeddings.detach(), rtol=tol, atol=tol * 0.1)
    torch.testing.assert_close(loss.detach().cpu(), ref.loss.detach(), rtol=tol, atol=tol * 0.1)
    gscale = float(x_o.grad.abs().max())
    torch.testing.assert_close(x_d.grad.cpu(), x_o.grad, rtol=10 * tol, atol=10 * tol * gscale)
    cscale = float(cb_o.grad.abs().max())
    torch.testing.assert_close(cb_d.grad.cpu(), cb_o.grad, rtol=10 * tol, atol=10 * tol * cscale)


def test_gumbel_philox_noise_is_the_recorded_draw(ops):
    """In-kernel Philox noise: hv_gumbel_uniforms reproduces the draw of a seed; feeding it back explicitly gives the same
    forward and backward bit for bit; the draw is uniform on [0, 1) (moments + a coarse histogram) and differs by seed."""
    n, d, k = 4096, 32, 256
    x = unit_rows(n, d, seed=9).cuda()
    cb = torch.nn.functional.normalize(torch.rand(k, d, generator=torch.Generator().manual_seed(2)), dim=-1).cuda()
    outs = []
    for uniforms in (None, ops.gumbel_uniforms(n, k, 1234, "cuda")):
        x_d, cb_d = x.clone().requires_grad_(True), cb.clone().requires_grad_(True)
        emb, ids, loss = ops.gumbel_apply(x_d, cb_d, 0.2, 0.25, uniforms=uniforms, seed=1234)
        (emb.sum() * 0.5 + loss.mean()).backward()
        outs.append((emb.detach(), ids, loss.detach(), x_d.grad, cb_d.grad))
    for name, a, b in zip(("emb", "ids", "loss", "g_x", "g_codebook"), *outs[:2]):
        if name == "g_codebook":    # folded with atomics: the order of the additions differs from launch to launch
            torch.testing.assert_close(a, b, rtol=1e-5, atol=1e-6 * float(b.abs().max()))
        else:
            assert torch.equal(a, b), name
    u = ops.gumbel_uniforms(n, k, 1234, "cuda")
    assert float(u.min()) >= 0.0 and float(u.max()) < 1.0
    assert abs(float(u.mean()) - 0.5) < 2e-3 and abs(float(u.var()) - 1.0 / 12.0) < 1e-3
    hist = torch.histc(u, bins=16, min=0.0, max=1.0) / u.numel()
    assert float((hist - 1.0 / 16).abs().max()) < 2e-3
    u2 = ops.gumbel_uniforms(n, k, 1235, "cuda")
    assert float((u == u2).float().mean()) < 1e-3
    # rows and columns are decorrelated (a counter-layout bug would repeat lanes or rows)
    assert abs(float(torch.corrcoef(torch.stack([u[:-1].flatten(), u[1:].flatten()]))[0, 1])) < 5e-3
    assert abs(float(torch.corrcoef(torch.stack([u[:, :-1].flatten(), u[:, 1:].flatten()]))[0, 1])) < 5e-3


def test_gumbel_module_training_step(ops):
    """Quantize(forward_mode=GUMBEL_SOFTMAX) in training mode runs the fused kernels: reproducible under torch.manual_seed,
    gradients reach the embedding table, ids equal the eval-mode (hard) ids, emb_out approaches the chosen code as T -> 0."""
    from modules.quantize import Quantize, QuantizeForwardMode
    torch.manual_seed(0)
    layer = Quantize(32, 256, do_kmeans_init=False, codebook_normalize=True, forward_mode=QuantizeForwardMode.GUMBEL_SOFTMAX).cuda()
    x = unit_rows(512, 32, seed=3).cuda().requires_grad_(True)
    layer.train()
    torch.manual_seed(42)
    a = layer(x, temperature=0.2)
    torch.manual_seed(42)
    b = layer(x, temperature=0.2)
    assert torch.equal(a.embeddings, b.embeddings) and torch.equal(a.ids, b.ids)
    c = layer(x, temperature=0.2)
    assert not torch.equal(a.embeddings, c.embeddings)           # a fresh draw
    (a.embeddings.pow(2).sum() + a.loss.sum()).backward()
    assert layer.embedding.weight.grad is not None and float(layer.embedding.weight.grad.abs().sum()) > 0
    assert x.grad is not None and torch.isfinite(x.grad).all()
    layer.eval()
    hard = layer(x.detach(), temperature=0.2)
    assert torch.equal(hard.ids, a.ids)
    layer.train()
    # noise of scale ~1 against distance gaps amplified by 1 / T = 1e4: the soft assignment collapses onto one code
    cold = layer(x.detach(), temperature=1e-4)
    cb = layer.effective_codebook().detach()
    dmin = torch.cdist(cold.embeddings, cb).min(dim=1).values
    assert float(dmin.median()) < 1e-4 and float((dmin < 1e-3).float().mean()) > 0.98   # (two codes can tie within T)


def test_gumbel_unsupported_shape_and_arguments(ops):
    from hidvae_b200 import _lib
    assert ops.gumbel_supported(32, 256) and not ops.gumbel_supported(32, 512) and not ops.gumbel_supported(48, 64)
    x = torch.zeros(4, 32, device="cuda")
    cb = torch.zeros(300, 32, device="cuda")
    with pytest.raises(_lib.HidvaeError, match="UNSUPPORTED"):
        ops.gumbel_apply(x, cb, 0.2, 0.25)
    with pytest.raises(_lib.HidvaeError, match="temperature"):
        ops.gumbel_apply(x, cb[:64].contiguous(), 0.0, 0.25)
    emb, ids, loss = ops.gumbel_apply(x[:0], cb[:64].contiguous(), 0.2, 0.25)
    assert emb.shape == (0, 32) and ids.shape == (0,) and loss.shape == (0,)


def test_hrqvae_gumbel_mode_levels_against_oracle(ops, monkeypatch):
    """HRqVae with codebook_mode = GUMBEL_SOFTMAX (the class default of the reference): the level loop calls the fused
    Gumbel kernels once per level (modules/h_rqvae.py:515-552).  The Philox seeds are pinned, the draws replayed through
    hv_gumbel_uniforms into the oracle's level loop: embeddings, ids, quantize loss and the gradient that reaches the
    encoder output must agree level by level."""
    from modules.h_rqvae import HRqVae
    from modules.quantize import QuantizeForwardMode
    torch.manual_seed(0)
    model = HRqVae(input_dim=64, embed_dim=32, hidden_dims=[48], codebook_size=128, codebook_kmeans_init=False,
                   codebook_normalize=True, codebook_mode=QuantizeForwardMode.GUMBEL_SOFTMAX, n_layers=3, n_cat_features=0,
                   commitment_weight=0.3).cuda().train()
    assert not model._can_fuse()                                  # Gumbel goes level by level
    n, temperature = 700, 0.2
    z = unit_rows(n, 32, seed=12).cuda().requires_grad_(True)
    seeds = iter([101, 202, 303])
    real_apply = ops.gumbel_apply
    monkeypatch.setattr(ops, "gumbel_apply", lambda x, cb, t, beta, uniforms=None, seed=None: real_apply(x, cb, t, beta, uniforms, next(seeds)))
    q = model.get_semantic_ids(z, gumbel_t=temperature)
    (q.embeddings.sum(dim=-1).pow(2).sum() + q.quantize_loss.sum()).backward()
    # oracle: the same three levels with the same uniforms
    z_o = z.detach().cpu().clone().requires_grad_(True)
    res, embs, ids, loss = z_o, [], [], 0.0
    for l, seed in enumerate((101, 202, 303)):
        cb = model.layers[l].effective_codebook().detach().cpu()
        u = ops.gumbel_uniforms(n, 128, seed, "cuda").cpu()
        out = O.quantize_level(res, cb, O.MODE_GUMBEL_SOFTMAX, 0.3, True, temperature, uniform=u)
        embs.append(out.embeddings), ids.append(out.ids)
        loss = loss + out.loss
        res = res - out.embeddings
    (torch.stack(embs, dim=-1).sum(dim=-1).pow(2).sum() + loss.sum()).backward()
    assert torch.equal(q.sem_ids.cpu(), torch.stack(ids, dim=1))
    # level l sees a residual that carries the round-off of the levels before it, amplified by 1 / T in the logits
    # (measured worst element: 1.0e-5 at level 2): 1e-4 for the chain, against 1e-5 for a single level (above)
    torch.testing.assert_close(q.embeddings.detach().cpu(), torch.stack(embs, dim=-1).detach(), rtol=1e-4, atol=2e-5)
    torch.testing.assert_close(q.quantize_loss.detach().cpu(), loss.detach(), rtol=1e-4, atol=2e-5)
    gs = float(z_o.grad.abs().max())
    torch.testing.assert_close(z.grad.cpu(), z_o.grad, rtol=1e-3, atol=1e-4 * gs)
    assert all(float(l.embedding.weight.grad.abs().sum()) > 0 for l in model.layers)
