"""GPU parity tests of the fused residual quantiser, called through the C ABI (ctypes -> libhidvae_b200.so).

Checker = oracle/ (pinned to the reference by tests/golden) on the same seeded inputs.
Bars (BASELINE.json north_star / SURVEY.md section 8c):
  * semantic IDs bit-exact, except rows whose fp32 top-2 distance gap is < 1e-5 relative (tests/helpers.check_ids)
  * emb_out / residuals / loss / g_x: rtol 1e-5, atol 1e-6 (fp32)
  * codebook gradient: rtol 1e-4, atol 1e-5 (atomic accumulation order)
"""
import numpy as np
import pytest
import torch

from helpers import check_ids, make_codebooks, npz, oracle_levels, ops, t, unit_rows
from oracle import rq as O

pytestmark = pytest.mark.gpu

MODES = {"ste": O.MODE_STE, "rot": O.MODE_ROTATION_TRICK}
ALGOS = ["simt", "tcgen05"]
VAL = dict(rtol=1e-5, atol=1e-6)
GCB = dict(rtol=1e-4, atol=1e-5)


def _dev(x):
    return x.cuda()


def _run_forward(ops, x, cbs, mode, training, beta, algo):
    return ops.rq_forward(_dev(x), _dev(cbs), mode, training, beta, want_emb=True, want_residuals=True,
                          want_loss=True, want_level_loss=True, want_final_residual=True, algo=algo)


def _compare_values(out, ref, rows):
    """out: RqForwardResult on GPU ([L,N,D] layout); ref: oracle RqOutput ([N,D,L] layout); rows: bool mask."""
    emb = out.emb_out.cpu().permute(1, 2, 0)
    res = out.residuals.cpu().permute(1, 2, 0)
    torch.testing.assert_close(emb[rows], ref.embeddings[rows], **VAL)
    torch.testing.assert_close(res[rows], ref.residuals[rows], **VAL)
    torch.testing.assert_close(out.loss.cpu()[rows], ref.quantize_loss[rows], **VAL)
    for l, ll in enumerate(ref.level_losses):
        torch.testing.assert_close(out.level_loss.cpu()[l][rows], ll[rows], **VAL)
    final_ref = ref.residuals[:, :, -1] - ref.embeddings[:, :, -1]
    torch.testing.assert_close(out.final_residual.cpu()[rows], final_ref[rows], **VAL)


# ---------------------------------------------------------------------------------------------------------------
# golden fixtures recorded from the real reference
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("algo", ALGOS)
@pytest.mark.parametrize("mname", ["ste", "rot"])
@pytest.mark.parametrize("training", [0, 1])
def test_golden_rq_c1(ops, golden_dir, algo, mname, training):
    """HRqVae.get_semantic_ids of the reference (modules/h_rqvae.py:481-583), D=32 K=256 L=3, forward + backward."""
    g = npz(golden_dir, "rq_c1.npz")
    tag = f"{mname}_train{training}"
    enc, weights, beta = t(g[f"{tag}/enc"]), t(g[f"{tag}/weights"]), float(g[f"{tag}/beta"])
    ws = [weights[l].clone().requires_grad_(True) for l in range(weights.shape[0])]
    cbs = torch.stack([O.effective_codebook(w, normalize=(l == 0)) for l, w in enumerate(ws)])
    out = _run_forward(ops, enc, cbs.detach(), MODES[mname], bool(training), beta, algo)
    assert torch.equal(out.ids.cpu(), t(g[f"{tag}/sem_ids"]))
    torch.testing.assert_close(out.emb_out.cpu().permute(1, 2, 0), t(g[f"{tag}/embeddings"]), **VAL)
    torch.testing.assert_close(out.residuals.cpu().permute(1, 2, 0), t(g[f"{tag}/residuals"]), **VAL)
    torch.testing.assert_close(out.loss.cpu(), t(g[f"{tag}/quantize_loss"]), **VAL)
    # backward through the autograd Function, codebook gradient chained through out_proj by PyTorch
    x_d = _dev(enc).requires_grad_(True)
    ws_d = [_dev(w.detach()).requires_grad_(True) for w in ws]
    cbs_d = torch.stack([O.effective_codebook(w, normalize=(l == 0)) for l, w in enumerate(ws_d)])
    emb, _res, ids, loss, _ll = ops.rq_apply(x_d, cbs_d, MODES[mname], bool(training), beta, algo=algo)
    g_emb = _dev(t(g[f"{tag}/g_emb"]))  # [N, D, L]
    ((emb.permute(1, 2, 0) * g_emb).sum() + (loss * _dev(t(g[f"{tag}/g_loss"]))).sum()).backward()
    torch.testing.assert_close(x_d.grad.cpu(), t(g[f"{tag}/grad_enc"]), rtol=2e-5, atol=2e-6)
    for l, w in enumerate(ws_d):
        torch.testing.assert_close(w.grad.cpu(), t(g[f"{tag}/grad_weights"][l]), **GCB)


@pytest.mark.parametrize("algo", ALGOS)
@pytest.mark.parametrize("mname", ["ste", "rot"])
@pytest.mark.parametrize("normalize", [0, 1])
@pytest.mark.parametrize("training", [0, 1])
def test_golden_single_level(ops, golden_dir, algo, mname, normalize, training):
    """One Quantize.forward of the reference (modules/quantize.py:100-154): D=32, K=64, N=48."""
    g = npz(golden_dir, "quantize_levels.npz")
    tag = f"{mname}_norm{normalize}_train{training}"
    x, w, beta = t(g[f"{tag}/x"]), t(g[f"{tag}/weight"]), float(g[f"{tag}/beta"])
    x_d = _dev(x).requires_grad_(True)
    w_d = _dev(w).requires_grad_(True)
    cb = O.effective_codebook(w_d, bool(normalize)).unsqueeze(0)
    emb, _res, ids, loss, _ll = ops.rq_apply(x_d, cb, MODES[mname], bool(training), beta, algo=algo)
    assert torch.equal(ids.cpu().view(-1), t(g[f"{tag}/ids"]))
    torch.testing.assert_close(emb[0].cpu(), t(g[f"{tag}/emb_out"]), **VAL)
    torch.testing.assert_close(loss.cpu(), t(g[f"{tag}/loss"]), **VAL)
    ((emb[0] * _dev(t(g[f"{tag}/g_emb"]))).sum() + (loss * _dev(t(g[f"{tag}/g_loss"]))).sum()).backward()
    torch.testing.assert_close(x_d.grad.cpu(), t(g[f"{tag}/grad_x"]), rtol=2e-5, atol=2e-6)
    torch.testing.assert_close(w_d.grad.cpu(), t(g[f"{tag}/grad_weight"]), **GCB)


# ---------------------------------------------------------------------------------------------------------------
# oracle on seeded synthetic inputs (BASELINE.json configs 1 and 4 at oracle-friendly sizes) and edge shapes
# ---------------------------------------------------------------------------------------------------------------
SHAPES = [
    # (n, d, k, L)
    (1024, 32, 256, 3),   # config 1
    (2048, 64, 4096, 4),  # config 4 shape, reduced N
    (1, 32, 256, 3),      # single row (the reference's .squeeze() corner, quantize.py:45)
    (127, 32, 256, 3),    # ragged: less than one row tile
    (300, 16, 100, 2),    # K not a multiple of the MMA tile, ragged rows
    (513, 64, 300, 2),    # K spanning two N tiles with padding
    (257, 32, 8, 4),      # tiny codebook
]


@pytest.mark.parametrize("algo", ALGOS)
@pytest.mark.parametrize("mname,training", [("ste", 1), ("rot", 1), ("rot", 0)])
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "n%d_d%d_k%d_L%d" % s)
def test_forward_vs_oracle(ops, algo, mname, training, shape):
    n, d, k, L = shape
    x = unit_rows(n, d, seed=n + d)
    cbs = make_codebooks(L, k, d, seed=k + L)
    beta = 0.4
    out = _run_forward(ops, x, cbs, MODES[mname], bool(training), beta, algo)
    match = check_ids(out.ids, x, cbs, MODES[mname], beta, bool(training))
    assert match.float().mean() > 0.995, f"only {float(match.float().mean()):.4f} of rows match on every level"
    if n == 1 and mname == "rot" and training:
        return  # the reference's rotation transform squeezes the batch dim at N == 1 (quantize.py:45): ids only
    ref = oracle_levels(x, cbs, MODES[mname], beta, bool(training))
    rows = match & (out.ids.cpu() == ref.sem_ids).all(dim=1)
    _compare_values(out, ref, rows)


@pytest.mark.parametrize("algo", ["simt", "simt_diff", "tcgen05"])
def test_randn_codebooks_large_k(ops, algo):
    """config 4 variant with randn codebooks (SURVEY.md section 8d)."""
    n, d, k, L = 4096, 64, 4096, 4
    x = unit_rows(n, d, seed=5)
    cbs = make_codebooks(L, k, d, seed=6, kind="randn")
    out = ops.rq_forward(_dev(x), _dev(cbs), O.MODE_STE, False, 0.25, algo=algo)
    match = check_ids(out.ids, x, cbs, O.MODE_STE, 0.25, False)
    assert match.float().mean() > 0.995


def test_empty_batch(ops):
    x = torch.empty(0, 32, device="cuda")
    cbs = _dev(make_codebooks(3, 256, 32, seed=1))
    out = ops.rq_forward(x, cbs, O.MODE_STE, True, 0.25, want_emb=True, want_loss=True)
    assert out.ids.shape == (0, 3) and out.emb_out.shape == (3, 0, 32) and out.loss.shape == (0,)


def test_exact_ties_take_first_index(ops):
    """Duplicate code rows: the lowest index must win (torch.min semantics, modules/quantize.py:122)."""
    d, k = 32, 64
    cb = make_codebooks(1, k, d, seed=2)
    cb[0, 40] = cb[0, 7]
    cb[0, 63] = cb[0, 7]
    x = cb[0, 7].repeat(200, 1) + 1e-3 * unit_rows(200, d, seed=3)
    for algo in ALGOS:
        ids = ops.rq_encode(_dev(x), _dev(cb), algo=algo).cpu().view(-1)
        assert (ids == 7).all(), algo


def test_exact_ties_across_chunks_units_and_halves(ops):
    """The tensor-core scan folds a row's 256 scores into column classes and chunk maxima; a second maximiser in the
    same class (other chunk), the other 128-code unit, the other column half or the next operand image must all send
    the row down the exact first-index path."""
    d, k = 32, 512
    gen = torch.Generator().manual_seed(5)
    for first, dups in [(5, [37]), (5, [133]), (5, [69]), (5, [5 + 256]), (100, [101, 228, 300]), (200, [201]), (31, [32, 63, 64])]:
        cb = make_codebooks(1, k, d, seed=6)
        for j in dups:
            cb[0, j] = cb[0, first]
        x = cb[0, first].repeat(300, 1) + 1e-3 * torch.randn(300, d, generator=gen)
        for algo in ALGOS:
            ids = ops.rq_encode(_dev(x), _dev(cb), algo=algo).cpu().view(-1)
            assert (ids == first).all(), (algo, first, dups, ids.unique())


def test_zero_rows_and_mixed_batch(ops):
    """All-zero rows score -|c|^2/2 for every code (massive near-ties at a normalised level 0): the kernel must
    stay finite, pick a code of minimal norm, and leave the other rows of the same warp untouched."""
    n, d, k, L = 300, 32, 256, 3
    x = unit_rows(n, d, seed=41)
    x[::7] = 0.0
    cbs = make_codebooks(L, k, d, seed=42)
    out = ops.rq_forward(_dev(x), _dev(cbs), O.MODE_STE, False, 0.25, want_emb=True, want_loss=True, algo="tcgen05")
    ids = out.ids.cpu()
    nz = x.abs().sum(1) > 0
    check_ids(ids[nz], x[nz], cbs, O.MODE_STE, 0.25, False)
    assert torch.isfinite(out.loss).all() and torch.isfinite(out.emb_out).all()
    # zero rows: the chosen level-0 code has (near-)minimal norm among the codes
    nrm = (cbs[0] ** 2).sum(1)
    assert (nrm[ids[~nz, 0]] <= nrm.min() * (1 + 1e-5)).all()


def test_backward_gradient_replicas(ops):
    """Large N: the codebook gradient is scatter-added into replicas (workspace) and folded; same numbers as the
    direct scatter-add up to fp32 summation order, g_x bit-identical."""
    n, d, k, L = 40000, 32, 256, 3
    assert ops.lib.hv_workspace_bytes(1, n, d, k, L) > 0 and ops.lib.hv_workspace_bytes(1, 1024, d, k, L) == 0  # op 1 = backward
    x, cbs = _dev(unit_rows(n, d, 51)), _dev(make_codebooks(L, k, d, 52))
    gen = torch.Generator().manual_seed(53)
    g_emb, g_loss = _dev(torch.randn(L, n, d, generator=gen)), _dev(torch.randn(n, generator=gen))
    ids = ops.rq_encode(x, cbs)
    gx_a, gc_a = ops.rq_backward(x, cbs, ids, O.MODE_ROTATION_TRICK, True, 0.4, g_emb, g_loss, None)
    gx_b, gc_b = ops.rq_backward(x, cbs, ids, O.MODE_ROTATION_TRICK, True, 0.4, g_emb, g_loss, None, use_workspace=False)
    assert torch.equal(gx_a, gx_b)
    # ~150 randomly signed O(1) terms per code: fp32 sums in two different orders differ by ~1e-4 absolute
    torch.testing.assert_close(gc_a, gc_b, rtol=1e-3, atol=3e-4)
    # and against a dense fp64 scatter-add of the per-row terms 2 (e - r_l) g_loss of the level-0 codebook
    e0 = cbs[0][ids[:, 0]].double()
    ref0 = torch.zeros(k, d, dtype=torch.float64, device="cuda").index_add_(0, ids[:, 0], 2.0 * (e0 - x.double()) * g_loss.double()[:, None])
    torch.testing.assert_close(gc_a[0].double(), ref0, rtol=1e-3, atol=3e-4)
    torch.testing.assert_close(gc_b[0].double(), ref0, rtol=1e-3, atol=3e-4)


@pytest.mark.parametrize("algo", ALGOS)
def test_ids_out_strided(ops, algo):
    """ids may be written into a caller-provided [N, L] view (e.g. a column block of the [N, L + L_tags] table the
    tokenizer caches, modules/tokenizer/h_semids.py:134-178)."""
    n, d, k, L = 500, 32, 256, 3
    x, cbs = unit_rows(n, d, 9), make_codebooks(L, k, d, 10)
    table = torch.full((n, L + 2), -1, dtype=torch.int64, device="cuda")
    ops.rq_encode(_dev(x), _dev(cbs), algo=algo, ids_out=table[:, :L])
    ref = ops.rq_encode(_dev(x), _dev(cbs), algo=algo)
    assert torch.equal(table[:, :L], ref) and (table[:, L:] == -1).all()


# ---------------------------------------------------------------------------------------------------------------
# backward
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("algo", ["simt", "tcgen05"])
@pytest.mark.parametrize("mname,training", [("ste", 1), ("rot", 1), ("ste", 0)])
@pytest.mark.parametrize("shape", [(1024, 32, 256, 3), (777, 64, 512, 4), (64, 16, 32, 2)],
                         ids=lambda s: "n%d_d%d_k%d_L%d" % s)
def test_backward_vs_oracle_autograd(ops, algo, mname, training, shape):
    n, d, k, L = shape
    beta = 0.4
    x = unit_rows(n, d, seed=21)
    cbs = make_codebooks(L, k, d, seed=22)
    gen = torch.Generator().manual_seed(23)
    g_emb = torch.randn(n, d, L, generator=gen)
    g_loss = torch.randn(n, generator=gen)
    g_ll = torch.randn(L, n, generator=gen)
    # GPU
    x_d = _dev(x).requires_grad_(True)
    cb_d = _dev(cbs).requires_grad_(True)
    emb, _r, ids, loss, level_loss = ops.rq_apply(x_d, cb_d, MODES[mname], bool(training), beta, algo=algo)
    ((emb.permute(1, 2, 0) * _dev(g_emb)).sum() + (loss * _dev(g_loss)).sum() + (level_loss * _dev(g_ll)).sum()).backward()
    # oracle autograd on the rows whose ids agree (a near-tie row follows another code and so other gradients)
    x_o = x.clone().requires_grad_(True)
    cb_o = [cbs[l].clone().requires_grad_(True) for l in range(L)]
    ref = O.rq_forward(x_o, cb_o, MODES[mname], beta, bool(training))
    rows = (ids.cpu() == ref.sem_ids).all(dim=1)
    # these seeded inputs hold no near-tie: every id must agree, so the codebook gradients are ALWAYS compared
    assert bool(rows.all()), f"{int((~rows).sum())} rows follow another code than the oracle; pick seeds without near-ties"
    ((ref.embeddings * g_emb).sum() + (ref.quantize_loss * g_loss).sum()
     + sum((ll * g_ll[l]).sum() for l, ll in enumerate(ref.level_losses))).backward()
    # absolute bar relative to the gradient's scale: h = g_emb - G cancels operands of size |g|_max, so an element's error is
    # a few fp32 ulps of the LARGEST values involved, not of itself (worst element measured at D = 64, L = 4: 2.4e-6)
    torch.testing.assert_close(x_d.grad.cpu(), x_o.grad, rtol=2e-5, atol=1e-6 * max(1.0, float(x_o.grad.abs().max())))
    for l in range(L):
        torch.testing.assert_close(cb_d.grad.cpu()[l], cb_o[l].grad, **GCB)


@pytest.mark.parametrize("mname,training", [("ste", 1), ("rot", 1), ("ste", 0)])
@pytest.mark.parametrize("shape", [(65536 + 77, 32, 256, 3), (70001, 64, 128, 2), (66000, 16, 512, 3)],
                         ids=lambda s: "n%d_d%d_k%d_L%d" % s)
def test_backward_large_n_variant_equals_row_kernel(ops, mname, training, shape):
    """From 65,536 rows on (codebooks within 96 KB) the backward runs its shared-memory / prefetching kernel
    (rq_bwd_smem_kernel: four floats per lane, eight for the rotation trick).  The same rows in two calls below that size run the
    row kernel, which the oracle tests above pin: g_x must be bit-identical where the per-row expressions are the same, and
    equal up to the order of the row sums (eight floats per lane instead of four) for the rotation-trick kernel -- with the
    bar of the oracle comparison; the codebook gradient equal up to the order of the sums."""
    n, d, k, L = shape
    beta = 0.4
    x = _dev(unit_rows(n, d, seed=51))
    cbs = _dev(make_codebooks(L, k, d, seed=52))
    gen = torch.Generator().manual_seed(53)
    g_emb = _dev(torch.randn(L, n, d, generator=gen))
    g_loss = _dev(torch.randn(n, generator=gen))
    mode = MODES[mname]
    ids = ops.rq_encode(x, cbs)
    gx, gcb = ops.rq_backward(x, cbs, ids, mode, bool(training), beta, g_emb, g_loss, None)
    h = n // 2
    gx_a, gcb_a = ops.rq_backward(x[:h], cbs, ids[:h], mode, bool(training), beta, g_emb[:, :h].contiguous(), g_loss[:h], None)
    gx_b, gcb_b = ops.rq_backward(x[h:], cbs, ids[h:], mode, bool(training), beta, g_emb[:, h:].contiguous(), g_loss[h:], None)
    gx_rows = torch.cat([gx_a, gx_b])
    if mname == "rot" and training:
        torch.testing.assert_close(gx, gx_rows, rtol=2e-5, atol=1e-6 * max(1.0, float(gx_rows.abs().max())))
    else:
        assert torch.equal(gx, gx_rows)
    ref = gcb_a + gcb_b
    torch.testing.assert_close(gcb, ref, rtol=1e-4, atol=1e-4 * float(ref.abs().max()))


@pytest.mark.parametrize("mname", ["ste", "rot"])
@pytest.mark.parametrize("shape", [(65536 + 77, 32, 256, 3), (66001, 64, 128, 2)], ids=lambda s: "n%d_d%d_k%d_L%d" % s)
def test_backward_large_n_variant_vs_oracle_autograd(ops, mname, shape):
    """The shared-memory backward kernel (from 65,536 rows on; four floats per lane, eight for the rotation trick) against
    the oracle's autograd directly, on the oracle's own ids (so that no near-tie row can follow another code)."""
    n, d, k, L = shape
    beta = 0.4
    x = unit_rows(n, d, seed=61)
    cbs = make_codebooks(L, k, d, seed=62)
    gen = torch.Generator().manual_seed(63)
    g_emb = torch.randn(n, d, L, generator=gen)
    g_loss = torch.randn(n, generator=gen)
    x_o = x.clone().requires_grad_(True)
    cb_o = [cbs[l].clone().requires_grad_(True) for l in range(L)]
    ref = O.rq_forward(x_o, cb_o, MODES[mname], beta, True)
    ((ref.embeddings * g_emb).sum() + (ref.quantize_loss * g_loss).sum()).backward()
    gx, gcb = ops.rq_backward(_dev(x), _dev(cbs), _dev(ref.sem_ids), MODES[mname], True, beta,
                              _dev(g_emb.permute(2, 0, 1).contiguous()), _dev(g_loss), None)
    torch.testing.assert_close(gx.cpu(), x_o.grad, rtol=2e-5, atol=1e-6 * max(1.0, float(x_o.grad.abs().max())))
    for l in range(L):   # sums of ~n / k terms per code: the bar scales with the gradient
        torch.testing.assert_close(gcb.cpu()[l], cb_o[l].grad, rtol=1e-4, atol=1e-5 * max(1.0, float(cb_o[l].grad.abs().max())))


def test_backward_broadcast_grad(ops):
    """The decoder consumes embs.sum(-1) (modules/h_rqvae.py:607): its gradient reaches the kernel as a
    level-broadcast view (level stride 0), and mean() makes g_loss a stride-0 scalar."""
    n, d, k, L = 512, 32, 256, 3
    x, cbs = unit_rows(n, d, 31), make_codebooks(L, k, d, 32)
    tgt = unit_rows(n, d, 33)
    x_d = _dev(x).requires_grad_(True)
    cb_d = _dev(cbs).requires_grad_(True)
    emb, _r, ids, loss, _ll = ops.rq_apply(x_d, cb_d, O.MODE_ROTATION_TRICK, True, 0.4, algo="simt")
    (((emb.permute(1, 2, 0).sum(-1) - _dev(tgt)) ** 2).sum() + loss.mean()).backward()
    x_o = x.clone().requires_grad_(True)
    cb_o = [cbs[l].clone().requires_grad_(True) for l in range(L)]
    ref = O.rq_forward(x_o, cb_o, O.MODE_ROTATION_TRICK, 0.4, True)
    assert torch.equal(ids.cpu(), ref.sem_ids)
    (((ref.embeddings.sum(-1) - tgt) ** 2).sum() + ref.quantize_loss.mean()).backward()
    torch.testing.assert_close(x_d.grad.cpu(), x_o.grad, rtol=2e-5, atol=2e-6)
    for l in range(L):
        torch.testing.assert_close(cb_d.grad.cpu()[l], cb_o[l].grad, **GCB)


# ---------------------------------------------------------------------------------------------------------------
# full-size, size-independent properties (BASELINE.json configs 4 and 5 shapes)
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape", [(65536, 64, 4096, 4), (1 << 20, 32, 256, 3), (38000 + 77, 64, 1500, 2)],
                         ids=["config4", "config5_chunk", "streamed_two_tiles_per_cta_ragged"])
def test_full_size_properties(ops, shape):
    """(the third shape: streamed operand images with two row tiles per CTA and one MMA issuer per warpgroup, an odd number
    of row tiles -- the last group's second tile is empty --, a ragged last tile and a padded last operand image)"""
    n, d, k, L = shape
    x = _dev(unit_rows(n, d, seed=41))
    cbs = _dev(make_codebooks(L, k, d, seed=42))
    out = ops.rq_forward(x, cbs, O.MODE_STE, False, 0.25, want_emb=True, want_loss=True, want_final_residual=True,
                         algo="tcgen05")
    ids = out.ids
    assert int(ids.min()) >= 0 and int(ids.max()) < k
    # (1) reconstruction identity: x - sum_l C_l[id_l] == final residual, emb_out_l == C_l[id_l] (eval semantics)
    r = x.clone()
    loss = torch.zeros(n, device="cuda")
    for l in range(L):
        e = cbs[l][ids[:, l]]
        torch.testing.assert_close(out.emb_out[l], e, rtol=0, atol=0)
        loss += 1.25 * ((r - e) ** 2).sum(-1)
        r = r - e
    torch.testing.assert_close(out.final_residual, r, **VAL)
    torch.testing.assert_close(out.loss, loss, **VAL)
    # (2) optimality: no code is closer than the chosen one by more than the near-tie allowance (checked with an
    #     fp32 torch table on a strided sample of rows, level 0)
    sample = torch.arange(0, n, max(1, n // 8192), device="cuda")
    table = ((x[sample] ** 2).sum(1, keepdim=True) + (cbs[0] ** 2).sum(1)[None] - 2 * x[sample] @ cbs[0].T)
    best = table.min(dim=1).values
    chosen = table.gather(1, ids[sample, :1]).view(-1)
    assert bool(((chosen - best) <= 1e-5 * best.abs() + 1e-7).all())
    # (3) the exact-fp32 CUDA-core kernel and the tensor-core kernel agree on (almost) every row
    ids_simt = ops.rq_encode(x[: 1 << 16], cbs, algo="simt")
    agree = (ids_simt == ids[: 1 << 16]).all(dim=1).float().mean()
    assert float(agree) > 0.999, float(agree)
    # (4) oracle on a 4096-row sample
    rows = torch.arange(0, n, n // 4096)[:4096]
    match = check_ids(ids[rows.cuda()], x[rows.cuda()].cpu(), cbs.cpu(), O.MODE_STE, 0.25, False)
    assert match.float().mean() > 0.995


# ---------------------------------------------------------------------------------------------------------------
# the resident-codebook kernel (D = 32, K <= 256, L <= 3: rows owned by threads, A operand in tensor memory, issuer warp,
# three shared accumulators): shapes around its unit / padding boundaries and long accumulator rings
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [8, 100, 128, 129, 200, 256])
@pytest.mark.parametrize("L", [1, 2, 3])
def test_resident_kernel_codebook_sizes(ops, k, L):
    """K below / at / above one 128-code unit (padded codes can never win, an all-padding unit 1 must lose to unit 0)."""
    n, d = 1000 + 37 * L + k, 32
    x = unit_rows(n, d, seed=k + L)
    cbs = make_codebooks(L, k, d, seed=3 * k + L)
    out = _run_forward(ops, x, cbs, O.MODE_ROTATION_TRICK, True, 0.4, "tcgen05")
    assert int(out.ids.max()) < k and int(out.ids.min()) >= 0
    match = check_ids(out.ids, x, cbs, O.MODE_ROTATION_TRICK, 0.4, True)
    assert match.float().mean() > 0.995
    ref = oracle_levels(x, cbs, O.MODE_ROTATION_TRICK, 0.4, True)
    _compare_values(out, ref, match & (out.ids.cpu() == ref.sem_ids).all(dim=1))


def test_resident_kernel_ties_across_units(ops):
    """Duplicate code rows inside a 16-column chunk, in another chunk of the same column class, and in the other unit:
    the lowest index wins (the unit-0 candidate keeps ties against unit 1)."""
    d, k = 32, 256
    gen = torch.Generator().manual_seed(11)
    for first, dups in [(5, [6]), (5, [21]), (5, [133]), (100, [116, 228]), (127, [128]), (0, [255]), (130, [131, 146, 250])]:
        cb = make_codebooks(3, k, d, seed=9)
        for j in dups:
            cb[0, j] = cb[0, first]
        x = cb[0, first].repeat(300, 1) + 1e-3 * torch.randn(300, d, generator=gen)
        ids = ops.rq_encode(_dev(x), _dev(cb), algo="tcgen05").cpu()
        assert (ids[:, 0] == first).all(), (first, dups, ids[:, 0].unique())


@pytest.mark.parametrize("training", [0, 1])
def test_resident_kernel_many_tiles_per_warpgroup(ops, training):
    """~13 row tiles per CTA: the request queue, the unit counter and the three accumulators wrap many times; every
    row must agree with the exact fp32 CUDA-core kernel (ids up to documented near-ties, values where ids agree)."""
    n, d, k, L = 148 * 128 * 13 + 77, 32, 256, 3
    x = _dev(unit_rows(n, d, seed=77))
    cbs = _dev(make_codebooks(L, k, d, seed=78))
    kw = dict(want_emb=True, want_loss=True) if training else {}
    a = ops.rq_forward(x, cbs, O.MODE_ROTATION_TRICK, bool(training), 0.4, algo="tcgen05", **kw)
    b = ops.rq_forward(x, cbs, O.MODE_ROTATION_TRICK, bool(training), 0.4, algo="simt", **kw)
    same = (a.ids == b.ids).all(dim=1)
    assert float(same.float().mean()) > 0.999
    # reconstruction identity on every row, whatever the ids: x - sum_l C_l[id_l] (eval) is what the next level saw
    if training:
        torch.testing.assert_close(a.emb_out[:, same], b.emb_out[:, same], **VAL)
        torch.testing.assert_close(a.loss[same], b.loss[same], **VAL)
    # rows that differ must be near-ties: check them against the oracle on a sample
    bad = torch.nonzero(~same).view(-1)[:512].cpu()
    if bad.numel():
        check_ids(a.ids[bad.cuda()], x[bad.cuda()].cpu(), cbs.cpu(), O.MODE_ROTATION_TRICK, 0.4, bool(training))


@pytest.mark.parametrize("shape", [(300000, 32, 256, 3), (40000, 64, 1500, 2)], ids=["row_owner_kernel", "streamed_kernel"])
def test_repeated_launches_are_bit_identical(ops, shape):
    """The forward kernels hand tiles, accumulators and turns around through barriers: twelve launches on the same rows must
    give the same ids (both kernels) and the same emb_out / loss bit for bit -- any race in the hand-overs would show up here."""
    n, d, k, L = shape
    x = _dev(unit_rows(n, d, seed=71))
    cbs = _dev(make_codebooks(L, k, d, seed=72))
    packed = ops.pack_codebooks(cbs)
    ids0 = ops.rq_encode(x, cbs, packed=packed).clone()
    out0 = ops.rq_forward(x, cbs, O.MODE_ROTATION_TRICK, True, 0.4, want_emb=True, want_loss=True, packed=packed)
    emb0, loss0, tids0 = out0.emb_out.clone(), out0.loss.clone(), out0.ids.clone()
    assert torch.equal(tids0[:, 0], ids0[:, 0])   # (later levels differ by design: training subtracts the rotated value)
    for it in range(12):
        assert torch.equal(ops.rq_encode(x, cbs, packed=packed), ids0), f"encode, launch {it}"
        out = ops.rq_forward(x, cbs, O.MODE_ROTATION_TRICK, True, 0.4, want_emb=True, want_loss=True, packed=packed)
        assert torch.equal(out.ids, tids0), f"training ids, launch {it}"
        assert torch.equal(out.emb_out, emb0) and torch.equal(out.loss, loss0), f"training values, launch {it}"


@pytest.mark.parametrize("cfg", [(32, 256, 3), (64, 1500, 2)], ids=["row_owner_kernel", "streamed_kernel"])
def test_row_counts_around_tile_and_wave_boundaries(ops, cfg):
    """Row counts around one tile, the three tiles a CTA keeps in flight, one wave of 148 CTAs and the switch from one to two
    (streamed kernel) / three (row-owner kernel) tiles per CTA: the tensor-core ids must match the exact-fp32 CUDA-core kernel
    on (almost) every row, and rows beyond n must never be written."""
    d, k, L = cfg
    cbs = _dev(make_codebooks(L, k, d, seed=81))
    packed = ops.pack_codebooks(cbs)
    wave = 148 * 128
    for n in (1, 2, 127, 128, 129, 255, 257, 383, 385, 512, wave - 1, wave, wave + 1, 2 * wave + 5, 3 * wave + 127, 4 * wave - 129):
        x = _dev(unit_rows(n, d, seed=n % 1000))
        table = torch.full((n + 3, L), -7, dtype=torch.int64, device="cuda")
        ops.rq_encode(x, cbs, packed=packed, ids_out=table[:n])
        assert bool((table[n:] == -7).all()), n
        ids = table[:n]
        assert int(ids.min()) >= 0 and int(ids.max()) < k, n
        ref = ops.rq_encode(x, cbs, algo="simt")
        agree = float((ids == ref).all(dim=1).float().mean())
        assert agree >= (0.998 if n > 1000 else 0.97), (n, agree)
