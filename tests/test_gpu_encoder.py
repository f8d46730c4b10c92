"""GPU parity tests of the fused encoder MLP (hv_encoder_forward, csrc/enc_mlp.cu) through the C ABI.

Precision contract (include/hidvae_b200.h): operands rounded to fp16 -- the 11-bit significand of TF32, which is what the
reference's GPU path computes with (modules/h_rqvae.py:21) -- fp32 accumulation.  The bars below are therefore those of
a TF32 GEMM chain against the fp32 oracle: |z - z_oracle| <= 2e-3 on unit-norm outputs (measured 4e-4 .. 8e-4; a cuBLAS
TF32 chain measures 4e-4 on the same inputs), and >= 99 % of rows with all three semantic ids equal to the fp32 oracle's
(measured 99.7 %; the bf16 alternative would be 97.8 %)."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from helpers import make_codebooks, npz, ops, t
from oracle import encoder as OE
from oracle import rq as O

pytestmark = pytest.mark.gpu
DIMS = [768, 512, 256, 128, 32]
TOL = 2e-3


@pytest.fixture(scope="module")
def weights():
    return OE.seeded_weights(DIMS, 2024)


def _x(n, seed):
    g = torch.Generator().manual_seed(seed)
    return F.normalize(torch.randn(n, DIMS[0], generator=g), dim=-1)


@pytest.mark.parametrize("normalize", [0, 1])
@pytest.mark.parametrize("precise", [0, 1])
def test_golden_reference_mlp(ops, golden_dir, weights, normalize, precise):
    g = npz(golden_dir, "encoder.npz")
    image = ops.encoder_pack([w.cuda() for w in weights])
    z = ops.encoder_forward(t(g["x"]).cuda(), image, normalize=bool(normalize), precise_silu=bool(precise)).cpu()
    ref = t(g[f"z_norm{normalize}"])
    bar = TOL if normalize else TOL * float(ref.abs().max())
    assert float((z - ref).abs().max()) <= bar


@pytest.mark.parametrize("n", [1, 127, 128, 129, 5000, 148 * 128 * 2 + 61])
@pytest.mark.parametrize("normalize", [0, 1])
def test_vs_oracle_ragged_sizes(ops, weights, n, normalize):
    x = _x(n, n)
    image = ops.encoder_pack([w.cuda() for w in weights])
    z = ops.encoder_forward(x.cuda(), image, normalize=bool(normalize)).cpu()
    ref = OE.mlp_forward(x, weights, bool(normalize))
    assert z.shape == ref.shape
    bar = TOL if normalize else TOL * float(ref.abs().max())
    assert float((z - ref).abs().max()) <= bar


def test_empty_and_errors(ops, weights):
    from hidvae_b200._lib import HidvaeError
    image = ops.encoder_pack([w.cuda() for w in weights])
    assert ops.encoder_forward(torch.empty(0, 768, device="cuda"), image).shape == (0, 32)
    with pytest.raises(ValueError):
        ops.encoder_forward(torch.zeros(4, 512, device="cuda"), image)
    with pytest.raises(RuntimeError):
        ops.encoder_forward(torch.zeros(4, 768), image)          # CPU tensor: no fallback
    assert not ops.encoder_supported([768, 512, 256, 32])
    with pytest.raises(HidvaeError):
        ops.encoder_pack([torch.zeros(512, 768, device="cuda"), torch.zeros(32, 512, device="cuda")])


def test_large_activations_saturate_not_overflow(ops, weights):
    """Rows scaled far outside the unit sphere: fp16 operands saturate (cvt.satfinite) instead of producing inf / NaN."""
    x = _x(256, 5) * 3.0e5
    image = ops.encoder_pack([w.cuda() for w in weights])
    z = ops.encoder_forward(x.cuda(), image, normalize=True)
    assert bool(torch.isfinite(z).all())


def test_full_size_chunk_deterministic_and_close_to_fp32(ops, weights):
    """A 2^19-row chunk (28 tiles per CTA): two runs are bit-identical, rows agree with an fp32 matmul chain on the
    device, and the rows of the output are unit vectors."""
    n = 1 << 19
    x = F.normalize(torch.randn(n, 768, device="cuda", generator=torch.Generator("cuda").manual_seed(3)), dim=-1)
    ws = [w.cuda() for w in weights]
    image = ops.encoder_pack(ws)
    z1 = ops.encoder_forward(x, image, normalize=True)
    z2 = ops.encoder_forward(x, image, normalize=True)
    assert torch.equal(z1, z2)
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        h = x
        for l, w in enumerate(ws):
            h = h @ w.t()
            if l < 3:
                h = F.silu(h)
        ref = F.normalize(h, dim=-1)
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev
    assert float((z1 - ref).abs().max()) <= TOL
    torch.testing.assert_close(z1.norm(dim=-1), torch.ones(n, device="cuda"), rtol=1e-5, atol=1e-5)


def test_semantic_id_agreement_through_the_tokenizer(ops, weights):
    """precompute_corpus_ids with the fused encoder against the fp32 oracle (encoder + quantiser) on 65,536 items:
    rows with all ids equal >= 99 %; with encoder_precision='fp32' the same call is bit-exact outside near-ties."""
    from helpers import check_ids
    from modules.tokenizer.h_semids import HSemanticIdTokenizer
    n = 65536
    x = _x(n, 11)
    cbs = make_codebooks(3, 256, 32, seed=4)
    z_ref = OE.mlp_forward(x, weights, True)
    ids_ref = O.rq_forward(z_ref, [cbs[l] for l in range(3)], O.MODE_STE, 0.25, False).sem_ids
    agree = {}
    for prec in ("fused", "fp32"):
        tok = HSemanticIdTokenizer(input_dim=768, output_dim=32, hidden_dims=[512, 256, 128], codebook_size=256, n_layers=3,
                                   n_cat_feats=0, hrqvae_codebook_normalize=True, chunk_items=1 << 14,
                                   encoder_precision=prec).cuda()
        with torch.no_grad():
            for lin, w in zip([m for m in tok.hrq_vae.encoder.mlp if isinstance(m, torch.nn.Linear)], weights):
                lin.weight.copy_(w)
            for l, layer in enumerate(tok.hrq_vae.layers):
                layer.embedding.weight.copy_(cbs[l])      # level 0 is re-normalised by out_proj: rows are unit already
        ids = tok.precompute_corpus_ids(x.cuda()).cpu()
        agree[prec] = float((ids == ids_ref).all(dim=1).float().mean())
        if prec == "fp32":
            with torch.no_grad():
                z_gpu = tok.hrq_vae.encode(x.cuda()).cpu()
            eff = tok.hrq_vae.effective_codebooks().detach().cpu()
            check_ids(ids, z_gpu, eff, O.MODE_STE, 0.25, False)
    assert agree["fused"] >= 0.99, agree
    assert agree["fp32"] >= 0.999, agree


def test_module_uses_fused_kernel_only_for_inference(weights):
    """MLP.forward: fused under no_grad on CUDA, PyTorch layers (autograd) otherwise; the image follows weight updates."""
    from modules.encoder import MLP
    mlp = MLP(768, [512, 256, 128], 32, normalize=True).cuda()
    with torch.no_grad():
        for lin, w in zip([m for m in mlp.mlp if isinstance(m, torch.nn.Linear)], weights):
            lin.weight.copy_(w)
    x = _x(300, 2).cuda()
    y_train = mlp(x)                       # grad enabled: PyTorch layers
    assert y_train.requires_grad
    with torch.no_grad():
        assert mlp.fused_available(x)
        y = mlp(x)
        assert float((y - y_train).abs().max()) <= TOL
        y3 = mlp(x.reshape(3, 100, 768))
        assert y3.shape == (3, 100, 32) and torch.equal(y3.reshape(300, 32), y)
        mlp.mlp[0].weight.mul_(-1.0)       # in-place update bumps the version counter: the image is re-packed
        y_neg = mlp(x)
        mlp.inference_precision = "fp32"
        y_neg_ref = mlp(x)
        assert float((y_neg - y_neg_ref).abs().max()) <= TOL
        assert float((y_neg - y).abs().max()) > 0.05


@pytest.mark.parametrize("n", [1, 129, 5000, 148 * 128 + 77])
@pytest.mark.parametrize("normalize", [0, 1])
def test_half_precision_items_are_bit_identical_to_rounded_fp32_items(ops, weights, n, normalize):
    """hv_encoder_forward_f16: items stored as fp16.  The fp32 kernel rounds its items to fp16 (round to nearest even) before
    the first GEMM, so feeding x.half() must give the SAME z bit for bit -- and, like the fp32 call, stay within the TF32-grade
    bar of the fp32 oracle on the original items."""
    x = _x(n, 700 + n)
    image = ops.encoder_pack([w.cuda() for w in weights])
    z32 = ops.encoder_forward(x.cuda(), image, normalize=bool(normalize))
    z16 = ops.encoder_forward(x.cuda().half(), image, normalize=bool(normalize))
    assert z16.dtype == torch.float32 and torch.equal(z16, z32)
    z16r = ops.encoder_forward(x.half().float().cuda(), image, normalize=bool(normalize))   # the rounded items as fp32
    assert torch.equal(z16r, z32)
    ref = OE.mlp_forward(x, weights, bool(normalize))
    bar = TOL if normalize else TOL * float(ref.abs().max())
    assert float((z16.cpu() - ref).abs().max()) <= bar


def test_half_precision_catalogue_through_the_tokenizer(ops, weights):
    """precompute_corpus_ids on an fp16 catalogue (device tensor and pinned host tensor): the id table equals the fp32
    catalogue's bit for bit with the fused encoder; with encoder_precision='fp32' the items are widened and the PyTorch
    layers run (ids of the rounded items)."""
    from modules.tokenizer.h_semids import HSemanticIdTokenizer
    n = 20000
    x = _x(n, 12)
    cbs = make_codebooks(3, 256, 32, seed=4)
    tok = HSemanticIdTokenizer(input_dim=768, output_dim=32, hidden_dims=[512, 256, 128], codebook_size=256, n_layers=3,
                               n_cat_feats=0, hrqvae_codebook_normalize=True, chunk_items=1 << 13, encoder_precision="fused").cuda()
    with torch.no_grad():
        for lin, w in zip([m for m in tok.hrq_vae.encoder.mlp if isinstance(m, torch.nn.Linear)], weights):
            lin.weight.copy_(w)
        for l, layer in enumerate(tok.hrq_vae.layers):
            layer.embedding.weight.copy_(cbs[l])
    ids32 = tok.precompute_corpus_ids(x.cuda()).clone()
    ids16 = tok.precompute_corpus_ids(x.cuda().half()).clone()
    assert torch.equal(ids16, ids32)
    ids16_host = tok.precompute_corpus_ids(x.half().pin_memory()).clone()
    assert torch.equal(ids16_host, ids32)
    tok.hrq_vae.encoder.inference_precision = "fp32"
    ids_fp32_path = tok.precompute_corpus_ids(x.cuda().half())
    assert float((ids_fp32_path == ids32).all(dim=1).float().mean()) >= 0.99
