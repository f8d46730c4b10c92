"""The fused tag heads (csrc/tag_heads.cu: tag_gate_kernel, tag_gemm_kernel<KIND>, tag_pack_kernel) against a float64
reference that rounds where the kernel rounds, against the fp32 PyTorch heads, through the tokenizer, and for row
independence.

Reference (`emulate`): torch float64 on the device.  The gate runs in fp64 on the fp32 embeddings; g, every GEMM weight
and every stored activation are rounded to fp16 (through fp32, round to nearest even) where the kernel stores them; the
GEMMs, biases, LayerNorm (statistics of the unrounded pre-activation, applied to its fp16 copy, as the kernel's two
sweeps do), ReLU and residual adds run in fp64.  What the reference does not model is the fp32 accumulation order and the
fp32 gate / statistics, which make some stored activation round to the neighbouring fp16 value.

Logit bound (`logit_bound`), per row: B = 2^-8 * max_c (sum_j |W3[c, j]| |u_j| + |b3[c]|), u = the operand of the last
Linear.  It allows every element of u an error of 4 fp16 half-ulps relative (2^-12 each): 2 for rounding to the other
neighbour and 2 inherited from the same flips upstream, which LayerNorm renormalises at every stage; the fp32
accumulation (K <= 704 terms, 2^-24 each) is three orders below.  Worst |dlogit| / B measured on a B200: see
test_against_fp64 (printed as "fp64-ratio").  pred must equal the emulated argmax on every row whose emulated top-2 gap
exceeds 2 B, and equal the argmax of the kernel's own logits everywhere (first index on ties); conf must be within 1e-5
relative of 1 / sum exp(logit - max) over the kernel's logits in fp64.

Against the fp32 PyTorch heads (`tag_precision="torch"` with fp32 matmuls), the bound on the fused-minus-fp32 logit is
B32 = 2^-7 * max_c (sum_j |W3[c, j]| |u_j| + |b3[c]|) (the fp16 rounding of every operand, 2^-11 relative, through about
eight stored layers); every disagreement must be a row whose fp32 top-2 gap is below 2 B32, and at least 99 % of the
predictions of each level agree.
"""
import types

import pytest
import torch
import torch.nn.functional as F
from torch import nn

from helpers import profiled, shipped_kernels

D, FIRST_HIDDEN, COUNTS = 32, 512, (38, 168, 348)
N_FP64 = 148 * 128 + 77                     # crosses the 18,944-row sub-chunk boundary, ragged last tile
CHUNK_ROWS = 148 * 128
FAMILIES = ("tag_gate_kernel", "tag_gemm_kernel", "tag_pack_kernel")
KERNELS = {f"tag_gemm_kernel<{k}>" for k in range(5)} | {"tag_gate_kernel", "tag_pack_kernel"}
# which kernels a forward launches, by use_norm
LAUNCHED = {True: {"tag_gate_kernel", "tag_gemm_kernel<0>", "tag_gemm_kernel<1>", "tag_gemm_kernel<2>", "tag_gemm_kernel<4>"},
            False: {"tag_gate_kernel", "tag_gemm_kernel<2>", "tag_gemm_kernel<3>", "tag_gemm_kernel<4>"}}


def _model(norm: bool, seed: int = 0, counts=COUNTS, device="cuda"):
    from modules.h_rqvae import HRqVae
    torch.manual_seed(seed)
    m = HRqVae(input_dim=768, embed_dim=D, hidden_dims=[FIRST_HIDDEN, 256, 128], codebook_size=256, codebook_kmeans_init=False,
               n_layers=len(counts), tag_class_counts=list(counts), use_batch_norm=norm)
    return m.to(device).eval()


def _regime(model, regime: str, seed: int = 1):
    g = torch.Generator(device="cpu").manual_seed(seed)
    with torch.no_grad():
        for tp in model.tag_predictors:
            for mod in tp.modules():
                if regime == "trained" and isinstance(mod, nn.Linear):
                    mod.weight.mul_(torch.empty(1).uniform_(0.7, 1.6, generator=g).item())
                    mod.bias.copy_(torch.randn(mod.bias.shape, generator=g) * 0.1)
                if regime == "trained" and isinstance(mod, nn.LayerNorm):
                    mod.weight.copy_(torch.rand(mod.weight.shape, generator=g) + 0.5)
                    mod.bias.copy_(torch.randn(mod.bias.shape, generator=g) * 0.1)
            if regime == "ties":     # small spread; classes 0 and 1 almost equal and on top for most rows
                last = tp.classifier[7]
                last.weight.mul_(0.05)
                last.weight[1].copy_(last.weight[0] + torch.randn(last.weight.shape[1], generator=g).to(last.weight) * 1e-5)
                last.bias.zero_()
                last.bias[:2] = 1.0
    model._tag_image = None


def _emb(n: int, seed: int = 2, levels: int = 3):
    g = torch.Generator(device="cpu").manual_seed(seed)
    return (torch.randn((levels, n, D), generator=g) * 0.3).cuda()


def r16(t):
    return t.float().half().double()


def emulate(tp, emb, i, norm):
    """(logits, u) of TagPredictor tp at level i in fp64, rounding to fp16 where the kernel does."""
    P = lambda m: (m.weight.detach().double(), m.bias.detach().double())
    x = torch.cat([emb[l].double() for l in range(i + 1)], dim=-1)
    (w0, b0), (w1, b1), (w2, b2) = P(tp.attention[0]), P(tp.attention[2]), P(tp.attention[4])
    a = F.gelu(F.relu(x @ w0.T + b0) @ w1.T + b1)
    g = x * torch.sigmoid(a @ w2.T + b2)
    if i > 0:
        g = g / g.norm(dim=-1, keepdim=True).clamp_min(1e-12)
    h = r16(g)

    def lin(m, v):
        w, b = P(m)
        return v @ r16(w).T + b

    def ln(z, m):   # statistics of z, applied to its fp16 copy
        mu, var = z.mean(-1, keepdim=True), z.var(-1, unbiased=False, keepdim=True)
        return (r16(z) - mu) / torch.sqrt(var + 1e-5) * m.weight.double() + m.bias.double()

    fe = tp.feature_extractor
    z = lin(fe[0], h)
    h = r16(F.relu(ln(z, fe[1]))) if norm else r16(F.relu(z))
    for blk in (tp.residual_block1, tp.residual_block2):
        u = lin(blk[0], h)
        t = r16(F.relu(ln(u, blk[1]))) if norm else r16(F.relu(u))
        v = F.relu(lin(blk[4], t))
        h = r16(h + ln(v, blk[7])) if norm else r16(h + v)
    cl = tp.classifier
    z = lin(cl[0], h)
    t = r16(F.relu(ln(z, cl[1]))) if norm else r16(F.relu(z))
    u = r16(F.relu(lin(cl[4], t)))
    return lin(cl[7], u), u


def logit_bound(last: nn.Linear, u, scale):
    w = last.weight.detach().double().abs()
    return scale * ((u.abs() @ w.T) + last.bias.detach().double().abs()).amax(dim=-1)


def top2_gap(logits):
    t = logits.topk(2, dim=-1).values
    return t[:, 0] - t[:, 1]


def _fused(model, emb, logits=True):
    from hidvae_b200 import ops
    with torch.no_grad():
        image = model._fused_tag_image(emb)
        assert image is not None
        n = emb.shape[1]
        pred = torch.empty((n, len(COUNTS)), dtype=torch.int64, device="cuda")
        conf = torch.empty((n, len(COUNTS)), dtype=torch.float32, device="cuda")
        lg = [torch.empty((n, c), device="cuda") for c in COUNTS] if logits else None
        ops.tag_heads_forward(emb, image, pred, conf, lg)
    return pred, conf, lg


# ---------------------------------------------------------------------------------------------------------------------
# float64 reference
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("regime", ["init", "trained", "ties"])
@pytest.mark.parametrize("norm", [True, False], ids=["layernorm", "identity"])
def test_against_fp64(norm, regime):
    """Every level of the chain against `emulate`.  Each cell runs every kernel of its use_norm (LAUNCHED) and asserts so
    under torch.profiler."""
    model = _model(norm)
    model.tag_inference_precision = "fused"
    _regime(model, regime)
    emb = _emb(N_FP64)
    launched = profiled(lambda: _fused(model, emb))[1].names
    assert LAUNCHED[norm] <= launched, launched
    pred, conf, logits = _fused(model, emb)
    near_ties = 0
    for i, tp in enumerate(model.tag_predictors):
        ref, u = [], []
        for lo in range(0, N_FP64, 4096):
            r, uu = emulate(tp, emb[:, lo:lo + 4096], i, norm)
            ref.append(r), u.append(uu)
        ref, u = torch.cat(ref), torch.cat(u)
        bound = logit_bound(tp.classifier[7], u, 2.0 ** -8)
        ratio = ((logits[i].double() - ref).abs().amax(-1) / bound).max().item()
        print(f"fp64-ratio norm={norm} regime={regime} level={i}: {ratio:.3f}")
        assert ratio <= 1.0
        gap = top2_gap(ref)
        clear = gap > 2 * bound
        assert torch.equal(pred[clear, i], ref.argmax(-1)[clear])
        assert torch.equal(pred[:, i], logits[i].argmax(-1))
        lg = logits[i].double()
        want = 1.0 / torch.exp(lg - lg.amax(-1, keepdim=True)).sum(-1)
        assert ((conf[:, i].double() - want).abs() / want).max().item() <= 1e-5
        near_ties += int((~clear).sum())
    if regime == "ties":
        assert near_ties >= 1000, near_ties


# ---------------------------------------------------------------------------------------------------------------------
# against the fp32 PyTorch heads
# ---------------------------------------------------------------------------------------------------------------------
def _torch_heads(model, emb):
    """fp32 logits and last-Linear operands of the PyTorch heads (fp32 matmuls)."""
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        out = []
        with torch.no_grad():
            for i, tp in enumerate(model.tag_predictors):
                seen = {}
                hook = tp.classifier[7].register_forward_pre_hook(lambda m, a: seen.__setitem__("u", a[0]))
                logits = tp(torch.cat(list(emb[: i + 1]), dim=-1))
                hook.remove()
                out.append((logits, seen["u"]))
        return out
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev


@pytest.mark.gpu
@pytest.mark.parametrize("norm", [True, False], ids=["layernorm", "identity"])
def test_against_fp32_torch_heads(norm):
    model = _model(norm)
    _regime(model, "trained")
    model.tag_inference_precision = "fused"
    emb = _emb(65536, seed=5)
    pred, _conf, _lg = _fused(model, emb, logits=False)
    for i, (logits, u) in enumerate(_torch_heads(model, emb)):
        want = logits.argmax(-1)
        agree = (pred[:, i] == want).float().mean().item()
        b32 = logit_bound(model.tag_predictors[i].classifier[7], u.double(), 2.0 ** -7)
        bad = pred[:, i] != want
        print(f"fp32-agreement norm={norm} level={i}: {agree:.5f} ({int(bad.sum())} rows differ)")
        assert agree >= 0.99
        assert bool((top2_gap(logits.double())[bad] < 2 * b32[bad]).all())


@pytest.mark.gpu
def test_predict_tags_fused_matches_torch_default_and_seq_shape():
    model = _model(True)
    emb = _emb(4096, seed=7)
    x = torch.zeros(4096, 768, device="cuda")
    with torch.no_grad():
        base = model.predict_tags(x, level_embeddings=emb)
        model.tag_inference_precision = "fused"
        fused = model.predict_tags(x, level_embeddings=emb)
        seq = model.predict_tags(x.reshape(64, 64, 768), level_embeddings=emb)
    assert (fused["predictions"] == base["predictions"]).float().mean().item() >= 0.99
    assert torch.allclose(fused["confidences"], base["confidences"], rtol=2e-2, atol=2e-3)
    assert torch.equal(seq["predictions"].reshape(4096, -1), fused["predictions"])
    # training mode and autograd keep the PyTorch heads
    model.train()
    assert model._fused_tag_image(emb) is None
    model.eval()
    assert model._fused_tag_image(emb) is None  # grad mode is on here


# ---------------------------------------------------------------------------------------------------------------------
# through the tokenizer
# ---------------------------------------------------------------------------------------------------------------------
def _tokenizer(layout: str, tag_precision: str):
    from modules.tokenizer.h_semids import HSemanticIdTokenizer
    torch.manual_seed(0)
    t = HSemanticIdTokenizer(input_dim=768, output_dim=D, hidden_dims=[FIRST_HIDDEN, 256, 128], codebook_size=256, n_layers=3,
                             tag_class_counts=list(COUNTS), use_concatenated_ids=layout == "concatenated",
                             use_interleaved_ids=layout == "interleaved", chunk_items=1 << 15, tag_precision=tag_precision)
    return t.cuda()


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["concatenated", "interleaved"])
def test_tokenizer_tag_columns(layout):
    ref, fused = _tokenizer(layout, "torch").eval(), _tokenizer(layout, "fused").eval()
    _regime(ref.hrq_vae, "trained")
    fused.load_state_dict(ref.state_dict())
    g = torch.Generator(device="cpu").manual_seed(11)
    items = torch.randn((65536 + 5, 768), generator=g).cuda()
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        want = ref.precompute_corpus_ids(items)
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev
    got = fused.precompute_corpus_ids(items)
    sem, tag = fused._columns()
    assert torch.equal(got[:, sem], want[:, sem])
    for c in tag:
        assert (got[:, c] == want[:, c]).float().mean().item() >= 0.99
    # an fp16 catalogue (device and pinned host) gives the same table bit for bit
    assert torch.equal(fused.precompute_corpus_ids(items.half()), got)
    assert torch.equal(fused.precompute_corpus_ids(items.cpu().pin_memory()), got)
    assert torch.equal(fused.precompute_corpus_ids(items.half().cpu().pin_memory()), got)
    # uncached items: _ids_of_features (tokenizer.forward's branch) agrees with the cached rows
    with torch.no_grad():
        assert torch.equal(fused._ids_of_features(items[:777]), got[:777])


# ---------------------------------------------------------------------------------------------------------------------
# row independence, bounds, sentinels
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def big_run():
    model = _model(True)
    _regime(model, "trained")
    model.tag_inference_precision = "fused"
    n = (1 << 20) + 61
    emb = _emb(n, seed=13)
    pred, conf, _ = _fused(model, emb, logits=False)
    return model, emb, pred, conf


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 127, 128, 129, CHUNK_ROWS - 1, CHUNK_ROWS, CHUNK_ROWS + 1])
def test_prediction_does_not_depend_on_n(big_run, n):
    model, emb, pred, conf = big_run
    p, c, _ = _fused(model, emb[:, :n].contiguous(), logits=False)
    assert torch.equal(p, pred[:n]) and torch.equal(c, conf[:n])


@pytest.mark.gpu
def test_prediction_does_not_depend_on_position(big_run):
    model, emb, pred, conf = big_run
    n = 3 * CHUNK_ROWS + 5
    shifted = emb[:, 1000:1000 + n]                        # strided view: rows start mid-tile
    p, c, _ = _fused(model, shifted, logits=False)
    assert torch.equal(p, pred[1000:1000 + n]) and torch.equal(c, conf[1000:1000 + n])


@pytest.mark.gpu
def test_sentinels_and_nan_row(big_run):
    from hidvae_b200 import ops
    model, emb, pred, conf = big_run
    n = 5000
    e = emb[:, :n].clone()
    e[:, 17] = float("nan")
    table = torch.full((n + 9, 7), -7, dtype=torch.int64, device="cuda")
    confs = torch.full((n + 9, 7), -3.0, device="cuda")
    with torch.no_grad():
        ops.tag_heads_forward(e, model._fused_tag_image(e), table[:n, 1::2], confs[:n, 1::2])
    others = torch.ones(n + 9, 7, dtype=torch.bool, device="cuda")
    others[:n, 1::2] = False
    assert bool((table[others] == -7).all()) and bool((confs[others] == -3.0).all())
    keep = torch.ones(n, dtype=torch.bool, device="cuda")
    keep[17] = False
    assert torch.equal(table[:n, 1::2][keep], pred[:n][keep])
    assert torch.equal(confs[:n, 1::2][keep], conf[:n][keep])


# ---------------------------------------------------------------------------------------------------------------------
# instantiation coverage: every tag_* kernel of the library is asserted by a cell
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("kernel", sorted(KERNELS))
def test_kernel_cell(kernel):
    model = _model(kernel != "tag_gemm_kernel<3>")
    model.tag_inference_precision = "fused"
    emb = _emb(300, seed=3)
    model._tag_image = None
    names = profiled(lambda: _fused(model, emb, logits=False))[1].names   # packs (tag_pack_kernel) and runs
    assert kernel in names, names


def test_every_shipped_tag_kernel_has_a_cell():
    assert {k for k in shipped_kernels() if k.startswith("tag_")} == KERNELS


# ---------------------------------------------------------------------------------------------------------------------
# CPU: ABI validation, fallback, cache invalidation
# ---------------------------------------------------------------------------------------------------------------------
def test_abi_validation_without_a_gpu():
    import ctypes
    from hidvae_b200 import _lib
    lib = _lib.lib
    counts = (ctypes.c_int * 3)(*COUNTS)
    img = ctypes.c_size_t(0)
    assert lib.hv_tag_heads_workspace_bytes(3, D, FIRST_HIDDEN, counts, 1, 1000, ctypes.byref(img)) > 0 and img.value > 0
    assert lib.hv_tag_heads_workspace_bytes(3, 64, FIRST_HIDDEN, counts, 1, 1000, ctypes.byref(img)) == 0 and img.value == 0
    ws = lambda n: lib.hv_tag_heads_workspace_bytes(3, D, FIRST_HIDDEN, counts, 1, n, None)
    assert ws(CHUNK_ROWS) == ws(10 * CHUNK_ROWS) > ws(128) == ws(1)

    def fwd(n=10, d=D, emb=16, image=16, pred=16, ws_=16):
        return lib.hv_tag_heads_forward(emb, 0, D, n, 3, d, FIRST_HIDDEN, counts, 1, image, 1 << 30, pred, 1, 1, None, 0, 0,
                                        None, ws_, 1 << 30, None)
    assert fwd(n=-1) == _lib.HV_ERR_BAD_SHAPE
    assert fwd(d=64) == _lib.HV_ERR_UNSUPPORTED
    assert fwd(n=0, emb=None) == _lib.HV_OK
    assert fwd(emb=None) == _lib.HV_ERR_NULL
    assert fwd(pred=None) == _lib.HV_ERR_NULL
    assert fwd(image=24) == _lib.HV_ERR_MISALIGNED
    params = (ctypes.c_void_p * 3)(16, 16, 16)
    assert lib.hv_tag_heads_pack(params, 3, 3, D, FIRST_HIDDEN, counts, 1, 16, 1 << 30, None) == _lib.HV_ERR_BAD_SHAPE
    assert lib.hv_tag_heads_pack(params, 102, 3, 64, FIRST_HIDDEN, counts, 1, 16, 1 << 30, None) == _lib.HV_ERR_UNSUPPORTED


def test_unserved_shapes_and_cpu_calls_keep_pytorch():
    wide = _model(True, counts=(5, 6, 7), device="cpu")
    wide_shape = wide._tag_heads_shape()
    assert wide_shape == (D, FIRST_HIDDEN, [5, 6, 7], True)
    from modules.h_rqvae import HRqVae
    m = HRqVae(input_dim=768, embed_dim=64, hidden_dims=[512, 256, 128], codebook_size=16, codebook_kmeans_init=False,
               n_layers=3, tag_class_counts=[5, 6, 7]).eval()                      # E = 192 at level 2: not served
    assert m._tag_heads_shape() is None
    wide.tag_inference_precision = "fused"
    emb = torch.randn(3, 50, D)
    with torch.no_grad():
        assert wide._fused_tag_image(emb) is None                                 # CPU tensors
        got = wide.predict_tags(torch.zeros(50, 768), level_embeddings=emb)
        wide.tag_inference_precision = "torch"
        want = wide.predict_tags(torch.zeros(50, 768), level_embeddings=emb)
    assert torch.equal(got["predictions"], want["predictions"])
    wide.tag_inference_precision = "bogus"
    with pytest.raises(ValueError):
        wide._fused_tag_image(emb)


def test_in_place_weight_update_repacks(monkeypatch):
    from hidvae_b200 import ops
    packs = []
    monkeypatch.setattr(ops, "tag_heads_pack", lambda params, *shape: packs.append(shape) or object())
    model = _model(True, counts=(5, 6, 7), device="cpu")
    model.tag_inference_precision = "fused"
    fake = types.SimpleNamespace(is_cuda=True)
    with torch.no_grad():
        first = model._fused_tag_image(fake)
        assert model._fused_tag_image(fake) is first and len(packs) == 1
        model.tag_predictors[1].classifier[4].weight.add_(1.0)
        assert model._fused_tag_image(fake) is not first and len(packs) == 2
        model.tag_predictors[2].residual_block2[7].bias.zero_()
        model._fused_tag_image(fake)
    assert len(packs) == 3
