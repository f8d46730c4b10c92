"""Gumbel-softmax levels under CUDA graphs: the Philox pair (seed, offset) in device memory (hv_gumbel_*_devrng,
csrc/gumbel.cu) and the seed that `ops.gumbel_apply` draws on the device while a graph is captured.

* CPU: the three entries are exported and bound, reject bad arguments before any CUDA call, and the ops layer rejects a
  malformed tensor seed; the library ships the same Gumbel kernel instantiations, and the kernels spill no more than before.
* A device pair gives the host pair's draw: uniforms, emb_out, ids, loss, lse and g_x bit for bit, g_codebook within the bar
  of tests/test_gpu_gumbel.py (its atomics add in a free order).
* A captured gumbel_apply draws a new seed at every replay, and each replay equals the eager call with the seed it drew.
* HRqVae in Gumbel mode as a captured level loop, under GraphedTrainStep (fused K = 128 and the dense K = 512 path), and the
  trainer with use_cuda_graph = True."""
import os
import re
import subprocess

import numpy as np
import pytest
import torch

from helpers import ROOT, family, lib_mod, ops, shipped_kernels, unit_rows

PKG = os.path.join(ROOT, "hid-vae_b200")
NEW_ENTRIES = ("hv_gumbel_uniforms_devrng", "hv_gumbel_forward_devrng", "hv_gumbel_backward_devrng")
SEED, OFFSET = 0x2F3A5B7C9D1E4F60, (1 << 33) + 12345      # the offset carries into the counter's high word
CB_BAR = dict(rtol=1e-4)                                  # g_codebook: + atol 1e-5 x its scale (tests/test_gpu_gumbel.py)
FAMILIES = ("gumbel_fwd_kernel", "gumbel_bwd_kernel", "gumbel_uniforms_kernel")
KERNEL = r"(gumbel_(?:fwd|bwd|uniforms)_kernel(?:ILi\d+EE)?)"                # mangled, as -Xptxas -v prints it


def _cb_close(a, b):
    torch.testing.assert_close(a, b, atol=1e-5 * float(b.abs().max()), **CB_BAR)


# ---------------------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------------------
def test_devrng_entries_are_declared_exported_and_bound(lib_mod):
    import ctypes
    header = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "hidvae_b200.h")).read(), flags=re.S)
    raw = ctypes.CDLL(lib_mod.LIB_PATH)
    for name in NEW_ENTRIES:
        assert re.search(r"\b%s\s*\(" % name, header), name
        assert hasattr(raw, name) and name in lib_mod.SIGNATURES, name


def test_devrng_argument_errors_before_any_cuda_call(lib_mod):
    """Fake, aligned device addresses: every call below must return before it touches them or the device."""
    L = lib_mod.lib
    x, cb, emb, lse, gx, gcb, u = 4096, 8192, 12288, 16384, 20480, 24576, 28672
    fwd = lambda n, d, rng: L.hv_gumbel_forward_devrng(x, n, d, cb, 64, 0.2, 0.25, None, rng, emb, None, None, lse, None)
    bwd = lambda n, d, rng: L.hv_gumbel_backward_devrng(x, n, d, cb, 64, 0.2, 0.25, None, rng, emb, lse, None, None, gx, gcb,
                                                         None)
    for call in (fwd, bwd):
        assert call(8, 32, None) == lib_mod.HV_ERR_NULL and "rng" in lib_mod.last_error()
        assert call(-1, 32, None) == lib_mod.HV_ERR_BAD_SHAPE and "bad shape" in lib_mod.last_error()
        assert call(8, 48, 256) == lib_mod.HV_ERR_UNSUPPORTED and "D=48" in lib_mod.last_error()
        assert call(0, 32, None) == lib_mod.HV_OK                          # n = 0: a no-op, rng not needed
    assert L.hv_gumbel_forward_devrng(x, 8, 32, cb, 64, 0.0, 0.25, None, 256, emb, None, None, lse, None) == \
        lib_mod.HV_ERR_BAD_SHAPE and "temperature" in lib_mod.last_error()
    assert L.hv_gumbel_uniforms_devrng(8, 64, None, u, None) == lib_mod.HV_ERR_NULL
    assert L.hv_gumbel_uniforms_devrng(-1, 64, 256, u, None) == lib_mod.HV_ERR_BAD_SHAPE
    assert L.hv_gumbel_uniforms_devrng(8, 0, 256, u, None) == lib_mod.HV_ERR_BAD_SHAPE
    assert L.hv_gumbel_uniforms_devrng(0, 64, None, None, None) == lib_mod.HV_OK


@pytest.mark.parametrize("seed", [torch.tensor([1, 0]), torch.tensor([1, 0], dtype=torch.int32), torch.tensor([1, 0, 0]),
                                  torch.tensor([1.0, 0.0])], ids=["cpu", "int32", "three", "float"])
def test_ops_reject_a_malformed_tensor_seed(ops, seed):
    x, cb = torch.zeros(4, 32), torch.zeros(64, 32)
    with pytest.raises(ValueError, match="CUDA int64 tensor of two elements"):
        ops.gumbel_apply(x, cb, 0.2, 0.25, seed=seed)
    with pytest.raises(ValueError, match="CUDA int64 tensor of two elements"):
        ops.gumbel_uniforms(4, 64, seed)


def test_same_gumbel_kernel_instantiations(lib_mod):
    """The device pair is a runtime pointer: the library ships the Gumbel instantiations it shipped before."""
    assert {k for k in shipped_kernels() if family(k) in FAMILIES} == \
        {f"gumbel_{f}_kernel<{d}>" for f in ("fwd", "bwd") for d in (16, 32, 64)} | {"gumbel_uniforms_kernel"}


def test_gumbel_kernels_spill_no_more_than_before(tmp_path):
    """-Xptxas -v of csrc/gumbel.cu: the forward kernels and the backward at D = 16 / 32 do not spill, the backward at D = 64
    spills at most the 232 bytes it spilled with host seeds only (CUDA 12.9; its row loop holds x, ge, v and a code in
    registers).  The backward keeps the device pair in shared memory for this reason."""
    nvcc = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "nvcc")
    if not os.path.isfile(nvcc):
        pytest.skip("nvcc not found")
    out = subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xptxas", "-v", "-c",
                          os.path.join(PKG, "csrc", "gumbel.cu"), "-o", str(tmp_path / "gumbel.o")],
                         check=True, capture_output=True, text=True).stderr
    spills = dict(re.findall(r"Function properties for \S*?%s\S*\s+\d+ bytes stack frame, (\d+) bytes spill stores" % KERNEL,
                             out))
    assert len(spills) == 7, out
    for name, nbytes in spills.items():
        assert int(nbytes) <= (232 if name == "gumbel_bwd_kernelILi64EE" else 0), (name, nbytes)


# ---------------------------------------------------------------------------------------------------------------------
# GPU: device pair == host pair
# ---------------------------------------------------------------------------------------------------------------------
def _level(lib_mod, x, cb, g_emb, g_loss, temperature=0.2, beta=0.3, host=None, rng=None, uniforms=None):
    """One forward + backward through the raw C entries: host=(seed, offset) or rng = the device pair."""
    L = lib_mod.lib
    n, d = x.shape
    k = cb.shape[0]
    emb, gx = torch.empty_like(x), torch.empty_like(x)
    ids = torch.empty(n, dtype=torch.int64, device=x.device)
    loss, lse = (torch.empty(n, device=x.device) for _ in range(2))
    gcb = torch.zeros_like(cb)
    up = uniforms.data_ptr() if uniforms is not None else None
    s = torch.cuda.current_stream().cuda_stream
    if rng is None:
        lib_mod.check(L.hv_gumbel_forward(x.data_ptr(), n, d, cb.data_ptr(), k, temperature, beta, up, host[0], host[1],
                                          emb.data_ptr(), ids.data_ptr(), loss.data_ptr(), lse.data_ptr(), s))
        lib_mod.check(L.hv_gumbel_backward(x.data_ptr(), n, d, cb.data_ptr(), k, temperature, beta, up, host[0], host[1],
                                           emb.data_ptr(), lse.data_ptr(), g_emb.data_ptr(), g_loss.data_ptr(), gx.data_ptr(),
                                           gcb.data_ptr(), s))
    else:
        lib_mod.check(L.hv_gumbel_forward_devrng(x.data_ptr(), n, d, cb.data_ptr(), k, temperature, beta, up, rng.data_ptr(),
                                                 emb.data_ptr(), ids.data_ptr(), loss.data_ptr(), lse.data_ptr(), s))
        lib_mod.check(L.hv_gumbel_backward_devrng(x.data_ptr(), n, d, cb.data_ptr(), k, temperature, beta, up, rng.data_ptr(),
                                                  emb.data_ptr(), lse.data_ptr(), g_emb.data_ptr(), g_loss.data_ptr(),
                                                  gx.data_ptr(), gcb.data_ptr(), s))
    return dict(emb=emb, ids=ids, loss=loss, lse=lse, g_x=gx, g_codebook=gcb)


def _assert_same(a, b, what):
    for name in ("emb", "ids", "loss", "lse", "g_x"):
        assert torch.equal(a[name], b[name]), f"{what}: {name}"
    _cb_close(a["g_codebook"], b["g_codebook"])


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 33, 4097, 65537])
@pytest.mark.parametrize("k", [1, 64, 256])
@pytest.mark.parametrize("d", [16, 32, 64])
def test_device_pair_equals_host_pair(lib_mod, ops, d, k, n):
    gen = torch.Generator().manual_seed(d * 1000 + k + n)
    x = unit_rows(n, d, seed=n + d).cuda()
    cb = torch.nn.functional.normalize(torch.rand(k, d, generator=gen), dim=-1).cuda()
    g_emb = (torch.randn(n, d, generator=gen) * 0.1).cuda()
    g_loss = (torch.rand(n, generator=gen) / n).cuda()
    rng = torch.tensor([SEED, OFFSET], dtype=torch.int64, device="cuda")
    u_host = torch.empty(n, k, device="cuda")
    lib_mod.check(lib_mod.lib.hv_gumbel_uniforms(n, k, SEED, OFFSET, u_host.data_ptr(), torch.cuda.current_stream().cuda_stream))
    u_dev = ops.gumbel_uniforms(n, k, rng)
    assert torch.equal(u_dev, u_host)
    host = _level(lib_mod, x, cb, g_emb, g_loss, host=(SEED, OFFSET))
    dev = _level(lib_mod, x, cb, g_emb, g_loss, rng=rng)
    _assert_same(dev, host, "device pair vs host pair")
    # both regenerate the recorded draw in the backward: the same level with that draw given explicitly
    _assert_same(_level(lib_mod, x, cb, g_emb, g_loss, host=(0, 0), uniforms=u_dev), dev, "explicit draw vs device pair")
    if n > 1:   # the offset moves the draw
        assert not torch.equal(ops.gumbel_uniforms(n, k, torch.tensor([SEED, 0], device="cuda")), u_dev)


@pytest.mark.gpu
def test_ops_device_seed_through_autograd(ops):
    """gumbel_apply with a tensor seed equals the int seed (offset 0) through autograd; the pair must be on x's device and
    well formed."""
    n, d, k = 3000, 32, 256
    x = unit_rows(n, d, seed=4).cuda()
    cb = torch.nn.functional.normalize(torch.rand(k, d, generator=torch.Generator().manual_seed(5)), dim=-1).cuda()
    outs = []
    for seed in (SEED, torch.tensor([SEED, 0], device="cuda")):
        xd, cbd = x.clone().requires_grad_(True), cb.clone().requires_grad_(True)
        emb, ids, loss = ops.gumbel_apply(xd, cbd, 0.2, 0.25, seed=seed)
        (emb.pow(2).sum() + loss.sum()).backward()
        outs.append((emb.detach(), ids, loss.detach(), xd.grad, cbd.grad))
    for name, a, b in zip(("emb", "ids", "loss", "g_x"), outs[0], outs[1]):
        assert torch.equal(a, b), name
    _cb_close(outs[1][4], outs[0][4])
    for bad in (torch.tensor([1, 0], dtype=torch.int32, device="cuda"), torch.tensor([1, 0, 0], device="cuda")):
        with pytest.raises(ValueError, match="CUDA int64 tensor of two elements"):
            ops.gumbel_apply(x, cb, 0.2, 0.25, seed=bad)


# ---------------------------------------------------------------------------------------------------------------------
# GPU: one captured call
# ---------------------------------------------------------------------------------------------------------------------
def _warm_then_capture(fn, warm=2):
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(warm):
            fn()
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = fn()
    return graph, out


@pytest.mark.gpu
def test_captured_call_draws_a_new_seed_per_replay(ops):
    n, d, k, temperature, beta = 4096, 32, 256, 0.2, 0.25
    gen = torch.Generator().manual_seed(21)
    x = unit_rows(n, d, seed=22).cuda().requires_grad_(True)
    cb = torch.nn.functional.normalize(torch.rand(k, d, generator=gen), dim=-1).cuda().requires_grad_(True)
    g_emb = (torch.randn(n, d, generator=gen) * 0.1).cuda()
    g_loss = (torch.rand(n, generator=gen) / n).cuda()
    u = torch.rand(n, k, generator=gen).cuda()

    def level(uniforms=None, seed=None):
        emb, ids, loss = ops.gumbel_apply(x, cb, temperature, beta, uniforms=uniforms, seed=seed)
        rng = emb.grad_fn.saved_tensors[-1]           # the pair the backward reads (None for an eager int seed)
        g_x, g_cb = torch.autograd.grad((emb * g_emb).sum() + (loss * g_loss).sum(), (x, cb))
        return dict(emb=emb.detach(), ids=ids, loss=loss.detach(), g_x=g_x, g_codebook=g_cb, rng=rng)

    graph, out = _warm_then_capture(level)
    assert out["rng"] is not None and out["rng"].dtype == torch.int64 and out["rng"].is_cuda
    replays = []
    for _ in range(5):
        graph.replay()
        replays.append({name: v.clone() for name, v in out.items()})
    seeds = [int(r["rng"][0]) for r in replays]
    assert len(set(seeds)) == 5, seeds
    assert all(0 <= s < 2 ** 62 for s in seeds) and all(int(r["rng"][1]) == 0 for r in replays)
    for i in range(5):
        for j in range(i):
            assert not torch.equal(replays[i]["emb"], replays[j]["emb"])
    for r, seed in zip(replays, seeds):
        eager = level(seed=seed)
        for name in ("emb", "ids", "loss", "g_x"):
            assert torch.equal(r[name], eager[name]), name
        _cb_close(r["g_codebook"], eager["g_codebook"])
    # explicit uniforms inside a graph: the same result as the eager call
    graph_u, out_u = _warm_then_capture(lambda: level(uniforms=u))
    graph_u.replay()
    eager = level(uniforms=u, seed=0)
    for name in ("emb", "ids", "loss", "g_x"):
        assert torch.equal(out_u[name], eager[name]), name
    _cb_close(out_u["g_codebook"], eager["g_codebook"])


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the model
# ---------------------------------------------------------------------------------------------------------------------
def _gumbel_hrqvae(k, tags=False):
    from modules.h_rqvae import HRqVae
    from modules.quantize import QuantizeForwardMode
    torch.manual_seed(0)
    np.random.seed(0)
    kw = dict(tag_class_counts=[5, 9, 17], tag_embed_dim=24, sem_id_uniqueness_weight=0.5, sem_id_uniqueness_margin=0.2) \
        if tags else {}
    m = HRqVae(input_dim=64, embed_dim=32, hidden_dims=[48], codebook_size=k, codebook_kmeans_init=False, codebook_normalize=True,
               codebook_mode=QuantizeForwardMode.GUMBEL_SOFTMAX, n_layers=3, n_cat_features=0, commitment_weight=0.3,
               dropout_rate=0.0, **kw).cuda().train()
    m.tag_prediction_loss.use_mixup = False
    for mod in m.modules():
        if isinstance(mod, torch.nn.Dropout):
            mod.p = 0.0
    return m


@pytest.mark.gpu
def test_hrqvae_gumbel_levels_captured_equal_eager_with_their_seeds(ops, monkeypatch):
    """get_semantic_ids + backward of HRqVae in Gumbel mode (L = 3) as one CUDA graph: a replay equals the eager level loop
    fed that replay's three per-level seeds, bit for bit (embeddings, ids, quantize loss, encoder-output gradient)."""
    model = _gumbel_hrqvae(128)
    assert not model._can_fuse()
    n, temperature = 2000, 0.2
    z = unit_rows(n, 32, seed=31).cuda().requires_grad_(True)
    real_apply = ops.gumbel_apply
    pairs = []

    def recording(x, cb, t, beta, uniforms=None, seed=None):
        out = real_apply(x, cb, t, beta, uniforms, seed)
        pairs.append(out[0].grad_fn.saved_tensors[-1])
        return out

    def run():
        pairs.clear()
        q = model.get_semantic_ids(z, gumbel_t=temperature)
        g_z, = torch.autograd.grad(q.embeddings.sum(dim=-1).pow(2).sum() + q.quantize_loss.sum(), (z,))
        return dict(emb=q.embeddings.detach(), ids=q.sem_ids, loss=q.quantize_loss.detach(), g_z=g_z)

    monkeypatch.setattr(ops, "gumbel_apply", recording)
    graph, out = _warm_then_capture(run)
    captured_pairs = list(pairs)
    assert len(captured_pairs) == 3 and all(p is not None for p in captured_pairs)
    seen = set()
    for _ in range(2):
        graph.replay()
        replay = {name: v.clone() for name, v in out.items()}
        seeds = [int(p[0]) for p in captured_pairs]
        assert len(set(seeds)) == 3 and not seen & set(seeds), seeds
        seen |= set(seeds)
        it = iter(seeds)
        monkeypatch.setattr(ops, "gumbel_apply", lambda x, cb, t, beta, uniforms=None, seed=None:
                            real_apply(x, cb, t, beta, uniforms, next(it)))
        eager = run()
        for name in ("emb", "ids", "loss", "g_z"):
            assert torch.equal(replay[name], eager[name]), name
        monkeypatch.setattr(ops, "gumbel_apply", recording)


@pytest.mark.gpu
@pytest.mark.parametrize("k", [128, 512], ids=["fused_k128", "dense_k512"])
def test_graphed_train_step_in_gumbel_mode(ops, k):
    """GraphedTrainStep with HRqVae in Gumbel mode.  On a fixed batch and without an optimizer step, consecutive replays of the
    micro-step differ only by the noise: the statistics vector must change at every replay.  K = 512 has no fused Gumbel
    instantiation and runs the dense PyTorch path, whose torch.rand draw on the device is graph-safe as it stands.  Then
    full steps: parameters stay finite and move."""
    from data.schemas import TaggedSeqBatch
    from hidvae_b200 import dist as hv_dist
    from hidvae_b200.graph_step import GraphedTrainStep
    assert ops.gumbel_supported(32, k) == (k <= 256)
    n, bs = 4096, 256
    g = torch.Generator().manual_seed(3)
    x = unit_rows(n, 64, 1).cuda()
    tags_emb = torch.randn(n, 3, 24, generator=g).cuda()
    tags_idx = torch.stack([torch.randint(0, c, (n,), generator=g) for c in (5, 9, 17)], dim=1).cuda()
    fixed = torch.arange(bs, device="cuda")
    fetch = lambda idx: TaggedSeqBatch(None, None, None, x[fixed], None, None, tags_emb[fixed], tags_idx[fixed])
    model = _gumbel_hrqvae(k, tags=True)
    grads = hv_dist.FlatGradAllReduce(model.parameters())
    opt = torch.optim.AdamW(model.parameters(), lr=torch.tensor(1e-3, device="cuda"), weight_decay=0.01, capturable=True)
    step = GraphedTrainStep(model, opt, grads, fetch, bs, n, gumbel_t=0.2,
                            generator=torch.Generator(device="cuda").manual_seed(11), warmup=3)
    before = torch.cat([p.detach().flatten() for p in model.parameters()]).clone()
    stats = []
    for _ in range(4):
        grads.zero()
        stats.append(step.micro_step().clone())
    assert torch.equal(torch.cat([p.detach().flatten() for p in model.parameters()]), before)   # no step taken
    for i in range(1, 4):
        assert not torch.equal(stats[i], stats[i - 1]), (i, stats)
    assert all(torch.isfinite(s).all() for s in stats)
    for _ in range(5):
        s = step()
    after = torch.cat([p.detach().flatten() for p in model.parameters()])
    assert torch.isfinite(after).all() and torch.isfinite(s).all() and not torch.equal(after, before)


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the trainer
# ---------------------------------------------------------------------------------------------------------------------
TRAINER_GIN = """
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
train.vae_codebook_mode = %modules.quantize.QuantizeForwardMode.GUMBEL_SOFTMAX
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
"""


@pytest.mark.gpu
def test_trainer_gumbel_mode_with_cuda_graph(tmp_path):
    """train(use_cuda_graph=True) in the trainer's default Gumbel-softmax mode: k-means init, replays, two evaluations; the RQ
    loss falls as in the eager run of the same config."""
    from hidvae_b200 import gin_lite
    import train_hidvae
    runs = {}
    try:
        for graphed in (False, True):
            gin_lite.clear_config()
            gin_lite.parse_config(TRAINER_GIN + f"train.use_cuda_graph = {graphed}\n")
            res = train_hidvae.train(save_dir_root=str(tmp_path / str(graphed)), dataset_folder="")
            logs = [h for h in res["history"] if "eval" not in h]
            evals = [h["eval"] for h in res["history"] if "eval" in h]
            assert len(logs) >= 6 and len(evals) == 2
            assert all(np.isfinite(h["loss"]) for h in logs)
            assert 0.0 <= evals[-1]["sem_id_repetition_rate"] <= 1.0 and evals[-1]["codebook_usage_0"] > 0.3
            runs[graphed] = [h["rqvae"] for h in logs]
    finally:
        gin_lite.clear_config()
    eager, graph = runs[False], runs[True]
    assert eager[-1] < eager[0] and graph[-1] < graph[0], runs
    # the two runs draw different noise and batches: the same fall, not the same numbers
    assert graph[-1] / graph[0] < 1.25 * eager[-1] / eager[0], runs
