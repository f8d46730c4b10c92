"""GPU parity tests of the k-means update kernels and the uniqueness-loss kernels (through the C ABI).

k-means bar: identical assignment and centroids (<= 1e-5) given identical initial rows and no empty cluster
(SURVEY.md section 8c); uniqueness loss: rtol 1e-5 on the value, 1e-4 on the feature gradient.
"""
import numpy as np
import pytest
import torch

from helpers import npz, ops, t, unit_rows
from oracle import kmeans as OK
from oracle import rq as O

pytestmark = pytest.mark.gpu


def _lloyd_gpu(ops, x, init_idx, max_iters=500):
    """Host loop of init/kmeans.py:63-77 over the kernels (no empty-cluster reseed needed in these fixtures)."""
    xd = x.cuda()
    c = xd[torch.as_tensor(init_idx, device="cuda")].clone().contiguous()
    k = c.shape[0]
    assign = None
    for it in range(max_iters):
        new_assign = ops.kmeans_assign(xd, c)
        sums, counts, changed = ops.kmeans_accumulate(xd, new_assign, k, assign)
        stats = ops.kmeans_finalize(sums, counts, c)
        assign = new_assign
        assert float(stats[1]) == 0.0, "fixture unexpectedly produced an empty cluster"
        if float(stats[0]) < 1e-10:
            return c, assign, it + 1
    raise AssertionError("k-means did not reach the reference's 1e-10 stop threshold")


@pytest.mark.parametrize("name", ["blobs", "unit32"])
def test_kmeans_matches_reference_golden(ops, golden_dir, name):
    g = npz(golden_dir, "kmeans.npz")
    x, init_idx = t(g[f"{name}/x"]), g[f"{name}/init_idx"]
    c, assign, iters = _lloyd_gpu(ops, x, init_idx)
    ref_assign = t(g[f"{name}/assignment"])
    agree = (assign.cpu() == ref_assign).float().mean()
    assert float(agree) == 1.0, f"assignment agreement {float(agree):.5f}"
    torch.testing.assert_close(c.cpu(), t(g[f"{name}/centroids"]), rtol=1e-5, atol=1e-6)


def test_kmeans_accumulate_is_deterministic_and_exact(ops):
    n, d, k = 20000, 32, 256
    x = unit_rows(n, d, 51).cuda()
    assign = torch.randint(0, k, (n,), generator=torch.Generator().manual_seed(52)).cuda()
    prev = assign.clone()
    prev[::7] = (prev[::7] + 1) % k
    s1, c1, ch1 = ops.kmeans_accumulate(x, assign, k, prev)
    s2, c2, ch2 = ops.kmeans_accumulate(x, assign, k, prev)
    assert torch.equal(s1, s2) and torch.equal(c1, c2)          # bit-reproducible
    assert int(ch1) == int((prev != assign).sum()) == int(ch2)
    ref_s = torch.zeros(k, d, dtype=torch.float64, device="cuda").index_add_(0, assign, x.double())
    ref_c = torch.bincount(assign, minlength=k).float()
    assert torch.equal(c1, ref_c)
    torch.testing.assert_close(s1.double(), ref_s, rtol=1e-5, atol=1e-5)
    _, _, ch_all = ops.kmeans_accumulate(x, assign, k, None)
    assert int(ch_all) == n


def test_kmeans_finalize_reseeds_empty_clusters(ops):
    k, d = 8, 16
    g = torch.Generator().manual_seed(53)
    sums = torch.randn(k, d, generator=g).cuda()
    counts = torch.tensor([3., 0., 5., 1., 0., 2., 7., 4.]).cuda()
    old = torch.randn(k, d, generator=g).cuda()
    reseed = torch.randn(k, d, generator=g).cuda()
    c = old.clone()
    stats = ops.kmeans_finalize(sums, counts, c, reseed)
    expect = torch.where(counts[:, None] > 0, sums / counts.clamp(min=1)[:, None], reseed)
    torch.testing.assert_close(c, expect, rtol=1e-6, atol=1e-7)
    assert float(stats[1]) == 2.0
    torch.testing.assert_close(stats[0], (expect - old).norm(dim=1).max(), rtol=1e-5, atol=1e-6)


@pytest.mark.parametrize("name", ["dups", "margin", "nodup"])
def test_uniqueness_matches_reference_golden(ops, golden_dir, name):
    g = npz(golden_dir, "uniqueness.npz")
    ids = t(g[f"{name}/ids"]).cuda()
    feats = t(g[f"{name}/feats"]).cuda().requires_grad_(True)
    margin, weight = float(g[f"{name}/margin"]), float(g[f"{name}/weight"])
    loss = ops.uniqueness_loss(ids, feats, margin, weight)
    torch.testing.assert_close(loss.cpu(), t(g[f"{name}/loss"]).float(), rtol=1e-5, atol=1e-7)
    loss.backward()
    torch.testing.assert_close(feats.grad.cpu(), t(g[f"{name}/grad_feats"]), rtol=1e-4, atol=1e-7)
    # the call as wired in HRqVae.forward: transposed ids (SURVEY quirk 1) -- a strided view, no copy
    wired = ops.uniqueness_loss(ids.transpose(0, 1), feats.detach(), margin, weight)
    torch.testing.assert_close(wired.cpu(), t(g[f"{name}/loss_as_wired"]).float(), rtol=1e-5, atol=1e-7)
    later = ops.count_rows_with_later_twin(ids)
    p_unique = (ids.shape[0] - float(later)) / ids.shape[0]
    assert abs(p_unique - float(g[f"{name}/p_unique"])) < 1e-7


def test_uniqueness_vs_oracle_large_batch(ops):
    """B = 4096 rows drawn from 3 x 12 codes (many collisions), fp32 features; oracle = [B, B, L] compare on CPU."""
    b, L, k = 4096, 3, 12
    g = torch.Generator().manual_seed(61)
    ids = torch.randint(0, k, (b, L), generator=g)
    feats = torch.randn(b, 32, generator=g)
    ref_feats = feats.clone().requires_grad_(True)
    ref = O.uniqueness_loss(ids, ref_feats, 0.1, 1.5)
    ref.backward()
    f = feats.cuda().requires_grad_(True)
    loss = ops.uniqueness_loss(ids.cuda(), f, 0.1, 1.5)
    loss.backward()
    torch.testing.assert_close(loss.cpu(), ref, rtol=1e-5, atol=1e-7)
    torch.testing.assert_close(f.grad.cpu(), ref_feats.grad, rtol=1e-4, atol=1e-7)
    p_ref = float(O.p_unique_ids(ids))
    p = (b - float(ops.count_rows_with_later_twin(ids.cuda()))) / b
    assert abs(p - p_ref) < 1e-7


def test_uniqueness_degenerate_batches(ops):
    feats = torch.randn(1, 32).cuda()
    assert float(ops.uniqueness_loss(torch.zeros(1, 3, dtype=torch.int64).cuda(), feats, 0.0, 1.0)) == 0.0
    ids = torch.zeros(0, 3, dtype=torch.int64).cuda()
    assert float(ops.uniqueness_loss(ids, torch.zeros(0, 32).cuda(), 0.0, 1.0)) == 0.0


def test_peer_allreduce_two_gpus():
    """hv_peer_allreduce (one kernel over NVLink peer memory) against NCCL on the codebook-gradient size: values,
    bit-identical results on every rank, CUDA-graph replay.  Needs two GPUs on the box (tools/check_peer_allreduce.py)."""
    import json
    import os
    import subprocess
    import sys

    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
                          "--master-port", "29547", os.path.join(root, "tools", "check_peer_allreduce.py")],
                         capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    line = [l for l in out.stdout.splitlines() if l.startswith("{")][-1]
    assert json.loads(line)["ok"] is True


def test_data_parallel_paths_on_nccl_two_gpus():
    """Sharded k-means == single-process k-means, the flat gradient all-reduce, item-sharded bulk assignment + gather and
    the trainer under torchrun on two GPUs over NCCL (tools/check_dp_nccl.py).  Needs two GPUs on the box."""
    import json
    import os
    import subprocess
    import sys

    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
                          "--master-port", "29549", os.path.join(root, "tools", "check_dp_nccl.py")],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, (out.stdout[-1500:] + out.stderr[-2500:])
    line = [l for l in out.stdout.splitlines() if l.startswith("{")][-1]
    assert json.loads(line)["ok"] is True


@pytest.mark.parametrize("n,d,k", [(70000, 32, 1024), (65536, 64, 4096), (40000, 16, 513)])
def test_kmeans_segmented_update_large_k(ops, n, d, k):
    """K * N beyond 2^24: the update sorts the rows by cluster and sums every segment in row order (hv_kmeans_accumulate
    with the sort workspace).  Exact counts, sums equal to a float64 reference within fp32 summation error, bit-identical
    from run to run, and the same sums (to fp32 round-off) as the scan form that small shapes use."""
    from hidvae_b200 import _lib
    x = unit_rows(n, d, 71).cuda()
    g = torch.Generator().manual_seed(72)
    assign = torch.randint(0, k, (n,), generator=g)
    assign[assign == 7] = 8                                  # cluster 7 is empty
    assign = assign.cuda()
    prev = assign.clone()
    prev[::5] = (prev[::5] + 3) % k
    s1, c1, ch1 = ops.kmeans_accumulate(x, assign, k, prev)
    s2, c2, _ = ops.kmeans_accumulate(x, assign, k, prev)
    assert torch.equal(s1, s2) and torch.equal(c1, c2)
    assert int(ch1) == int((prev != assign).sum())
    ref_counts = torch.bincount(assign, minlength=k).float()
    assert torch.equal(c1, ref_counts) and float(c1[7]) == 0.0 and float(s1[7].abs().max()) == 0.0
    ref = torch.zeros(k, d, dtype=torch.float64, device="cuda").index_add_(0, assign, x.double())
    torch.testing.assert_close(s1.double(), ref, rtol=1e-5, atol=1e-5)
    # scan form (no workspace) on the same inputs through the raw C ABI
    sums = torch.empty_like(s1)
    counts = torch.empty_like(c1)
    _lib.check(_lib.lib.hv_kmeans_accumulate(x.data_ptr(), n, d, assign.data_ptr(), None, k, sums.data_ptr(), counts.data_ptr(),
                                             None, None, 0, torch.cuda.current_stream().cuda_stream))
    torch.testing.assert_close(sums, s1, rtol=1e-5, atol=1e-5)
    assert torch.equal(counts, c1)


def test_kmeans_run_large_codebook_reaches_fixed_point(ops):
    """Kmeans.run at the stress shape (K = 4096, D = 64, 65,536 rows): the segmented update is deterministic, so the Lloyd
    loop reaches the reference's 1e-10 stop threshold; inertia must not increase from one update to the next."""
    from init.kmeans import Kmeans
    x = unit_rows(65536, 64, 5).cuda()
    np.random.seed(3)
    torch.manual_seed(3)
    km = Kmeans(k=4096, max_iters=60)
    out = km.run(x)
    assert out.centroids.shape == (4096, 64) and out.assignment.shape == (65536,)
    d_final = (x - out.centroids[out.assignment]).pow(2).sum()
    np.random.seed(3)
    torch.manual_seed(3)
    short = Kmeans(k=4096, max_iters=2).run(x)
    d_short = (x - short.centroids[short.assignment]).pow(2).sum()
    assert float(d_final) <= float(d_short) * (1 + 1e-6)


@pytest.mark.parametrize("b", [6000, 65536])
def test_uniqueness_sorted_path_equals_pairwise_sweep(ops, b):
    """>= 4096 rows take the sorted path (runs of identical tuples); it must give the pairwise sweep's statistics and
    feature gradient (the sweep is the form verified against the reference golden and the oracle)."""
    import ctypes
    from hidvae_b200 import _lib
    g = torch.Generator().manual_seed(81)
    ids = torch.randint(0, 24, (b, 3), generator=g).cuda()
    ids[100] = ids[4000]                                          # a pair far apart in row order
    feats = torch.randn(b, 32, generator=g).cuda()
    margin, weight = 0.05, 1.5
    stream = torch.cuda.current_stream().cuda_stream
    ws = torch.empty(int(_lib.lib.hv_sort_workspace_bytes(b)), dtype=torch.uint8, device="cuda")
    res = {}
    for name, (wp, wb) in {"sorted": (ws.data_ptr(), ws.numel()), "sweep": (None, 0)}.items():
        stats = torch.empty(3, dtype=torch.float64, device="cuda")
        _lib.check(_lib.lib.hv_uniq_forward(ids.data_ptr(), b, 3, ids.stride(0), ids.stride(1), feats.data_ptr(), 32, margin,
                                            stats.data_ptr(), wp, wb, stream))
        gf = torch.zeros_like(feats)
        gout = torch.ones(1, device="cuda")
        _lib.check(_lib.lib.hv_uniq_backward(ids.data_ptr(), b, 3, ids.stride(0), ids.stride(1), feats.data_ptr(), 32, margin,
                                             ctypes.c_float(weight), stats.data_ptr(), gout.data_ptr(), gf.data_ptr(), wp, wb, stream))
        res[name] = (stats.cpu(), gf.cpu())
    assert float(res["sorted"][0][1]) == float(res["sweep"][0][1]) > 0          # pairs
    assert float(res["sorted"][0][2]) == float(res["sweep"][0][2])              # rows with a later twin
    torch.testing.assert_close(res["sorted"][0][0], res["sweep"][0][0], rtol=1e-9, atol=1e-9)
    torch.testing.assert_close(res["sorted"][1], res["sweep"][1], rtol=1e-4, atol=1e-7)
