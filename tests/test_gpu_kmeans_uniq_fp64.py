"""The k-means update and the uniqueness loss against float64, for every shipped instantiation of their kernels.

k-means update (hv_kmeans_accumulate / hv_kmeans_finalize).  References:
  (a) float64 per-cluster sums, sums of |x| and counts (index_add_ in float64 on the device);
  (b) a numpy float32 emulation of each form's documented order, which the kernel must match bit for bit (torch.equal):
      segmented -- one compensated (Kahan) chain per cluster over its rows in ascending order, then s - comp;
      scan      -- thread t takes rows t, t + 256, ... of the cluster in one compensated chain (then s - comp), the xor
                   tree over lanes 16 ... 1, then the 8 warp partials added in order from warp 0.
  Inputs whose fp32 sums are exact (small integers times 2^-6) must give the float64 sums exactly in both forms: every
  member is counted exactly once, whatever the order.
Bars (per element, u = 2^-24, S = sum over the cluster of |x|):
  * forward error |sum - sum64| <= c u S.  A compensated chain over m terms returns s with |error| <= (2u + O(m u^2)) S
    (Knuth; Higham, "Accuracy and Stability of Numerical Algorithms", section 4.3); forming s - comp adds one rounding of
    a value <= S.  m u <= 2^-4 for every shape here (2^20 rows), so the second-order term is below u S: the corrected
    chain is within 4 u S.  Segmented form: that chain is the sum, c = 4.  Scan form: each thread's chain (4 u S_t), then
    a butterfly of depth 5 and 7 further additions of the warp partials, each adding at most u times the sum of |x| below
    it: c = 4 + 5 + 7 = 16.  The constants follow from the order, not from measurements.
  * centroids: |mean - mean64| <= 1e-5 (|mean64| + S / count), the DESIGN.md centroid bar (1e-5 relative) with the
    magnitude of the members as the scale where the mean itself cancels.
  * counts and n_changed exact (prev = None, a given prev, K > N).
  * finalize: means within one rounding of the float64 quotient, reseeds and the empty count exact, the shift
    max ||c_new - c_old|| within (ceil(d / 32) + 8) u relative of its float64 value (per-lane chains, 5 xor levels, sqrt).

Uniqueness loss (hv_uniq_forward / hv_uniq_backward).  Reference in float64 on the device: rows grouped by exact tuple
(torch.unique(dim=0)), the pairs i < j inside each group listed explicitly, cos with F.normalize semantics (norm clamped at
1e-12), hinge, value, and float64 autograd for the feature gradient; pinned to oracle.rq.uniqueness_loss / p_unique_ids
on the CPU.  Bars: pairs and rows with a later twin exact; value rtol 1e-6 plus the fp32 error of a cosine,
(2d + 8 + |margin|) u per pair (d-term fma dot products, two norms, two scalings, the hinge); feature gradient
1e-4 x max |g_ref| (per class of rows: above and below the clamp; rows of a pair whose float64 cosine is within 1e-5 of
the margin are left out, since the hinge may switch there), plus, per active pair of the row, (2d + 8) u |coef| |e| / |f|
(e = fhat_j - fhat_i: a few fp32 roundings of that pair's term) and 2^-40 |coef| / |f| (float64's own rounding) -- which is
all that is left where the gradient vanishes (d = 1, identical rows); identical feature rows give exactly 0.

Hash keys: `row_key` (narrow rows) and the warp key of wide rows (width > 64) are ported to Python with uint64
wraparound.  The narrow port is pinned bit for bit to the keys the sorted path leaves in its workspace.  mix64(h, v) is a
bijection in v, so a last id can be solved for: distinct tuples with equal keys must never count as pairs, and identical
tuples among them must still be found.

Each GPU cell runs under torch.profiler and asserts which instantiation ran; test_every_kmeans_uniq_kernel_has_a_cell
lists the shipped kernels with cuobjdump (CPU) and fails when one has no cell.
"""
import ctypes
import math
from typing import NamedTuple

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from helpers import NEAR_TIE_REL, assert_launched, family, lib_mod, ops, profiled, shipped_kernels, unit_rows
from oracle import kmeans as OK
from oracle import rq as O

gpu = pytest.mark.gpu

U = 2.0 ** -24
C_SEG, C_SCAN = 4, 16          # forward-error constants of the two k-means forms (module docstring)
CENTROID_BAR = 1e-5
UNIQ_VAL_RTOL = 1e-6
UNIQ_GRAD = 1e-4
DIMS = (4, 8, 16, 32, 64, 128)
SORT_FROM_ROWS = 4096          # uniq.cu kSortFromRows
SEGMENTED_ABOVE = 1 << 24      # kmeans.cu / ops.kmeans_accumulate: segmented form when K * N > 2^24

FAMILIES = ("kmeans_accumulate_kernel", "kmeans_segsum_kernel", "uniq_kernel", "uniq_sorted_kernel",   # templates
            "kmeans_keys_kernel", "kmeans_finalize_kernel", "uniq_keys_kernel")                       # plain kernels
KM_FAMILY = ("kmeans_accumulate_kernel", "kmeans_segsum_kernel", "kmeans_keys_kernel")
UQ_FAMILY = ("uniq_kernel", "uniq_sorted_kernel", "uniq_keys_kernel")


def _stream():
    return torch.cuda.current_stream().cuda_stream


def report(tag, ratios):
    print(f"fp64-ratio {tag}: " + ", ".join(f"{k} {v:.3g}" for k, v in ratios.items()))
    bad = {k: v for k, v in ratios.items() if not v <= 1.0}
    assert not bad, f"{tag}: outside the bar (error / bar): {bad}"


def bar_ratio(got, ref, bar):
    """max |got - ref| / bar elementwise (0 / 0 counts as 0; inf for a non-finite value)."""
    if got.numel() == 0:
        return 0.0
    got = got.double()
    if not bool(torch.isfinite(got).all()):
        return math.inf
    err = (got - ref).abs()
    r = torch.where(err == 0, torch.zeros_like(err), err / bar)
    return float(r.max())


# ---------------------------------------------------------------------------------------------------------------------
# k-means: references
# ---------------------------------------------------------------------------------------------------------------------
def km_reference(x, assign, k):
    """float64 per-cluster sums [K, D], sums of |x| [K, D] and counts [K] (int64), on x's device."""
    d = x.shape[1]
    xd = x.double()
    s = torch.zeros(k, d, dtype=torch.float64, device=x.device).index_add_(0, assign, xd)
    a = torch.zeros(k, d, dtype=torch.float64, device=x.device).index_add_(0, assign, xd.abs())
    return s, a, torch.bincount(assign, minlength=k)


def kahan_chains(x, chain, n_chains):
    """fp32 compensated sum of the rows of every chain in ascending row order; returns s - comp [n_chains, D]."""
    x = np.asarray(x, dtype=np.float32)
    chain = np.asarray(chain, dtype=np.int64)
    s = np.zeros((n_chains, x.shape[1]), np.float32)
    comp = np.zeros_like(s)
    if chain.size:
        order = np.lexsort((np.arange(chain.size), chain))
        counts = np.bincount(chain, minlength=n_chains)
        starts = np.cumsum(counts) - counts
        by_len = np.argsort(-counts, kind="stable")
        sorted_len = counts[by_len]
        for r in range(int(counts.max())):
            live = by_len[: int(np.searchsorted(-sorted_len, -r, side="left"))]
            v = x[order[starts[live] + r]]
            sl, cl = s[live], comp[live]
            y = v - cl
            t = sl + y
            comp[live] = (t - sl) - y
            s[live] = t
    return s - comp


def emulate_segmented(x, assign, k):
    return kahan_chains(x, assign, k)


def emulate_scan(x, assign, k):
    n, d = np.asarray(x).shape
    part = kahan_chains(x, np.asarray(assign) * 256 + np.arange(n) % 256, k * 256).reshape(k, 8, 32, d)
    for off in (16, 8, 4, 2, 1):
        part = part + part[:, :, np.arange(32) ^ off]
    tot = np.zeros((k, d), np.float32)
    for w in range(8):
        tot = tot + part[:, w, 0]
    return tot


# ---------------------------------------------------------------------------------------------------------------------
# k-means: the accumulate matrix
# ---------------------------------------------------------------------------------------------------------------------
class KCase(NamedTuple):
    name: str
    n: int
    k: int
    assign: str      # "random" | "uniform" | "skewed" | "all0"
    empty: tuple     # clusters kept empty
    prev: bool
    values: str      # "unit" | "exact"
    ws: str          # "ops" | "always" (raw ABI, workspace given) | "none" | "small" (raw ABI)
    emulate: bool = True


SCAN_CASES = [
    KCase("mixed", 5003, 37, "random", (0, 5, 36), True, "unit", "ops"),
    KCase("k1", 3001, 1, "all0", (), False, "unit", "ops"),
    KCase("k_gt_n", 100, 300, "random", (1,), True, "unit", "ops"),
    KCase("n1", 1, 3, "random", (), True, "unit", "ops"),
    KCase("n0", 0, 5, "random", (), False, "unit", "ops"),
    KCase("uniform", 8192, 32, "uniform", (), True, "unit", "ops"),
    KCase("skewed", 20000, 64, "skewed", (2,), True, "unit", "ops"),
    KCase("exact", 30011, 17, "random", (3,), True, "exact", "ops"),
    KCase("kn_2p24", 65536, 256, "random", (7,), True, "unit", "always"),        # K * N = 2^24: still the scan form
    KCase("no_ws", 70001, 300, "random", (), True, "unit", "none"),              # K * N > 2^24 without a workspace
    KCase("small_ws", 70001, 300, "random", (), False, "unit", "small"),         # ... with one byte too few
]
SEG_CASES = [
    KCase("kn_2p24_plus_k", 65537, 256, "random", (7,), True, "unit", "ops"),   # K * N = 2^24 + K
    KCase("mixed", 5003, 5101, "random", (0, 5100), True, "unit", "ops"),       # K not a power of two, K > N
    KCase("skewed", 20000, 1000, "skewed", (2,), True, "unit", "ops"),
    KCase("uniform", 40000, 500, "uniform", (), True, "unit", "ops"),
    KCase("exact", 30011, 1000, "random", (3,), False, "exact", "ops"),
]
KM_CELLS = [(form, d, c) for form, cases in (("scan", SCAN_CASES), ("segmented", SEG_CASES)) for d in DIMS for c in cases]


def km_inputs(case, d, seed):
    g = torch.Generator().manual_seed(seed)
    n, k = case.n, case.k
    if case.values == "exact":
        x = torch.randint(-64, 65, (n, d), generator=g).float() * 2.0 ** -6
    else:
        x = unit_rows(n, d, seed + 1) + 0.05                        # members with a non-zero mean
    if case.assign == "uniform":
        a = torch.arange(n) % k
    elif case.assign == "all0":
        a = torch.zeros(n, dtype=torch.int64)
    else:
        a = torch.randint(0, k, (n,), generator=g)
        if case.assign == "skewed":                                 # one cluster holds 92 % of the rows
            a[torch.rand(n, generator=g) < 0.92] = 1 % k
    for e in case.empty:
        a[a == e] = (e + 1) % k
    prev = None
    if case.prev:
        prev = a.clone()
        flip = torch.rand(n, generator=g) < 0.3
        prev[flip] = (prev[flip] + 1 + torch.randint(0, max(k - 1, 1), (int(flip.sum()),), generator=g)) % k
    return x, a, prev


def raw_accumulate(lib_mod, x, a, k, prev, ws_mode):
    n, d = x.shape
    sums = torch.empty(k, d, device="cuda")
    counts = torch.empty(k, device="cuda")
    changed = torch.empty((), dtype=torch.int64, device="cuda")
    need = int(lib_mod.lib.hv_sort_workspace_bytes(n))
    nbytes = {"always": need, "small": need - 1, "none": 0}[ws_mode]
    ws = torch.empty(max(nbytes, 1), dtype=torch.uint8, device="cuda")
    lib_mod.check(lib_mod.lib.hv_kmeans_accumulate(x.data_ptr() if n else None, n, d, a.data_ptr() if n else None,
                                                   None if prev is None else prev.data_ptr(), k, sums.data_ptr(),
                                                   counts.data_ptr(), changed.data_ptr(),
                                                   ws.data_ptr() if nbytes else None, nbytes, _stream()))
    return sums, counts, changed


def check_sums(tag, x, a, k, sums, counts, c_form, ops, emulated=None, exact=False):
    """Counts exact, sums within c u S of float64 (bit-exact where the inputs make fp32 exact), centroids within the
    DESIGN.md bar, and bit-equal to the emulation of the form's order when given."""
    s64, abs64, cnt = km_reference(x, a, k)
    assert torch.equal(counts, cnt.float()), f"{tag}: counts differ"
    if exact:
        assert torch.equal(sums.double(), s64), f"{tag}: exact-input sums differ from float64"
    centroids = torch.zeros(k, x.shape[1], device="cuda")
    ops.kmeans_finalize(sums, counts, centroids)
    full = cnt > 0
    c64 = s64[full] / cnt[full, None]
    r = {"sums": bar_ratio(sums, s64, c_form * U * abs64),
         "centroids": bar_ratio(centroids[full], c64, CENTROID_BAR * (c64.abs() + abs64[full] / cnt[full, None]))}
    report(tag, r)
    if emulated is not None:
        em = torch.from_numpy(emulated).cuda()
        if not torch.equal(sums, em):
            ulps = float(((sums.double() - em.double()).abs() / (em.double().abs() * U).clamp(min=1e-45)).max())
            raise AssertionError(f"{tag}: sums differ from the emulated order (up to {ulps:.3g} half-ulps)")
    if bool((~full).any()):
        assert float(sums[~full].abs().max()) == 0.0, f"{tag}: an empty cluster has a non-zero sum"


@gpu
@pytest.mark.parametrize("form,d,case", KM_CELLS, ids=[f"{f}-d{d}-{c.name}" for f, d, c in KM_CELLS])
def test_kmeans_accumulate_cell(ops, lib_mod, form, d, case):
    x, a, prev = km_inputs(case, d, 1000 + d)
    assert (case.k * case.n > SEGMENTED_ABOVE and case.ws in ("ops", "always")) == (form == "segmented")
    xd, ad = x.cuda(), a.cuda()
    pd = None if prev is None else prev.cuda()

    def call():
        if case.ws == "ops":
            return ops.kmeans_accumulate(xd, ad, case.k, pd)
        return raw_accumulate(lib_mod, xd, ad, case.k, pd, case.ws)

    (sums, counts, changed), launches = profiled(call)
    emulated = None
    if case.emulate:
        emulated = (emulate_segmented if form == "segmented" else emulate_scan)(x.numpy(), a.numpy(), case.k)
    check_sums(f"{form}-d{d}-{case.name}", xd, ad, case.k, sums, counts, C_SEG if form == "segmented" else C_SCAN, ops,
               emulated, exact=case.values == "exact")
    want_changed = case.n if prev is None else int((prev != a).sum())
    assert int(changed) == want_changed
    again = call()
    assert torch.equal(again[0], sums) and torch.equal(again[1], counts)     # bit-reproducible
    expected = {f"kmeans_accumulate_kernel<{d}>"} if form == "scan" else {"kmeans_keys_kernel", f"kmeans_segsum_kernel<{d}>"}
    skip = assert_launched(launches, expected, KM_FAMILY)
    if skip:
        pytest.skip(skip)


def _identical_rows(n_same, n_other, k, d, cluster, seed):
    """n_same copies of one row (positive mean) in `cluster`, then n_other unit rows assigned at random."""
    g = torch.Generator().manual_seed(seed)
    v = F.normalize(torch.rand(d, generator=g) + 0.1, dim=0)
    x = torch.cat([v.expand(n_same, d), unit_rows(n_other, d, seed + 1)])
    a = torch.cat([torch.full((n_same,), cluster, dtype=torch.int64), torch.randint(0, k, (n_other,), generator=g)])
    perm = torch.randperm(x.shape[0], generator=g)
    return x[perm].contiguous(), a[perm].contiguous()


@gpu
def test_kmeans_segmented_cluster_of_65536_identical_rows(ops):
    """One cluster of 65,536 identical rows at K = 4096, D = 64 (segmented form): a plain fp32 chain in row order is 6e-4
    relative off the mean here; the compensated chain stays within C_SEG u S."""
    k, d = 4096, 64
    x, a = _identical_rows(65536, 4096, k, d, 11, 91)
    xd, ad = x.cuda(), a.cuda()
    (sums, counts, changed), launches = profiled(lambda: ops.kmeans_accumulate(xd, ad, k, None))
    check_sums("segmented-identical-65536", xd, ad, k, sums, counts, C_SEG, ops, emulate_segmented(x.numpy(), a.numpy(), k))
    assert int(changed) == x.shape[0]
    skip = assert_launched(launches, {"kmeans_keys_kernel", "kmeans_segsum_kernel<64>"}, KM_FAMILY)
    if skip:
        pytest.skip(skip)


@gpu
def test_kmeans_scan_long_chains_of_identical_rows(ops):
    """K = 16 at 2^20 rows (K * N = 2^24: scan form), 90 % of them one identical row in one cluster: every thread's chain
    holds ~3,700 rows of that cluster."""
    k, d, n = 16, 32, 1 << 20
    n_same = int(n * 0.9)
    x, a = _identical_rows(n_same, n - n_same, k, d, 3, 92)
    xd, ad = x.cuda(), a.cuda()
    (sums, counts, _), launches = profiled(lambda: ops.kmeans_accumulate(xd, ad, k, None))
    check_sums("scan-identical-2^20", xd, ad, k, sums, counts, C_SCAN, ops, emulate_scan(x.numpy(), a.numpy(), k))
    skip = assert_launched(launches, {"kmeans_accumulate_kernel<32>"}, KM_FAMILY)
    if skip:
        pytest.skip(skip)


FINALIZE = [(1, 4), (8, 16), (37, 33), (300, 64), (513, 100), (4096, 5)]


@gpu
@pytest.mark.parametrize("k,d", FINALIZE)
@pytest.mark.parametrize("reseed", [True, False])
def test_kmeans_finalize_against_float64(ops, k, d, reseed):
    g = torch.Generator().manual_seed(k * 7 + d)
    counts = torch.randint(0, 50, (k,), generator=g).float()
    counts[::3] = 0.0
    if k == 1:
        counts[0] = 7.0
    sums = torch.randn(k, d, generator=g) * counts[:, None]
    old = torch.randn(k, d, generator=g)
    rs = torch.randn(k, d, generator=g) if reseed else None
    c = old.clone().cuda()
    stats, launches = profiled(lambda: ops.kmeans_finalize(sums.cuda(), counts.cuda(), c, None if rs is None else rs.cuda()))
    c, stats = c.cpu(), stats.cpu()
    full = counts > 0
    mean64 = sums.double()[full] / counts.double()[full, None]
    r = {"means": bar_ratio(c[full], mean64, U * mean64.abs())}
    empty_expect = rs[~full] if reseed else old[~full]
    assert torch.equal(c[~full], empty_expect)
    assert float(stats[1]) == float((~full).sum())
    shift64 = float((c.double() - old.double()).norm(dim=1).max())
    r["shift"] = abs(float(stats[0]) - shift64) / ((math.ceil(d / 32) + 8) * U * shift64)
    report(f"finalize-k{k}-d{d}-{'reseed' if reseed else 'keep'}", r)
    skip = assert_launched(launches, {"kmeans_finalize_kernel"}, ("kmeans_finalize_kernel",))
    if skip:
        pytest.skip(skip)


def _argmin_check_fp64(x, centroids, assign, chunk=8192):
    """Every row's cluster is the float64 argmin of |x - c|^2, or within NEAR_TIE_REL of it (helpers.check_ids' rule)."""
    c64 = centroids.double()
    cn = (c64 * c64).sum(1)
    worst = 0.0
    for s in range(0, x.shape[0], chunk):
        xs = x[s:s + chunk].double()
        dist = (xs * xs).sum(1, keepdim=True) - 2.0 * xs @ c64.t() + cn[None]
        best = dist.min(dim=1).values
        got = dist.gather(1, assign[s:s + chunk, None]).view(-1)
        rel = (got - best) / best.abs().clamp(min=1e-300)
        worst = max(worst, float(rel.max()))
    assert worst < NEAR_TIE_REL, f"an assignment is not the argmin of its centroids: relative gap {worst:.3e}"
    return worst


@gpu
@pytest.mark.parametrize("n,d,k,form", [(20000, 32, 256, "scan"), (65536, 64, 4096, "segmented")],
                         ids=["bench-init-20000x32-k256", "stress-65536x64-k4096"])
def test_kmeans_run_ends_at_a_fixed_point(n, d, k, form):
    """Kmeans.run ends when an update moves no centroid by 1e-10: the centroids are then the float64 means of the final
    assignment (within the form's bound and the centroid bar), and the assignment is the argmin of those centroids."""
    from init.kmeans import Kmeans
    x = unit_rows(n, d, 7).cuda()
    np.random.seed(5)
    torch.manual_seed(5)
    km = Kmeans(k=k, max_iters=3000)
    out = km.run(x)
    assert km.n_iters < 3000, "no fixed point within 3000 Lloyd iterations"
    s64, abs64, cnt = km_reference(x, out.assignment, k)
    assert bool((cnt > 0).all())
    mean64 = s64 / cnt[:, None]
    c_form = C_SEG if form == "segmented" else C_SCAN
    bound = (c_form * U * abs64 + U * s64.abs()) / cnt[:, None]          # the sum's bound, then the division's rounding
    r = {"centroids_bound": bar_ratio(out.centroids, mean64, bound),
         "centroids_bar": bar_ratio(out.centroids, mean64, CENTROID_BAR * (mean64.abs() + abs64 / cnt[:, None])),
         "argmin_gap": _argmin_check_fp64(x, out.centroids, out.assignment) / NEAR_TIE_REL}
    report(f"kmeans-run-{n}x{d}-k{k} ({km.n_iters} iterations)", r)


# ---------------------------------------------------------------------------------------------------------------------
# uniqueness loss: float64 reference
# ---------------------------------------------------------------------------------------------------------------------
class URef(NamedTuple):
    hinge_sum: float
    pairs: int
    has_later: int
    value: float
    g: torch.Tensor        # float64 [rows_f, d]
    g_floor: torch.Tensor  # float64 [rows_f]: rounding allowance where the gradient itself vanishes (check_uniq)
    i: torch.Tensor        # pair rows (i < j)
    j: torch.Tensor
    cos: torch.Tensor      # float64 cosine of every pair


def group_pairs(ids):
    """All pairs i < j of rows with identical tuples (O(rows + pairs)) and the number of rows with a later twin."""
    rows, dev = ids.shape[0], ids.device
    if rows == 0:
        e = torch.zeros(0, dtype=torch.int64, device=dev)
        return e, e, 0
    _, inv = torch.unique(ids, dim=0, return_inverse=True)
    order = torch.argsort(inv, stable=True)
    counts = torch.bincount(inv)
    starts = counts.cumsum(0) - counts
    g_sorted = inv[order]
    after = counts[g_sorted] - (torch.arange(rows, device=dev) - starts[g_sorted]) - 1
    p = torch.repeat_interleave(torch.arange(rows, device=dev), after)
    first = torch.repeat_interleave(after.cumsum(0) - after, after)
    q = p + 1 + (torch.arange(p.numel(), device=dev) - first)
    return order[p], order[q], int((after > 0).sum())


def uniq_reference(ids, feats, margin, weight):
    i, j, has_later = group_pairs(ids)
    f = feats.detach().double().requires_grad_(True)
    fi = F.normalize(f[i], p=2, dim=-1, eps=1e-12)
    fj = F.normalize(f[j], p=2, dim=-1, eps=1e-12)
    cos = (fi * fj).sum(-1)
    hinge = F.relu(cos - margin)
    value = weight * hinge.mean() if i.numel() else f.sum() * 0.0
    value.backward()
    with torch.no_grad():
        d = feats.shape[1]
        inv = 1.0 / f.norm(dim=1).clamp(min=1e-12)
        per_pair = abs(weight) / max(i.numel(), 1) * (hinge > 0) * ((2 * d + 8) * U * (fi - fj).norm(dim=1) + 2.0 ** -40)
        floor = torch.zeros(f.shape[0], dtype=torch.float64, device=f.device)
        floor.index_add_(0, i, per_pair * inv[i]).index_add_(0, j, per_pair * inv[j])
    return URef(float(hinge.sum()), int(i.numel()), has_later, float(value.detach()), f.grad, floor, i, j, cos.detach())


def uniq_value_bound(d, margin):
    return (2 * d + 8 + abs(margin)) * U


def check_uniq(tag, ref, stats, value, g, feats, d, margin, weight, identical_feats=False):
    """Exact counts, value / hinge sum within rtol 1e-6 plus the cosine bound, gradient within 1e-4 x max |g_ref|."""
    stats = stats.double().cpu()
    assert int(stats[1]) == ref.pairs and float(stats[1]) == ref.pairs, f"{tag}: pairs {float(stats[1])} != {ref.pairs}"
    assert int(stats[2]) == ref.has_later and float(stats[2]) == ref.has_later, \
        f"{tag}: rows with a later twin {float(stats[2])} != {ref.has_later}"
    cb = uniq_value_bound(d, margin)
    r = {"hinge_sum": abs(float(stats[0]) - ref.hinge_sum) / (UNIQ_VAL_RTOL * abs(ref.hinge_sum) + ref.pairs * cb + 1e-300)}
    if value is not None:
        r["value"] = abs(float(value) - ref.value) / (UNIQ_VAL_RTOL * abs(ref.value) + abs(weight) * cb + 1e-300)
    if g is not None and g.numel():
        g = g.double()
        if identical_feats:
            assert torch.equal(g, torch.zeros_like(g)), f"{tag}: identical features must give a zero gradient"
        rows_f = feats.shape[0]
        keep = torch.ones(rows_f, dtype=torch.bool, device=g.device)
        near = (ref.cos - margin).abs() < 1e-5
        keep[ref.i[near]] = False
        keep[ref.j[near]] = False
        clamped = feats.double().norm(dim=1) < 1e-12
        for name, rows in (("g", keep & ~clamped), ("g_clamped", keep & clamped)):
            if bool(rows.any()):
                gm = float(ref.g[rows].abs().max())
                r[name] = bar_ratio(g[rows], ref.g[rows], UNIQ_GRAD * gm + ref.g_floor[rows, None])
    report(tag, r)


def raw_uniq(lib_mod, ids, feats, margin, weight, ws_mode, g_out=1.0):
    """hv_uniq_forward + hv_uniq_backward through the C ABI; ws_mode "sorted" gives the sort workspace, "none" withholds it."""
    rows, width = ids.shape
    d = 0 if feats is None else feats.shape[1]
    stats = torch.empty(3, dtype=torch.float64, device="cuda")
    need = int(lib_mod.lib.hv_sort_workspace_bytes(rows))
    ws = torch.empty(max(need, 1), dtype=torch.uint8, device="cuda") if ws_mode == "sorted" else None
    wp, wb = (ws.data_ptr(), need) if ws is not None else (None, 0)
    fp = None if feats is None else feats.data_ptr()
    lib_mod.check(lib_mod.lib.hv_uniq_forward(ids.data_ptr(), rows, width, ids.stride(0), ids.stride(1), fp, d,
                                              ctypes.c_float(margin), stats.data_ptr(), wp, wb, _stream()))
    g = None
    if feats is not None:
        g = torch.zeros_like(feats)
        go = torch.full((1,), g_out, device="cuda")
        lib_mod.check(lib_mod.lib.hv_uniq_backward(ids.data_ptr(), rows, width, ids.stride(0), ids.stride(1), fp, d,
                                                   ctypes.c_float(margin), ctypes.c_float(weight), stats.data_ptr(),
                                                   go.data_ptr(), g.data_ptr(), wp, wb, _stream()))
    return stats, g, ws


def uniq_expected(rows, ws_mode):
    if rows >= SORT_FROM_ROWS and ws_mode == "sorted":
        return {"uniq_keys_kernel", "uniq_sorted_kernel<false>", "uniq_sorted_kernel<true>"}
    return {"uniq_kernel<false>", "uniq_kernel<true>"}


# ---------------------------------------------------------------------------------------------------------------------
# uniqueness loss: inputs
# ---------------------------------------------------------------------------------------------------------------------
def plant_ids(rows, width, kind, seed):
    """int64 [rows, width]: 'distinct' tuples, 'pairs' (about 40 % of rows copy an earlier row's tuple), or 'run2048'
    (2,048 rows share one tuple, the rest as 'pairs')."""
    g = torch.Generator().manual_seed(seed)
    base = torch.randint(0, 1 << 40, (rows, width), generator=g)
    base[:, 0] = torch.arange(rows)                                   # distinct before planting
    src = torch.arange(rows)
    if kind in ("pairs", "run2048") and rows >= 2:
        follow = torch.rand(rows, generator=g) < 0.4
        follow[0] = False
        follow[1] = True
        lead = (torch.rand(rows, generator=g) * torch.arange(rows)).long()   # an earlier row
        src = torch.where(follow, lead, src)
        while True:                                                       # follow chains down to their leaders
            nxt = src[src]
            if torch.equal(nxt, src):
                break
            src = nxt
    if kind == "run2048":
        pos = torch.randperm(rows, generator=g)[:2048]
        src[pos] = int(src[pos.min()])
    return base[src].contiguous(), src


def make_feats(rows, d, kind, src, seed):
    """float32 [rows, d]: 'random', 'near<eps>' (every follower within eps x |f| of its leader), 'identical' (followers
    copy their leader), 'clamped' (a third of the rows scaled below the 1e-12 clamp, a tenth exactly zero)."""
    g = torch.Generator().manual_seed(seed)
    f = torch.randn(rows, d, generator=g) * (torch.rand(rows, 1, generator=g) * 4 + 0.25)
    if kind.startswith("near"):
        eps = float(kind[4:])
        noise = torch.randn(rows, d, generator=g)
        noise = noise / noise.norm(dim=1, keepdim=True).clamp(min=1e-30)
        f = f[src] + eps * f[src].norm(dim=1, keepdim=True) * noise * (src != torch.arange(rows))[:, None]
    elif kind == "identical":
        f = f[src].clone()
    elif kind == "clamped":
        small = torch.rand(rows, generator=g) < 0.33
        f[small] = f[small] / f[small].norm(dim=1, keepdim=True).clamp(min=1e-30) * 3e-13
        f[torch.rand(rows, generator=g) < 0.1] = 0.0
    return f.float().contiguous()


class UCell(NamedTuple):
    rows: int
    width: int
    d: int
    ids: str
    feats: str
    margin: float
    weight: float
    ws: str          # "sorted" (workspace given) | "none"

    @property
    def id(self):
        return (f"r{self.rows}-w{self.width}-d{self.d}-{self.ids}-{self.feats}-m{self.margin:g}-wt{self.weight:g}"
                f"-{'sort' if self.rows >= SORT_FROM_ROWS and self.ws == 'sorted' else 'sweep'}")


def _ucells():
    cells = []
    for rows in (2, 255, 256, 257, 4095, 4096, 8192):                       # tile edges, the dispatch
        for width in (1, 3, 64, 65):                                         # narrow and wide keys
            cells.append(UCell(rows, width, 32, "pairs", "random", 0.1, 1.5, "sorted"))
    cells.append(UCell(65536, 3, 32, "pairs", "random", 0.1, 1.5, "sorted"))
    for rows in (4096, 8192):                                                # >= 4096 rows without a workspace: sweep
        for width in (3, 65):
            cells.append(UCell(rows, width, 32, "pairs", "random", 0.1, 1.5, "none"))
    for rows in (257, 8192):
        for d in (0, 1, 33):
            cells.append(UCell(rows, 3, d, "pairs", "random", 0.1, 1.5, "sorted"))
        cells.append(UCell(rows, 3, 32, "distinct", "random", 0.1, 1.5, "sorted"))
    for rows in (4095, 8192):                                                # a run of 2,048 identical tuples
        for margin, weight in ((-1.5, 0.7), (1.0, 1.0), (0.1, 0.0)):         # margin < 0, margin >= 1, weight 0
            cells.append(UCell(rows, 3, 32, "run2048", "random", margin, weight, "sorted"))
    for rows in (257, 8192):                                                 # near-duplicate and clamped features
        for feats in ("near1e-1", "near1e-2", "near1e-3", "near1e-4", "identical"):
            cells.append(UCell(rows, 3, 32, "pairs", feats, 0.1, 1.5, "sorted"))
        cells.append(UCell(rows, 3, 32, "pairs", "clamped", -0.5, 1.5, "sorted"))
    return cells


U_CELLS = _ucells()


@gpu
@pytest.mark.parametrize("cell", U_CELLS, ids=[c.id for c in U_CELLS])
def test_uniqueness_cell(lib_mod, cell):
    ids, src = plant_ids(cell.rows, cell.width, cell.ids, cell.rows + cell.width)
    feats = make_feats(cell.rows, cell.d, cell.feats, src, cell.rows * 3 + cell.d)
    ids_d, feats_d = ids.cuda(), feats.cuda()
    (stats, g, _), launches = profiled(lambda: raw_uniq(lib_mod, ids_d, feats_d, cell.margin, cell.weight, cell.ws))
    ref = uniq_reference(ids_d, feats_d, cell.margin, cell.weight)
    if cell.ids == "distinct":
        assert ref.pairs == 0
    pairs = float(stats[1])
    value = cell.weight * float(stats[0]) / pairs if pairs > 0 else 0.0
    check_uniq(cell.id, ref, stats, value, g, feats_d, cell.d, cell.margin, cell.weight,
               identical_feats=cell.feats == "identical")
    if cell.margin >= 1.0 or cell.weight == 0.0:
        assert torch.equal(g, torch.zeros_like(g))
    skip = assert_launched(launches, uniq_expected(cell.rows, cell.ws), UQ_FAMILY)
    if skip:
        pytest.skip(skip)


@gpu
@pytest.mark.parametrize("b", [128, 8192])
def test_uniqueness_as_wired(ops, b):
    """The call of HRqVae.forward: ids [B, 3] handed over transposed (3 rows of B ids, a strided view: the wide-row warp
    key), feats [B, 32].  Level rows 0 and 2 are planted identical, so the loss is non-zero and has a backward."""
    g = torch.Generator().manual_seed(b)
    ids = torch.randint(0, 256, (b, 3), generator=g)
    ids[:, 2] = ids[:, 0]
    feats = torch.randn(b, 32, generator=g).cuda().requires_grad_(True)
    wired = ids.cuda().transpose(0, 1)
    assert not wired.is_contiguous()

    def forward_backward():
        loss = ops.uniqueness_loss(wired, feats, 0.1, 1.5)
        return loss, torch.autograd.grad(loss, feats)[0]

    (loss, grad), launches = profiled(forward_backward)
    ref = uniq_reference(wired, feats, 0.1, 1.5)
    assert ref.pairs == 1
    stats = ops.uniq_stats(wired, feats.detach(), 0.1)
    check_uniq(f"as-wired-B{b}", ref, stats, loss, grad, feats.detach(), 32, 0.1, 1.5)
    assert float(ops.count_rows_with_later_twin(wired)) == 1.0
    skip = assert_launched(launches, {"uniq_kernel<false>", "uniq_kernel<true>"}, UQ_FAMILY)
    if skip:
        pytest.skip(skip)


# ---------------------------------------------------------------------------------------------------------------------
# hash keys: Python ports with uint64 wraparound, colliding tuples
# ---------------------------------------------------------------------------------------------------------------------
M64 = (1 << 64) - 1
H0 = 0x243F6A8885A308D3
GOLD = 0x9E3779B97F4A7C15
MUL = 0xFF51AFD7ED558CCD
MUL_INV = pow(MUL, -1, 1 << 64)


def mix64(h, v):
    h ^= (v + GOLD + (h << 6) + (h >> 2)) & M64
    h = (h * MUL) & M64
    return h ^ (h >> 33)


def mix64_solve(h, target):
    """The v with mix64(h, v) == target (mix64 is a bijection in v)."""
    t = target ^ (target >> 33)                  # h ^= h >> 33 undone (shift >= 32: one step inverts it)
    t = (t * MUL_INV) & M64
    return ((t ^ h) - GOLD - ((h << 6) & M64) - (h >> 2)) & M64


def u64(v):
    return int(v) & M64


def s64(v):
    return v - (1 << 64) if v >= 1 << 63 else v


def row_key(row):
    h = H0
    for v in row:
        h = mix64(h, u64(v))
    return h


def row_keys_np(ids):
    """Vectorised row_key of every row of an int64 array (uint64 arithmetic wraps)."""
    ids = np.ascontiguousarray(ids, dtype=np.int64).view(np.uint64)
    h = np.full(ids.shape[0], H0, dtype=np.uint64)
    for c in range(ids.shape[1]):
        h ^= ids[:, c] + np.uint64(GOLD) + (h << np.uint64(6)) + (h >> np.uint64(2))
        h *= np.uint64(MUL)
        h ^= h >> np.uint64(33)
    return h


def wide_lane_state(row, lane, upto):
    """State of `lane` of the wide-row key after its columns < upto."""
    h = (H0 + lane) & M64
    for c in range(lane, min(upto, len(row)), 32):
        h = mix64(h, u64(row[c]))
    return h


def wide_key(row):
    """tile_keys for width > 64: lane l hashes columns l, l + 32, ... from H0 + l, then mixes in l + 1; lanes xor-combined."""
    h = 0
    for lane in range(32):
        h ^= mix64(wide_lane_state(row, lane, len(row)), lane + 1)
    return h


def narrow_collider(row, new_first):
    """A tuple with row's key: first id replaced, last id solved for."""
    out = [u64(v) for v in row]
    out[0] = u64(new_first)
    h = H0
    for v in out[:-1]:
        h = mix64(h, v)
    target = H0
    for v in row[:-1]:
        target = mix64(target, u64(v))
    out[-1] = mix64_solve(h, mix64(target, u64(row[-1])))
    return [s64(v) for v in out]


def wide_collider(row, lane, new_value):
    """A tuple with row's wide key: two columns of one lane changed (lane, lane + 32), the lane's state unchanged."""
    out = [u64(v) for v in row]
    c0, c1 = lane, lane + 32
    out[c0] = u64(new_value)
    after = wide_lane_state(row, lane, c1 + 1)
    out[c1] = mix64_solve(wide_lane_state(out, lane, c1), after)
    return [s64(v) for v in out]


def test_hash_ports_self_consistent():
    """CPU: the solver inverts mix64, the vectorised port equals the scalar one, and the constructed colliders are
    distinct tuples with equal keys (narrow and wide)."""
    rng = np.random.default_rng(0)
    for _ in range(200):
        h, v = int(rng.integers(0, 1 << 63)) * 2 + 1, int(rng.integers(0, 1 << 63))
        assert mix64_solve(h, mix64(h, v)) == v
    ids = rng.integers(-(1 << 62), 1 << 62, size=(50, 3), dtype=np.int64)
    assert [int(k) for k in row_keys_np(ids)] == [row_key(r) for r in ids.tolist()]
    row = ids[0].tolist()
    col = narrow_collider(row, row[0] + 1)
    assert col != row and row_key(col) == row_key(row)
    assert int(row_keys_np(np.array([row, col]))[0]) == int(row_keys_np(np.array([row, col]))[1])
    wrow = rng.integers(0, 1000, size=96).tolist()
    wcol = wide_collider(wrow, 5, 12345)
    assert wcol != wrow and sum(a != b for a, b in zip(wrow, wcol)) == 2 and wide_key(wcol) == wide_key(wrow)


def _collision_ids(rows, width, wide, seed):
    """Rows A, B (distinct, equal key), and a copy of each; three more colliders of A; the rest distinct filler.
    Returns ids and the positions of (A, B, A', B')."""
    rng = np.random.default_rng(seed)
    ids = rng.integers(0, 1 << 40, size=(rows, width), dtype=np.int64)
    ids[:, 0] = np.arange(rows) + (1 << 41)
    a = rng.integers(0, 1000, size=width).tolist()
    make = (lambda r, i: wide_collider(r, i % 32, 5000 + i)) if wide else (lambda r, i: narrow_collider(r, 5000 + i))
    b = make(a, 0)
    others = [make(a, i) for i in range(1, 4)]
    pos = rng.choice(rows, size=7, replace=False)
    for p, t in zip(pos, [a, b, a, b] + others):
        ids[p] = t
    key = wide_key if wide else row_key
    assert len({key(ids[p].tolist()) for p in pos}) == 1 and len({tuple(ids[p].tolist()) for p in pos}) == 5
    return torch.from_numpy(ids), pos


@gpu
@pytest.mark.parametrize("rows,ws", [(300, "none"), (8192, "sorted")], ids=["sweep-300", "sorted-8192"])
def test_narrow_key_collisions_and_port(lib_mod, rows, ws):
    """Width 3: distinct tuples with one key are not pairs; their copies are.  On the sorted path the keys left in the
    workspace (keys_in, the first 256-aligned block: cub does not write its input) equal the Python port bit for bit."""
    ids, pos = _collision_ids(rows, 3, False, rows)
    feats = torch.randn(rows, 8, generator=torch.Generator().manual_seed(3)).cuda()
    ids_d = ids.cuda()
    (stats, g, wsbuf), launches = profiled(lambda: raw_uniq(lib_mod, ids_d, feats, -0.5, 1.0, ws))
    ref = uniq_reference(ids_d, feats, -0.5, 1.0)
    assert ref.pairs == 2 and ref.has_later == 2
    check_uniq(f"narrow-collisions-{rows}", ref, stats, None, g, feats, 8, -0.5, 1.0)
    if ws == "sorted":
        assert wsbuf.data_ptr() % 256 == 0
        keys = wsbuf[: rows * 8].view(torch.int64).cpu().numpy().view(np.uint64)
        assert np.array_equal(keys, row_keys_np(ids.numpy())), "device row keys differ from the Python port"
        assert len(set(keys[pos].tolist())) == 1
    skip = assert_launched(launches, uniq_expected(rows, ws), UQ_FAMILY)
    if skip:
        pytest.skip(skip)


@gpu
@pytest.mark.parametrize("width", [96, 200])
def test_wide_key_collisions(lib_mod, width):
    """Width > 64 (warp key of the sweep): colliding distinct tuples are not pairs, their copies are."""
    rows = 300
    ids, pos = _collision_ids(rows, width, True, width)
    feats = torch.randn(rows, 8, generator=torch.Generator().manual_seed(4)).cuda()
    ids_d = ids.cuda()
    (stats, g, _), launches = profiled(lambda: raw_uniq(lib_mod, ids_d, feats, -0.5, 1.0, "none"))
    ref = uniq_reference(ids_d, feats, -0.5, 1.0)
    assert ref.pairs == 2
    check_uniq(f"wide-collisions-w{width}", ref, stats, None, g, feats, 8, -0.5, 1.0)
    skip = assert_launched(launches, {"uniq_kernel<false>", "uniq_kernel<true>"}, UQ_FAMILY)
    if skip:
        pytest.skip(skip)


# ---------------------------------------------------------------------------------------------------------------------
# CPU: references pinned, argument checks, coverage
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("rows,width,values", [(2, 3, 1), (60, 3, 3), (300, 1, 40), (257, 4, 2)])
def test_uniq_reference_matches_oracle(rows, width, values):
    g = torch.Generator().manual_seed(rows)
    ids = torch.randint(0, values, (rows, width), generator=g)
    feats = torch.randn(rows, 16, generator=g)
    feats[3 % rows] = 0.0
    ref = uniq_reference(ids, feats, 0.1, 1.3)
    f = feats.clone().requires_grad_(True)
    want = O.uniqueness_loss(ids, f, 0.1, 1.3)
    assert abs(ref.value - float(want)) <= 1e-6 * max(1.0, abs(float(want)))
    if want.requires_grad:
        want.backward()
        torch.testing.assert_close(ref.g.float(), f.grad, rtol=1e-4, atol=1e-6)
    assert abs((rows - ref.has_later) / rows - float(O.p_unique_ids(ids))) < 1e-7
    same = (ids[:, None] == ids[None]).all(-1).triu(1)
    assert ref.pairs == int(same.sum())


def test_kmeans_references_pinned():
    """CPU: the float64 sums equal oracle.kmeans.lloyd_update's means; the emulation of either order equals float64 on
    exact inputs and stays within its bound on 20,000 identical rows, where a plain fp32 chain does not."""
    x = unit_rows(3000, 8, 3)
    c = x[:20].clone()
    new_c, assign, n_empty = OK.lloyd_update(x, c, lambda: 0)
    s64, abs64, cnt = km_reference(x, assign, 20)
    full = cnt > 0
    torch.testing.assert_close((s64[full] / cnt[full, None]).float(), new_c[full], rtol=1e-5, atol=1e-6)
    xe = (torch.randint(-64, 65, (5000, 4)).float() * 2.0 ** -6)
    ae = torch.randint(0, 7, (5000,))
    se, _, _ = km_reference(xe, ae, 7)
    assert np.array_equal(emulate_scan(xe.numpy(), ae.numpy(), 7), se.float().numpy())
    assert np.array_equal(emulate_segmented(xe.numpy(), ae.numpy(), 7), se.float().numpy())
    v = np.full((20000, 4), 0.3, np.float32) + np.arange(4, dtype=np.float32) * np.float32(0.1)
    a0 = np.zeros(20000, np.int64)
    exact = v.astype(np.float64).sum(0)
    plain = np.cumsum(v, axis=0, dtype=np.float32)[-1].astype(np.float64)
    seg = emulate_segmented(v, a0, 1)[0].astype(np.float64)
    bound = C_SEG * U * np.abs(v).astype(np.float64).sum(0)
    assert (np.abs(seg - exact) <= bound).all() and not (np.abs(plain - exact) <= bound).all()


def test_argument_checks(ops):
    """The Python wrappers reject what the kernels would misread, before any device work (CPU tensors suffice)."""
    x = torch.zeros(10, 4)
    with pytest.raises(ValueError, match="int64"):
        ops.kmeans_accumulate(x, torch.zeros(10, dtype=torch.int32), 3)
    with pytest.raises(ValueError, match="assign"):
        ops.kmeans_accumulate(x, torch.zeros(9, dtype=torch.int64), 3)
    with pytest.raises(ValueError, match="prev_assign"):
        ops.kmeans_accumulate(x, torch.zeros(10, dtype=torch.int64), 3, torch.zeros(10, dtype=torch.int32))
    with pytest.raises(ValueError, match="prev_assign"):
        ops.kmeans_accumulate(x, torch.zeros(10, dtype=torch.int64), 3, torch.zeros(5, 2, dtype=torch.int64))
    with pytest.raises(ValueError, match="feats"):
        ops.uniqueness_loss(torch.zeros(6, 3, dtype=torch.int64), torch.zeros(5, 8), 0.1, 1.0)
    with pytest.raises(ValueError, match="feats"):
        ops.uniq_stats(torch.zeros(6, 3, dtype=torch.int64), torch.zeros(6 * 8), 0.1)
    with pytest.raises(RuntimeError, match="CUDA"):                         # valid shapes reach the device check
        ops.kmeans_accumulate(x, torch.zeros(10, dtype=torch.int64), 3)


def test_every_kmeans_uniq_kernel_has_a_cell():
    """Every k-means and uniqueness kernel in the built library (16 instantiations of the four templates, three plain
    kernels) is the expected kernel of some cell of this file (CPU only: reads the library with cuobjdump)."""
    shipped = {k for k in shipped_kernels() if family(k) in FAMILIES}
    assert {family(s) for s in shipped} == set(FAMILIES), sorted(shipped)
    assert len(shipped) == 16 + 3, sorted(shipped)
    covered = {"kmeans_finalize_kernel"} if FINALIZE else set()
    for form, d, _ in KM_CELLS:
        covered |= {f"kmeans_accumulate_kernel<{d}>"} if form == "scan" else {"kmeans_keys_kernel", f"kmeans_segsum_kernel<{d}>"}
    for c in U_CELLS:
        covered |= uniq_expected(c.rows, c.ws)
    unreached = sorted(shipped - covered)
    assert not unreached, f"{len(unreached)} of {len(shipped)} shipped kernels have no test cell: {unreached}"
    assert not sorted(covered - shipped), f"cells expect kernels the library does not ship: {sorted(covered - shipped)}"
