"""Every shipped instantiation of the quantiser kernels against a float64 reference evaluated on the device.

The reference (`reference` below) is plain torch in float64: the residual chain that follows the kernel's OWN ids (so a
documented near-tie at one level does not turn into spurious mismatches downstream), with the detach structure of
oracle/rq.py (quantize_level, rotation_trick, quantize_loss), and fp64 autograd of that gather-based chain for the backward.
It covers eval, per-level loss gradients, level-broadcast g_emb and stride-0 g_loss, and is pinned once to oracle.rq_forward
autograd (test_reference_matches_oracle_autograd, CPU).  Ids are checked on every row and level: the kernel's code must
satisfy d64(chosen) - d64(min) <= NEAR_TIE_REL |d64(min)| on the fp64 residual.

Each cell of the instantiation matrix names the kernel it expects (e.g. rq_bwd_smem_kernel<32,8,true,true,3>), runs once
under torch.profiler and asserts that this kernel and no other of its family was launched; test_every_shipped_instantiation
_has_a_cell lists the instantiations in libhidvae_b200.so (cuobjdump) and fails when one has no cell.

Bars (those of tests/test_gpu_rq.py and tests/test_gpu_gumbel.py; the measured worst ratio error / bar is printed as
"fp64-ratio" and recorded in each test's docstring):
  * emb_out / residuals / final residual: rtol 1e-5, atol 1e-6 x max(1, |value|max); loss / level_loss: rtol 1e-5, atol 1e-6.
    The fp32 error of a residual is a few ulps of the row's NORM per level, so an element much smaller than its row needs an
    atol of that size.  Rows are unit-norm and every level shrinks them, so the scale is 1 except where a level cannot shrink
    the residual: with K = 1 the rotation trick returns |o| = |r|, and |r - o| can be up to twice |r| at every level (at L = 5
    the unscaled bar was exceeded 1.5-fold at D = 8)
  * g_x: rtol 2e-5, atol 1e-6 x max(1, |g_x|max)   (h = g_emb - G cancels operands of size |g|max)
  * codebook gradient: rtol 1e-4, atol 1e-5 x max(1, |g_cb|max)   (fp32 sums of ~N / K terms in atomic order)
"""
import math
from typing import NamedTuple, Optional

import pytest
import torch
import torch.nn.functional as F

from helpers import NEAR_TIE_REL, assert_launched, family, make_codebooks, ops, profiled, shipped_kernels, unit_rows
from oracle import rq as O

STE, ROT = O.MODE_STE, O.MODE_ROTATION_TRICK
MODES = {"ste": (STE, True), "rot": (ROT, True), "eval": (STE, False)}   # name -> (mode, training)
BETA = 0.4
VAL = (1e-5, 1e-6)
GX = (2e-5, 1e-6)     # atol scaled by max(1, |g_x|max)
GCB = (1e-4, 1e-5)    # atol scaled by max(1, |g_cb|max)
GUMBEL_VAL = (1e-5, 1e-6)
GUMBEL_GRAD = (1e-4, 1e-4)   # atol scaled by the gradient's max

FAMILIES = ("rq_bwd_kernel", "rq_bwd_smem_kernel", "rq_fwd_simt_kernel", "rq_fwd_tc_kernel", "rq_fwd_tc_v11_kernel",
            "gumbel_fwd_kernel", "gumbel_bwd_kernel")
BWD_FAMILY = ("rq_bwd_kernel", "rq_bwd_smem_kernel")
FWD_FAMILY = ("rq_fwd_simt_kernel", "rq_fwd_tc_kernel", "rq_fwd_tc_v11_kernel")
GUMBEL_FAMILY = ("gumbel_fwd_kernel", "gumbel_bwd_kernel")


# ---------------------------------------------------------------------------------------------------------------------
# float64 reference
# ---------------------------------------------------------------------------------------------------------------------
class Ref(NamedTuple):
    emb: torch.Tensor         # [L, N, D]
    res: torch.Tensor         # [L, N, D]  input of every level
    level_loss: torch.Tensor  # [L, N]
    loss: torch.Tensor        # [N]
    final: torch.Tensor       # [N, D]
    g_x: Optional[torch.Tensor]
    g_cb: Optional[torch.Tensor]


def _level(r, e, mode, training, beta):
    """emb_out and loss of one level given the code row e (modules/quantize.py:131-148, oracle/rq.py:quantize_level)."""
    if training and mode == ROT:   # oracle.rotation_trick: u, q, w detached; r enters linearly
        u = r / (r.norm(dim=-1, keepdim=True) + 1e-8)
        q = e / (e.norm(dim=-1, keepdim=True) + 1e-8)
        w = F.normalize(u + q, p=2, dim=-1, eps=1e-6).detach()
        u, q = u.detach(), q.detach()
        o = r - 2 * (r * w).sum(-1, keepdim=True) * w + 2 * (r * u).sum(-1, keepdim=True) * q
    elif training:                 # STE
        o = r + (e - r).detach()
    else:                          # eval: emb_out = e whatever the mode
        o = e
    ll = ((r.detach() - e) ** 2).sum(-1) + beta * ((r - e.detach()) ** 2).sum(-1)   # oracle.quantize_loss
    return o, ll


def reference(x, cbs, ids, mode, training, beta, g_emb=None, g_loss=None, g_ll=None, chunk=1 << 20):
    """fp64 forward along the given ids [N, L] and, when any upstream gradient is given, fp64 autograd of
    sum(emb_out g_emb) + sum(loss g_loss) + sum(level_loss g_ll).  g_emb is [L, N, D] (any strides), g_loss [N], g_ll [L, N]."""
    n, d = x.shape
    n_levels = cbs.shape[0]
    assert int(ids.min()) >= 0 and int(ids.max()) < cbs.shape[1], "ids out of range"
    grad = g_emb is not None or g_loss is not None or g_ll is not None
    cb = cbs.detach().double().requires_grad_(grad)
    f64 = dict(dtype=torch.float64, device=x.device)
    emb, res, lls = torch.empty(n_levels, n, d, **f64), torch.empty(n_levels, n, d, **f64), torch.empty(n_levels, n, **f64)
    final = torch.empty(n, d, **f64)
    g_x = torch.zeros(n, d, **f64) if grad else None
    g_cb = torch.zeros_like(cb) if grad else None
    for s in range(0, n, chunk):
        e_ = min(n, s + chunk)
        xs = x[s:e_].detach().double().requires_grad_(grad)
        with torch.enable_grad():
            r, objective = xs, 0.0
            for l in range(n_levels):
                o, ll = _level(r, cb[l][ids[s:e_, l]], mode, training, beta)
                res[l, s:e_], emb[l, s:e_], lls[l, s:e_] = r.detach(), o.detach(), ll.detach()
                if g_emb is not None:
                    objective = objective + (o * g_emb[l, s:e_].double()).sum()
                if g_loss is not None:
                    objective = objective + (ll * g_loss[s:e_].double()).sum()
                if g_ll is not None:
                    objective = objective + (ll * g_ll[l, s:e_].double()).sum()
                r = r - o
            final[s:e_] = r.detach()
            if grad:
                gx, gc = torch.autograd.grad(objective, (xs, cb), allow_unused=True)
                if gx is not None:
                    g_x[s:e_] = gx
                if gc is not None:
                    g_cb += gc
    return Ref(emb, res, lls, lls.sum(0), final, g_x, g_cb)


def check_ids_fp64(ids, res, cbs, rows_per_chunk_elems=1 << 27):
    """Every row and level: d64(chosen) - d64(min) <= NEAR_TIE_REL |d64(min)| on the fp64 residual `res` [L, N, D]
    (the residual that follows the kernel's own earlier choices).  Returns the number of rows that took a near-tie."""
    n_levels, n, _ = res.shape
    k = cbs.shape[1]
    assert int(ids.min()) >= 0 and int(ids.max()) < k, "ids out of range"
    step = max(1, rows_per_chunk_elems // k)
    near = torch.zeros(n, dtype=torch.bool, device=res.device)
    for l in range(n_levels):
        cb = cbs[l].double()
        cc = (cb * cb).sum(1)
        for s in range(0, n, step):
            r = res[l, s:s + step]
            table = (r * r).sum(1, keepdim=True) + cc[None] - 2.0 * r @ cb.T
            dmin = table.min(1).values
            dch = table.gather(1, ids[s:s + step, l:l + 1]).squeeze(1)
            gap = dch - dmin
            bad = gap > NEAR_TIE_REL * dmin.abs()
            assert not bool(bad.any()), (
                f"level {l}: {int(bad.sum())} rows chose a code farther than the near-tie allowance; worst relative gap "
                f"{float((gap / dmin.abs().clamp(min=1e-300)).max()):.3e} (rows {(torch.nonzero(bad).view(-1)[:8] + s).tolist()})")
            near[s:s + step] |= gap > 0
    return int(near.sum())


def ratio(got, ref, rtol, atol):
    """max |got - ref| / (atol + rtol |ref|): <= 1 means inside the bar (inf for a non-finite element)."""
    if got.numel() == 0:
        return 0.0
    got = got.double()
    if not bool(torch.isfinite(got).all()):
        return math.inf
    return float(((got - ref).abs() / (atol + rtol * ref.abs())).max())


def assert_bars(tag, ratios):
    print(f"fp64-ratio {tag}: " + ", ".join(f"{k} {v:.3g}" for k, v in ratios.items()))
    bad = {k: v for k, v in ratios.items() if not v <= 1.0}
    assert not bad, f"{tag}: outside the bar (ratio error / bar): {bad}"


def forward_ratios(out, ref):
    vec = lambda got, want: ratio(got, want, VAL[0], VAL[1] * max(1.0, float(want.abs().max())))
    r = {}
    if out.emb_out is not None:
        r["emb_out"] = vec(out.emb_out, ref.emb)
    if out.residuals is not None:
        r["residuals"] = vec(out.residuals, ref.res)
    if out.level_loss is not None:
        r["level_loss"] = ratio(out.level_loss, ref.level_loss, *VAL)
    if out.loss is not None:
        r["loss"] = ratio(out.loss, ref.loss, *VAL)
    if out.final_residual is not None:
        r["final_residual"] = vec(out.final_residual, ref.final)
    return r


def grad_ratios(g_x, g_cb, ref, rows=None):
    rx = ref.g_x if rows is None else ref.g_x[rows]
    gx = g_x if rows is None else g_x[rows]
    return {"g_x": ratio(gx, rx, GX[0], GX[1] * max(1.0, float(rx.abs().max()))),
            "g_codebooks": ratio(g_cb, ref.g_cb, GCB[0], GCB[1] * max(1.0, float(ref.g_cb.abs().max())))}


# ---------------------------------------------------------------------------------------------------------------------
# the instantiation matrix
# ---------------------------------------------------------------------------------------------------------------------
class Cell(NamedTuple):
    kernel: str     # expected instantiation
    d: int
    k: int
    L: int
    n: int
    mode: str       # "ste" | "rot" | "eval"
    algo: str       # forward algorithm ("" for a backward cell)
    grads: str      # backward: "full" (g_emb, g_loss[, g_level_loss]) | "bcast" (level stride 0, g_loss stride 0)
    g_ll: bool = False   # backward: pass g_level_loss

    @property
    def id(self):
        return f"{self.kernel}-n{self.n}-k{self.k}-L{self.L}-{self.mode}{'-' + self.algo if self.algo else ''}" + (
            f"-{self.grads}{'-gll' if self.g_ll else ''}" if not self.algo else "")


def _b(v):
    return "true" if v else "false"


def _flags(mname):
    mode, train = MODES[mname]
    return mode == ROT and train, train


def _bwd_cells():
    cells = []
    for mname in ("ste", "rot", "eval"):
        rot, train = _flags(mname)
        fl = f"{_b(rot)},{_b(train)}"
        for d in (16, 32, 64):                       # row kernel, exact level counts
            for L in (1, 2, 3, 4):
                cells.append(Cell(f"rq_bwd_kernel<{d},{fl},{L}>", d, 100, L, 1000 + 13 * L + d, mname, "",
                                  "full" if L % 2 else "bcast", g_ll=bool(L % 2)))
        for d in (4, 8, 16, 32, 64, 128):            # row kernel, runtime level count (NL = 0)
            for L in ((1, 3, 5, 8) if d in (4, 8, 128) else (5, 8)):
                cells.append(Cell(f"rq_bwd_kernel<{d},{fl},0>", d, 100, L, 1000 + 13 * L + d, mname, "",
                                  "full" if L % 2 else "bcast", g_ll=bool(L % 2)))
        for d in (16, 32, 64):                       # shared-memory kernel: N >= 65,536, L K D 4 <= 96 KB
            for L in (1, 2, 3, 4):
                k = min(256, 96 * 1024 // (4 * L * d))
                cells.append(Cell(f"rq_bwd_smem_kernel<{d},{8 if rot else 4},{fl},{L}>", d, k, L, 65536 + 2 * d + L, mname, "",
                                  "full" if L % 2 else "bcast"))
    # dispatch boundaries (D32 K256 L3 is the production shape and sits exactly on the 96 KB limit)
    cells += [
        Cell("rq_bwd_kernel<32,false,true,3>", 32, 256, 3, 65535, "ste", "", "full"),
        Cell("rq_bwd_smem_kernel<32,4,false,true,3>", 32, 256, 3, 65536, "ste", "", "full"),
        Cell("rq_bwd_smem_kernel<32,8,true,true,3>", 32, 256, 3, 65536, "rot", "", "full"),
        Cell("rq_bwd_kernel<32,true,true,3>", 32, 257, 3, 65536 + 5, "rot", "", "full"),
        Cell("rq_bwd_kernel<32,true,true,3>", 32, 256, 3, 65536 + 5, "rot", "", "full", g_ll=True),
    ]
    return cells


def _fwd_cells():
    cells = []
    for d in (4, 8, 16, 32, 64, 128):
        for algo in ("simt", "simt_diff"):
            for mname in ("eval", "ste", "rot"):
                rot, _ = _flags(mname)
                for k in (1, 129):
                    for L in (1, 5):
                        cells.append(Cell(f"rq_fwd_simt_kernel<{d},{_b(rot)},{_b(algo == 'simt_diff')}>", d, k, L,
                                          1000 + 7 * L + k % 7, mname, algo, ""))
    # generation 4: four warpgroups when every operand image stays resident, else two (streamed)
    for d, k, L, nwg in ((16, 256, 2, 4), (16, 4096, 2, 2), (32, 512, 1, 4), (32, 4096, 2, 2), (32, 256, 5, 2),
                         (32, 256, 8, 2), (64, 256, 1, 4), (64, 300, 2, 2)):
        for mname in ("eval", "rot"):
            rot, _ = _flags(mname)
            cells.append(Cell(f"rq_fwd_tc_kernel<{d},{_b(rot)},{nwg}>", d, k, L, 3000 + 77 + d, mname, "tcgen05", ""))
    # generation 11 (D = 32, K <= 256, L <= 3): no outputs (encode), outputs, rotation trick with outputs
    cells += [Cell("rq_fwd_tc_v11_kernel<false,false>", 32, 256, 3, 20000 + 33, "eval", "tcgen05_encode", ""),
              Cell("rq_fwd_tc_v11_kernel<false,true>", 32, 256, 3, 20000 + 33, "eval", "tcgen05", ""),
              Cell("rq_fwd_tc_v11_kernel<false,true>", 32, 200, 2, 20000 + 33, "ste", "tcgen05", ""),
              Cell("rq_fwd_tc_v11_kernel<true,true>", 32, 256, 3, 20000 + 33, "rot", "tcgen05", "")]
    return cells


BWD_CELLS = _bwd_cells()
FWD_CELLS = _fwd_cells()
# Gumbel: (D, N) with every backward CTA walking >= 3 tiles of 16 rows and every forward warp >= 3 rows (2 x 148 CTAs of
# 8 warps at D <= 32, 148 CTAs at D = 64 in the backward)
GUMBEL_SHAPES = [(16, 16384 + 5), (32, 16384 + 5), (64, 8192 + 3)]


def _inputs(cell, seed):
    x = unit_rows(cell.n, cell.d, seed=seed).cuda()
    cbs = make_codebooks(cell.L, cell.k, cell.d, seed=seed + 1).cuda()
    return x, cbs


def _grads(cell, seed):
    gen = torch.Generator().manual_seed(seed)
    if cell.grads == "bcast":   # the decoder's embs.sum(-1): one [N, D] gradient for every level; mean(): a stride-0 g_loss
        g_emb = torch.randn(cell.n, cell.d, generator=gen).cuda().expand(cell.L, cell.n, cell.d)
        g_loss = torch.full((1,), 1.0 / cell.n).cuda().expand(cell.n)
    else:
        g_emb = torch.randn(cell.L, cell.n, cell.d, generator=gen).cuda()
        g_loss = torch.randn(cell.n, generator=gen).cuda()
    g_ll = torch.randn(cell.L, cell.n, generator=gen).cuda() if cell.g_ll else None
    return g_emb, g_loss, g_ll


@pytest.mark.gpu
@pytest.mark.parametrize("cell", BWD_CELLS, ids=lambda c: c.id)
def test_backward_cell(ops, cell):
    """One backward instantiation against fp64 autograd along the forward's ids.  Worst ratio measured over all cells
    (B200): g_x 0.31, g_codebooks 0.04."""
    mode, train = MODES[cell.mode]
    x, cbs = _inputs(cell, seed=cell.n + cell.d + cell.L)
    ids = ops.rq_forward(x, cbs, mode, train, BETA, algo="simt").ids
    g_emb, g_loss, g_ll = _grads(cell, seed=cell.k + cell.L)
    if cell.grads == "bcast":
        assert g_emb.stride(0) == 0 and g_loss.stride(0) == 0
    (g_x, g_cb), launches = profiled(lambda: ops.rq_backward(x, cbs, ids, mode, train, BETA, g_emb, g_loss, g_ll))
    ref = reference(x, cbs, ids, mode, train, BETA, g_emb, g_loss, g_ll)
    assert_bars(cell.id, grad_ratios(g_x, g_cb, ref))
    skip = assert_launched(launches, {cell.kernel}, BWD_FAMILY)
    if skip:
        pytest.skip(skip)


@pytest.mark.gpu
@pytest.mark.parametrize("cell", FWD_CELLS, ids=lambda c: c.id)
def test_forward_cell(ops, cell):
    """One forward instantiation: ids on every row and level (fp64 near-tie rule), and every output value of every row
    against the fp64 chain along the kernel's ids.  Worst ratio measured over all cells (B200, before the atol of vector
    values was scaled): emb_out 0.63, residuals 1.5 (K = 1, rotation trick, L = 5, D = 8; every other cell <= 0.58),
    level_loss 0.32, loss 0.29, final_residual 0.91."""
    mode, train = MODES[cell.mode]
    x, cbs = _inputs(cell, seed=cell.n + cell.k + cell.L)
    if cell.algo == "tcgen05_encode":
        run = lambda: ops.rq_forward(x, cbs, mode, train, BETA, algo="tcgen05")
    else:
        run = lambda: ops.rq_forward(x, cbs, mode, train, BETA, want_emb=True, want_residuals=True, want_loss=True,
                                     want_level_loss=True, want_final_residual=True, algo=cell.algo)
    out, launches = profiled(run)
    ref = reference(x, cbs, out.ids, mode, train, BETA)
    check_ids_fp64(out.ids, ref.res, cbs)
    assert_bars(cell.id, forward_ratios(out, ref))
    skip = assert_launched(launches, {cell.kernel}, FWD_FAMILY)
    if skip:
        pytest.skip(skip)


@pytest.mark.gpu
def test_backward_replicas_start_at_32768_rows_and_match_direct_scatter(ops):
    """Gradient replicas (scratch copies of [L, K, D] the CTAs spread their reductions over) start at 32,768 rows; with
    and without them g_x is bit-identical and both codebook gradients meet the fp64 bar.  Worst ratio measured: g_x 0.17,
    g_codebooks 0.04."""
    d, k, L = 32, 256, 3
    assert ops.lib.hv_workspace_bytes(1, 32767, d, k, L) == 0 and ops.lib.hv_workspace_bytes(1, 32768, d, k, L) > 0
    cell = Cell("rq_bwd_kernel<32,true,true,3>", d, k, L, 32768, "rot", "", "full")
    x, cbs = _inputs(cell, seed=3)
    ids = ops.rq_forward(x, cbs, ROT, True, BETA, algo="simt").ids
    g_emb, g_loss, _ = _grads(cell, seed=4)
    ref = reference(x, cbs, ids, ROT, True, BETA, g_emb, g_loss)
    gx_a, gc_a = ops.rq_backward(x, cbs, ids, ROT, True, BETA, g_emb, g_loss, None)
    gx_b, gc_b = ops.rq_backward(x, cbs, ids, ROT, True, BETA, g_emb, g_loss, None, use_workspace=False)
    assert torch.equal(gx_a, gx_b)
    assert_bars("replicas", grad_ratios(gx_a, gc_a, ref))
    assert_bars("no replicas", grad_ratios(gx_b, gc_b, ref))


@pytest.mark.gpu
def test_backward_nine_levels_is_unsupported_without_a_launch(ops):
    from hidvae_b200 import _lib
    x = torch.zeros(100, 32, device="cuda")
    cbs = torch.zeros(9, 16, 32, device="cuda")
    ids = torch.zeros(100, 9, dtype=torch.int64, device="cuda")

    def call():
        with pytest.raises(_lib.HidvaeError, match="UNSUPPORTED"):
            ops.rq_backward(x, cbs, ids, STE, True, BETA, None, torch.ones(100, device="cuda"), None)

    _, launches = profiled(call)
    assert not {n for n in launches.names if family(n) in BWD_FAMILY}


def test_every_shipped_instantiation_has_a_cell():
    """Every instantiation of the quantiser and Gumbel kernels in the built library is the expected kernel of some cell of
    this file (CPU only: reads the library with cuobjdump)."""
    shipped = {k for k in shipped_kernels() if family(k) in FAMILIES}
    assert {family(s) for s in shipped} == set(FAMILIES), sorted(shipped)
    covered = {c.kernel for c in BWD_CELLS + FWD_CELLS}
    covered |= {f"{fam}<{d}>" for fam in GUMBEL_FAMILY for d, _ in GUMBEL_SHAPES}
    unreached = sorted(shipped - covered)
    assert not unreached, f"{len(unreached)} of {len(shipped)} shipped instantiations have no test cell: {unreached}"
    assert not sorted(covered - shipped), f"cells expect kernels the library does not ship: {sorted(covered - shipped)}"


@pytest.mark.parametrize("mname", ["ste", "rot", "eval"])
@pytest.mark.parametrize("grads", ["full", "bcast"])
def test_reference_matches_oracle_autograd(mname, grads):
    """The fp64 reference (gather along given ids) against oracle.rq_forward autograd (its own argmin) in float64 on the CPU,
    with g_emb, g_loss and g_level_loss (full) or a level-broadcast g_emb and a stride-0 g_loss (bcast)."""
    n, d, k, L = 300, 16, 32, 3
    mode, train = MODES[mname]
    x = unit_rows(n, d, seed=7).double()
    cbs = make_codebooks(L, k, d, seed=8).double()
    gen = torch.Generator().manual_seed(9)
    if grads == "bcast":
        g_emb, g_loss, g_ll = torch.randn(n, d, generator=gen).double().expand(L, n, d), torch.full((1,), 0.5).double().expand(n), None
    else:
        g_emb, g_loss, g_ll = (torch.randn(L, n, d, generator=gen).double(), torch.randn(n, generator=gen).double(),
                               torch.randn(L, n, generator=gen).double())
    x_o = x.clone().requires_grad_(True)
    cb_o = [cbs[l].clone().requires_grad_(True) for l in range(L)]
    o = O.rq_forward(x_o, cb_o, mode, BETA, train)
    obj = (o.embeddings * g_emb.permute(1, 2, 0)).sum() + (o.quantize_loss * g_loss).sum()
    if g_ll is not None:
        obj = obj + sum((ll * g_ll[l]).sum() for l, ll in enumerate(o.level_losses))
    obj.backward()
    ref = reference(x, cbs, o.sem_ids, mode, train, BETA, g_emb, g_loss, g_ll, chunk=128)
    close = dict(rtol=1e-12, atol=1e-13)
    torch.testing.assert_close(ref.emb, o.embeddings.detach().permute(2, 0, 1), **close)
    torch.testing.assert_close(ref.res, o.residuals.detach().permute(2, 0, 1), **close)
    torch.testing.assert_close(ref.loss, o.quantize_loss.detach(), **close)
    torch.testing.assert_close(ref.level_loss, torch.stack(o.level_losses).detach(), **close)
    torch.testing.assert_close(ref.g_x, x_o.grad, **close)
    torch.testing.assert_close(ref.g_cb, torch.stack([c.grad for c in cb_o]), **close)


# ---------------------------------------------------------------------------------------------------------------------
# the bench's training shapes at full size
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("shape,mname,fwd_kernel,bwd_kernel", [
    ((1 << 22, 32, 256, 3), "ste", "rq_fwd_tc_v11_kernel<false,true>", "rq_bwd_smem_kernel<32,4,false,true,3>"),
    ((1 << 22, 32, 256, 3), "rot", "rq_fwd_tc_v11_kernel<true,true>", "rq_bwd_smem_kernel<32,8,true,true,3>"),
    ((65536, 64, 4096, 4), "rot", "rq_fwd_tc_kernel<64,true,2>", "rq_bwd_kernel<64,true,true,4>"),
], ids=["bench_4Mi_ste", "bench_4Mi_rot", "c4_rot"])
def test_training_step_full_size(ops, shape, mname, fwd_kernel, bwd_kernel):
    """The training forward (rq_apply, tensor-core kernel) and its autograd backward at the size the benchmark runs, every
    row against fp64: ids, emb_out, loss, level_loss (a second forward call that also writes it: same kernel, same ids),
    g_x and the codebook gradient.  The 4 Mi-row backward runs the shared-memory kernel with about 300 row iterations per
    warp and gradient replicas; C4 runs the streamed forward and the row kernel with replicas.
    Worst ratio measured (B200): 4 Mi STE 0.10 (g_codebooks), 4 Mi rotation 0.55 (final residual), C4 0.47 (final residual)."""
    n, d, k, L = shape
    mode, train = MODES[mname]
    x = unit_rows(n, d, seed=91).cuda().requires_grad_(True)
    cbs = make_codebooks(L, k, d, seed=92).cuda().requires_grad_(True)
    gen = torch.Generator(device="cuda").manual_seed(93)
    g_emb = torch.randn(L, n, d, device="cuda", generator=gen)
    g_loss = torch.randn(n, device="cuda", generator=gen)

    def step():
        emb, _res, ids, loss, _ll = ops.rq_apply(x, cbs, mode, train, BETA, want_residuals=False, want_level_loss=False)
        torch.autograd.backward([emb, loss], [g_emb, g_loss])
        return emb.detach(), ids, loss.detach()

    (emb, ids, loss), launches = profiled(step)
    full = ops.rq_forward(x.detach(), cbs.detach(), mode, train, BETA, want_level_loss=True, want_final_residual=True)
    assert torch.equal(full.ids, ids)
    ref = reference(x, cbs, ids, mode, train, BETA, g_emb, g_loss, chunk=1 << 19)
    near = check_ids_fp64(ids, ref.res, cbs)
    r = {"emb_out": ratio(emb, ref.emb, *VAL), "loss": ratio(loss, ref.loss, *VAL)}
    r.update(forward_ratios(full, ref))
    r.update(grad_ratios(x.grad, cbs.grad, ref))
    assert_bars(f"{shape} {mname} (rows on a near-tie: {near})", r)
    skip = assert_launched(launches, {fwd_kernel}, FWD_FAMILY) or assert_launched(launches, {bwd_kernel}, BWD_FAMILY)
    if skip:
        pytest.skip(skip)


# ---------------------------------------------------------------------------------------------------------------------
# exact accounting of the codebook-gradient scatter
# ---------------------------------------------------------------------------------------------------------------------
ACCOUNTING = [(m, L, kern, rep) for m in ("eval", "ste") for L in (1, 3, 4, 5) for kern in ("row", "smem")
              for rep in (True, False) if not (kern == "smem" and L == 5)]


@pytest.mark.gpu
@pytest.mark.parametrize("mname,L,kernel,replicas", ACCOUNTING, ids=lambda v: str(v))
def test_gradient_scatter_accounting_is_exact(ops, mname, L, kernel, replicas):
    """Inputs whose fp32 result is exact, so that a lost, duplicated or wrongly folded row or replica shows as an inequality
    (4 Mi rows, D = 32, K = 128, random ids, g_loss = 0, g_emb small integers in [-4, 4]):
      * eval: G = 0, so g_x must be exactly 0 and the codebook gradient the per-code integer sum of g_emb (at most
        4 x 2^22 / 128 ~ 2^17 in magnitude, far below 2^24: exact in any order), equal to the fp64 index_add_ bit for bit;
      * STE training: G telescopes to g_emb of level 0 (every h = g_emb_l - G_{l+1} is a small integer), so g_x must equal
        g_emb[0] exactly and the codebook gradient (2 (e - r) g_loss) must be exactly 0.
    The row kernel is forced at this size by a zero g_level_loss."""
    n, d, k = (1 << 22) + 3, 32, 128
    mode, train = MODES[mname]
    gen = torch.Generator(device="cuda").manual_seed(100 + L)
    x = torch.randn(n, d, device="cuda", generator=gen)
    cbs = make_codebooks(L, k, d, seed=101).cuda()
    ids = torch.randint(0, k, (n, L), device="cuda", generator=gen)
    g_emb = torch.randint(-4, 5, (L, n, d), device="cuda", generator=gen).float()
    g_loss = torch.zeros(n, device="cuda")
    g_ll = torch.zeros(L, n, device="cuda") if kernel == "row" else None
    (g_x, g_cb), launches = profiled(lambda: ops.rq_backward(x, cbs, ids, mode, train, BETA, g_emb, g_loss, g_ll,
                                                             use_workspace=replicas))
    if train:
        assert torch.equal(g_x, g_emb[0]), "g_x != g_emb[level 0]"
        assert torch.equal(g_cb, torch.zeros_like(g_cb)), f"codebook gradient not 0: max |.| {float(g_cb.abs().max())}"
    else:
        assert torch.equal(g_x, torch.zeros_like(g_x)), f"g_x not 0: max |.| {float(g_x.abs().max())}"
        for l in range(L):
            ref = torch.zeros(k, d, dtype=torch.float64, device="cuda").index_add_(0, ids[:, l], g_emb[l].double())
            diff = (g_cb[l].double() - ref).abs()
            assert torch.equal(g_cb[l], ref.float()), f"level {l}: {int((diff > 0).sum())} elements differ, max {float(diff.max())}"
    assert ops.lib.hv_workspace_bytes(1, n, d, k, L) > 0
    fl = f"{_b(False)},{_b(train)}"
    expected = f"rq_bwd_kernel<32,{fl},{L if L <= 4 else 0}>" if kernel == "row" else f"rq_bwd_smem_kernel<32,4,{fl},{L}>"
    skip = assert_launched(launches, {expected}, BWD_FAMILY)
    if skip:
        pytest.skip(skip)


# ---------------------------------------------------------------------------------------------------------------------
# Gumbel-softmax level across tiles
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("temperature", [0.2, 1.0])
@pytest.mark.parametrize("k", [1, 31, 256])
@pytest.mark.parametrize("d,n", GUMBEL_SHAPES, ids=lambda v: str(v))
def test_gumbel_across_tiles(ops, d, n, k, temperature):
    """gumbel_apply forward and backward against fp64 autograd of oracle.quantize_level on the same uniforms, with enough rows
    that every backward CTA carries its per-code gradient across >= 3 tiles and every forward warp walks >= 3 rows.  Bars of
    tests/test_gpu_gumbel.py.  Worst ratio measured (B200): emb_out 0.18, loss 0.09, g_x 0.02, g_codebook 0.01.
    K = 1 found a kernel defect: the softmax term a_k = -w_k (ge.c_k - ge.emb) / T is exactly 0 when emb equals the code, but
    the kernel summed ge.emb in another order than ge.c_k, and the difference (fp32 noise times 1 / T) reached g_x at 77 times
    the bar; both sums now run in the same order."""
    gen = torch.Generator(device="cuda").manual_seed(n + k)
    x = unit_rows(n, d, seed=k).cuda()
    cb = F.normalize(torch.rand(k, d, generator=torch.Generator().manual_seed(k + d)), dim=-1).cuda()
    u = torch.rand(n, k, device="cuda", generator=gen)
    g_emb = torch.randn(n, d, device="cuda", generator=gen) * 0.1
    g_loss = torch.rand(n, device="cuda", generator=gen) / n
    x_d, cb_d = x.clone().requires_grad_(True), cb.clone().requires_grad_(True)

    def run():
        emb, ids, loss = ops.gumbel_apply(x_d, cb_d, temperature, BETA, uniforms=u)
        ((emb * g_emb).sum() + (loss * g_loss).sum()).backward()
        return emb.detach(), ids, loss.detach()

    (emb, ids, loss), launches = profiled(run)
    x_o, cb_o = x.double().requires_grad_(True), cb.double().requires_grad_(True)
    ref = O.quantize_level(x_o, cb_o, O.MODE_GUMBEL_SOFTMAX, BETA, True, temperature, uniform=u.double())
    ((ref.embeddings * g_emb.double()).sum() + (ref.loss * g_loss.double()).sum()).backward()
    check_ids_fp64(ids.view(-1, 1), x.double().unsqueeze(0), cb.unsqueeze(0))
    gs, cs = float(x_o.grad.abs().max()), float(cb_o.grad.abs().max())
    assert_bars(f"gumbel d{d} n{n} k{k} T{temperature}", {
        "emb_out": ratio(emb, ref.embeddings.detach(), *GUMBEL_VAL), "loss": ratio(loss, ref.loss.detach(), *GUMBEL_VAL),
        "g_x": ratio(x_d.grad, x_o.grad, GUMBEL_GRAD[0], GUMBEL_GRAD[1] * gs),
        "g_codebook": ratio(cb_d.grad, cb_o.grad, GUMBEL_GRAD[0], GUMBEL_GRAD[1] * cs)})
    skip = assert_launched(launches, {f"gumbel_fwd_kernel<{d}>", f"gumbel_bwd_kernel<{d}>"}, GUMBEL_FAMILY)
    if skip:
        pytest.skip(skip)


# ---------------------------------------------------------------------------------------------------------------------
# edges of the rotation trick in training
# ---------------------------------------------------------------------------------------------------------------------
EDGE_FWD = [("simt", 32), ("tcgen05", 32), ("tcgen05", 64)]   # exact fp32 kernel, generation 11, generation 4


def _edge_batch(edge, d, n):
    x = unit_rows(n, d, seed=200 + d)
    if edge == "zero_rows":
        cbs = make_codebooks(3, 256, d, seed=201)
        special = torch.arange(n) % 7 == 0
        x[special] = 0.0
    elif edge == "code_rows":
        cbs = make_codebooks(3, 256, d, seed=202)
        special = torch.arange(n) % 5 == 0
        x[special] = cbs[0][torch.arange(n)[special] % 256]
    else:   # "neg_code_k1": u + q = 0 exactly, the 1e-6 floor of |u + q| applies
        cbs = make_codebooks(2, 1, d, seed=203)
        special = torch.arange(n) % 3 == 0
        x[special] = -cbs[0][0]
    return x.cuda(), cbs.cuda(), special.cuda()


@pytest.mark.gpu
@pytest.mark.parametrize("edge", ["zero_rows", "code_rows", "neg_code_k1"])
@pytest.mark.parametrize("algo,d", EDGE_FWD, ids=lambda v: str(v))
def test_rotation_trick_edges(ops, edge, algo, d):
    """Rotation trick in training with degenerate rows mixed into a batch of 65,573 rows; forward on `algo`, backward on
    both backward kernels (shared-memory kernel; row kernel, forced by a g_level_loss).  Every output is finite.
      * zero rows: u = 0, w = q / |q|, o = 0 at every level -- well conditioned: every row is held to the bars.
      * rows equal to -c_0 with K = 1: u + q = 0 exactly (in fp32 and fp64), w = 0 by the 1e-6 floor, o = -r -- well
        conditioned (u, q are well defined): every row is held to the bars.
      * rows equal to a code: r_1 = r_0 - o_0 is rounding noise along r_0 (fp32 ~1e-7 |r|, fp64 ~4e-8 |r| from the 1e-8
        eps), so u_1 = r_1 / (|r_1| + 1e-8) has a norm anywhere in [0, 1) and possibly the other sign.  Every forward value
        after level 0 is O(|r_1|) in absolute terms and stays inside atol; the codebook gradient 2 (e - r) g_loss depends on
        r only in absolute terms and is held to its bar.  g_x passes the level-1 Jacobian h - 2 (h.w) w + 2 (h.q) u,
        which differs by up to 8 |h_1| between the two chains: on those rows the random-gradient run asserts only that g_x
        is finite and within 8 |g|-scales of the reference; a second run with a gradient at level 0 only (h_l = 0 for
        l >= 1, the level-0 Jacobian is well conditioned at r = e) holds every row to the bar.
    Worst ratio measured (B200): emb_out 0.24, residuals 0.35, final_residual 0.44, g_x 0.19, g_codebooks 0.06."""
    n = 65536 + 37
    mode, train = ROT, True
    x, cbs, special = _edge_batch(edge, d, n)
    L = cbs.shape[0]
    out = ops.rq_forward(x, cbs, mode, train, BETA, want_emb=True, want_residuals=True, want_loss=True, want_level_loss=True,
                         want_final_residual=True, algo=algo)
    for t in out[1:]:
        assert bool(torch.isfinite(t).all())
    ref = reference(x, cbs, out.ids, mode, train, BETA)
    check_ids_fp64(out.ids, ref.res, cbs)
    assert_bars(f"{edge} {algo} d{d} forward", forward_ratios(out, ref))

    gen = torch.Generator(device="cuda").manual_seed(204)
    g_emb = torch.randn(L, n, d, device="cuda", generator=gen)
    g_loss = torch.randn(n, device="cuda", generator=gen)
    g_ll = torch.randn(L, n, device="cuda", generator=gen)
    level0 = torch.zeros_like(g_emb)
    level0[0] = g_emb[0]
    level0_ll = torch.zeros_like(g_ll)
    level0_ll[0] = g_ll[0]
    runs = [("random", g_emb, g_loss, g_ll)]
    if edge == "code_rows":
        runs.append(("level 0 only", level0, None, level0_ll))
    for what, ge, gl, gll in runs:
        for kern, gll_arg in (("smem", None), ("row", gll)):
            g_x, g_cb = ops.rq_backward(x, cbs, out.ids, mode, train, BETA, ge, gl, gll_arg)
            assert bool(torch.isfinite(g_x).all()) and bool(torch.isfinite(g_cb).all())
            r = reference(x, cbs, out.ids, mode, train, BETA, ge, gl, gll_arg)
            tag = f"{edge} {algo} d{d} {kern} kernel, {what} gradient"
            if edge == "code_rows" and what == "random":
                scale = float(r.g_x.abs().max())
                assert float((g_x[special].double() - r.g_x[special]).abs().max()) <= 8 * scale, tag
                assert_bars(tag, grad_ratios(g_x, g_cb, r, rows=~special))
            else:
                assert_bars(tag, grad_ratios(g_x, g_cb, r))
