"""The fused encoder (enc_mlp_kernel, csrc/enc_mlp.cu) against a float64 reference that rounds where the kernel rounds, and
bit for bit on an integer-valued network.

tests/test_gpu_encoder.py holds the kernel to the fp32 oracle within 2e-3.  Most of that error is the fp16 rounding of the
operands, which does not depend on whether the kernel is right, so that bar cannot tell a correct kernel from a subtly
wrong one.  This file takes the rounding out of the comparison.

Reference (`reference`): plain torch in float64 on the device, chunked over rows.  x and every W are rounded to fp16 (round
to nearest even, satfinite emulated by clamping to +-65504 first), each GEMM runs in fp64, SiLU in fp64, every hidden
activation is rounded to fp16 (satfinite) as the next GEMM's operand, and the last layer and F.normalize(eps=1e-12) run in
fp64.  Each rounding to fp16 goes through fp32, as the kernel converts fp32 values.  fp16 subnormals are KEPT: the tcgen05
kind::f16 MMAs of the B200 honour subnormal operands from shared memory (x, W) and from tensor memory (hidden
activations), which test_fp16_subnormal_operands_are_kept pins exactly.  Two CPU tests pin the reference: without
rounding it is oracle.encoder.mlp_forward, with rounding it is a hand-written numpy fp16 chain.

What is left between kernel and reference is the fp32 accumulation inside the MMAs (its order and rounding are not
modelled) and the SiLU evaluation (ex2 + rcp for precise_silu=1, one tanh.approx for 0).  Both show up as hidden
activations that round to the neighbouring fp16 value.  Every instantiation enc_mlp_kernel<PRECISE, HALF_IN> runs with
normalize 0 and 1 on three weight sets: the suite's seeded nn.Linear-scale weights, a trained-like scale (hidden
activations of RMS 1) and a small scale that puts most hidden activations into fp16 subnormals.  Each cell checks max
|dz|, the RMS of dz and the share of rows whose max |dz| is <= 1e-5; when normalize=0, dz is divided by the RMS row norm
of z.  The bars (BARS) were measured on a B200 and set with about 2x margin.  With trained-like weights precise_silu=1
must also be strictly closer to the reference than precise_silu=0 (RMS 2.9e-5 against 3.9e-5).  At the two smaller
scales silu(a) is close to a / 2, the tanh term is below fp16 resolution, and both forms measure the same RMS to three
digits, so no order is asserted there.

Integer network (`int_weights`, `int_items`): sparse weights in {-1, 0, +1} with 4 non-zeros per output and items that are
multiples of 32.  Every pre-activation is then 0 or at least 32 in magnitude, and both SiLU forms round to ReLU in fp16:
silu(>= 32) rounds to the value, silu(<= -32) to +-0 (tanh.approx returns exactly +-1 for |h| >= 16).  Every value is an
integer multiple of 32 below 2^14, exact in fp16 and in fp32 accumulation, so the exact result is a ReLU chain in fp64
plus the kernel's fp32 normalize tail (`exact_tail`): a sequential fmaf sum of squares, sqrt.rn, rcp.rn, one multiply.
Those cases compare every row with torch.equal, at row counts from 1 to the bench's shard, and with entries and layer-1
pre-activations beyond 65504 (the clamps of satfinite).

Each cell asserts under torch.profiler which instantiation ran; test_every_shipped_instantiation_has_a_cell reads the
library with cuobjdump and fails when an instantiation has no cell.
"""
import functools

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from helpers import assert_launched, family, ops, profiled, shipped_kernels
from oracle import encoder as OE

DIMS = [768, 512, 256, 128, 32]
F16_MAX = 65504.0
SUBNORMALS_KEPT = True
FAMILIES = ("enc_mlp_kernel",)
KERNELS = {(p, h): f"enc_mlp_kernel<{'true' if p else 'false'},{'true' if h else 'false'}>" for p in (0, 1) for h in (0, 1)}
N_STAT = 148 * 128 + 77                       # every CTA busy, a ragged last tile
WITHIN = 1e-5

# (regime, precise, normalize) -> (max |dz|, RMS dz, least share of rows with max |dz| <= WITHIN).  Measured on a B200
# (1000 W power limit) at N_STAT rows, identical for fp32 and fp16 items: the bars are 2x the max and the RMS and half the
# share, rounded.  With hidden activations rounded toward zero (cvt.rz) every cell measures an RMS of 3.3x to 8.9x the
# correct kernel's and no row within 1e-5.
BARS = {
    ("seeded", 1, 0): (5.3e-4, 5.8e-5, 0.15),      # measured 2.65e-4, 2.92e-5, 0.313
    ("seeded", 1, 1): (6.2e-4, 5.9e-5, 0.15),      # 3.11e-4, 2.97e-5, 0.311
    ("seeded", 0, 0): (5.3e-4, 5.8e-5, 0.15),      # 2.65e-4, 2.92e-5, 0.315
    ("seeded", 0, 1): (6.2e-4, 5.9e-5, 0.15),      # 3.10e-4, 2.96e-5, 0.313
    ("trained", 1, 0): (7.3e-4, 5.7e-5, 0.21),     # 3.64e-4, 2.85e-5, 0.425
    ("trained", 1, 1): (7.5e-4, 5.8e-5, 0.21),     # 3.75e-4, 2.88e-5, 0.423
    ("trained", 0, 0): (7.6e-4, 7.9e-5, 0.02),     # 3.78e-4, 3.94e-5, 0.042
    ("trained", 0, 1): (8.2e-4, 8.0e-5, 0.02),     # 4.10e-4, 3.97e-5, 0.043
    ("subnormal", 1, 0): (1.4e-3, 1.2e-4, 0.38),   # 6.89e-4, 5.86e-5, 0.767
    ("subnormal", 1, 1): (1.5e-3, 1.2e-4, 0.38),   # 7.66e-4, 5.99e-5, 0.767
    ("subnormal", 0, 0): (1.4e-3, 1.2e-4, 0.38),   # 6.89e-4, 5.86e-5, 0.768
    ("subnormal", 0, 1): (1.5e-3, 1.2e-4, 0.38),   # 7.66e-4, 6.00e-5, 0.768
}


# ---------------------------------------------------------------------------------------------------------------------
# float64 reference
# ---------------------------------------------------------------------------------------------------------------------
def round_f16(t):
    """cvt.rn.satfinite.f16x2.f32 of t rounded to fp32 first (the kernel converts fp32 values), returned in t's dtype."""
    r = t.float().clamp(-F16_MAX, F16_MAX).half().to(t.dtype)
    if not SUBNORMALS_KEPT:
        r = torch.where(r.abs() < 2.0 ** -14, torch.zeros_like(r), r)
    return r


def reference(x, weights, normalize, rounding=True, chunk=1 << 18):
    """fp64 z [N, 32] of the MLP on x (fp32 or fp16, any device), rounding to fp16 where the kernel does when `rounding`."""
    ws = [w.to(x.device).double() for w in weights]
    if rounding:
        ws = [round_f16(w) for w in ws]
    out = torch.empty(x.shape[0], ws[-1].shape[0], dtype=torch.float64, device=x.device)
    for s in range(0, x.shape[0], chunk):
        h = x[s:s + chunk].double()
        if rounding:
            h = round_f16(h)
        for l, w in enumerate(ws):
            h = h @ w.T
            if l < len(ws) - 1:
                h = F.silu(h)
                if rounding:
                    h = round_f16(h)
        out[s:s + chunk] = F.normalize(h, p=2, dim=-1, eps=1e-12) if normalize else h
    return out


# ---------------------------------------------------------------------------------------------------------------------
# weights and items
# ---------------------------------------------------------------------------------------------------------------------
def unit_rows(n, seed):
    g = torch.Generator().manual_seed(seed)
    return F.normalize(torch.randn(n, DIMS[0], generator=g), dim=-1)


def scaled_weights(seed, act_rms, out_rms):
    """Gaussian weights scaled layer by layer on 2,048 unit rows so that every hidden activation has RMS `act_rms`
    and z has RMS `out_rms`."""
    g = torch.Generator().manual_seed(seed)
    h = unit_rows(2048, seed + 1).double()
    ws = []
    for l, (i, o) in enumerate(zip(DIMS[:-1], DIMS[1:])):
        w = torch.randn(o, i, generator=g, dtype=torch.float64)
        a = h @ w.T
        if l < 3:
            c = 1.0
            for _ in range(40):      # silu is not homogeneous: fixed point on the scale
                c *= act_rms / float(F.silu(c * a).pow(2).mean().sqrt())
        else:
            c = out_rms / float(a.pow(2).mean().sqrt())
        w *= c
        h = F.silu(h @ w.T) if l < 3 else h
        ws.append(w.float())
    return ws


@functools.lru_cache(maxsize=None)
def regime_weights(regime):
    if regime == "seeded":
        return OE.seeded_weights(DIMS, 2024)
    if regime == "trained":
        return scaled_weights(31, 1.0, 1.0)
    return scaled_weights(37, 2.0 ** -15, 2.0 ** -15)       # "subnormal": fp16 subnormals are |h| < 2^-14


def int_weights(seed, nnz=4):
    """Sparse integer weights [out, in]: `nnz` entries of +-1 per output, the rest 0."""
    g = torch.Generator().manual_seed(seed)
    ws = []
    for i, o in zip(DIMS[:-1], DIMS[1:]):
        cols = torch.rand(o, i, generator=g).argsort(dim=1)[:, :nnz]
        signs = (torch.randint(0, 2, (o, nnz), generator=g) * 2 - 1).float()
        ws.append(torch.zeros(o, i).scatter_(1, cols, signs))
    return ws


def int_items(n, seed, device="cuda", amp=3, chunk=1 << 20):
    """[N, 768] fp32 items 32 k, k uniform in [-amp, amp]."""
    g = torch.Generator(device=device).manual_seed(seed)
    x = torch.empty(n, DIMS[0], device=device)
    for s in range(0, n, chunk):
        e = min(n, s + chunk)
        x[s:e] = torch.randint(-amp, amp + 1, (e - s, DIMS[0]), generator=g, device=device, dtype=torch.float32)
    return x.mul_(32.0)


def int_chain(x, weights, chunk=1 << 18):
    """Exact z of the integer network: fp64 ReLU chain (integers below 2^53 are exact) with the satfinite clamps."""
    ws = [w.to(x.device).double() for w in weights]
    out = torch.empty(x.shape[0], DIMS[-1], dtype=torch.float64, device=x.device)
    for s in range(0, x.shape[0], chunk):
        h = x[s:s + chunk].double().clamp(-F16_MAX, F16_MAX)
        for l, w in enumerate(ws):
            h = h @ w.T
            if l < len(ws) - 1:
                h = h.clamp(0.0, F16_MAX)
        out[s:s + chunk] = h
    return out


def exact_tail(z64):
    """The kernel's normalize tail in fp32 on integer-valued z: ss = fmaf(z_d, z_d, ss) for d = 0..31 (each step is exact
    in fp64, then rounded once), inv = 1 / max(sqrt(ss), 1e-12) (sqrt.rn, rcp.rn), z * inv."""
    ss = torch.zeros(z64.shape[0], dtype=torch.float32, device=z64.device)
    for d in range(z64.shape[1]):
        ss = (ss.double() + z64[:, d] * z64[:, d]).float()
    inv = torch.ones_like(ss).div(torch.sqrt(ss).clamp(min=1e-12))
    return z64.float() * inv[:, None]


def exact_z(x, weights, normalize):
    z64 = int_chain(x, weights)
    return exact_tail(z64) if normalize else z64.float()


def run_cell(ops, x, image, precise, half_in, normalize, **kw):
    """encoder_forward under the profiler; asserts that exactly the expected instantiation ran."""
    xin = x.half() if half_in else x
    z, launches = profiled(lambda: ops.encoder_forward(xin, image, normalize=bool(normalize), precise_silu=bool(precise),
                                                       **kw))
    assert launches.recorded, "torch.profiler recorded no CUDA kernel"
    assert_launched(launches, {KERNELS[(precise, half_in)]}, FAMILIES)
    return z


def fwd(ops, x, image, precise, normalize=1, **kw):
    return ops.encoder_forward(x, image, normalize=bool(normalize), precise_silu=bool(precise), **kw)


def stats(z, ref, normalize):
    scale = 1.0 if normalize else float(ref.pow(2).sum(1).mean().sqrt())
    d = (z.double() - ref) / scale
    row = d.abs().amax(1)
    if not bool(torch.isfinite(z).all()):
        return {"max": float("inf"), "rms": float("inf"), "within": 0.0}
    return {"max": float(row.max()), "rms": float(d.pow(2).mean().sqrt()), "within": float((row <= WITHIN).double().mean())}


@functools.lru_cache(maxsize=None)
def stat_case(regime, normalize):
    x = unit_rows(N_STAT, 97).cuda()
    return x, reference(x, regime_weights(regime), normalize)


def instantiation_cells():
    return [(p, h, nz) for p in (0, 1) for h in (0, 1) for nz in (0, 1)]


def cell_id(c):
    return f"precise{c[0]}-half{c[1]}-norm{c[2]}"


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the references themselves
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("regime", ["seeded", "trained", "subnormal"])
@pytest.mark.parametrize("normalize", [0, 1])
def test_reference_without_rounding_is_the_fp32_oracle(regime, normalize):
    x = unit_rows(300, 5)
    w = regime_weights(regime)
    ref = reference(x, w, normalize, rounding=False)
    want = OE.mlp_forward(x, w, bool(normalize)).double()
    scale = float(want.abs().max())
    assert float((ref - want).abs().max()) <= 1e-5 * scale


def test_reference_with_rounding_is_a_numpy_half_chain():
    x = unit_rows(6, 8).numpy()
    for regime in ("seeded", "trained", "subnormal"):
        ws = [w.numpy() for w in regime_weights(regime)]
        ref = reference(torch.from_numpy(x), regime_weights(regime), 0).numpy()
        for r in range(x.shape[0]):
            h = x[r].astype(np.float16).astype(np.float64)
            for l, w in enumerate(ws):
                h = w.astype(np.float16).astype(np.float64) @ h
                if l < 3:
                    h = (h / (1.0 + np.exp(-h))).astype(np.float32).astype(np.float16).astype(np.float64)
            np.testing.assert_allclose(ref[r], h, rtol=1e-12, atol=1e-300)


def test_regimes_have_the_activation_scales_they_claim():
    x = unit_rows(1024, 3).double()
    for regime, lo, hi in (("trained", 0.7, 1.4), ("subnormal", 2.0 ** -16, 2.0 ** -14)):
        h = x
        for l, w in enumerate(regime_weights(regime)[:3]):
            h = F.silu(h @ w.double().T)
            rms = float(h.pow(2).mean().sqrt())
            assert lo <= rms <= hi, (regime, l, rms)
            if regime == "subnormal":
                assert float((h.abs() < 2.0 ** -14).double().mean()) >= 0.6, (l, "share of fp16 subnormals")


def test_integer_network_is_exact_and_the_tail_is_fp32_normalize():
    """The premises of the bit-exact cases: pre-activations are 0 or >= 32 in magnitude and below 2^14, the fp64 rounding
    reference equals the ReLU chain (so both SiLU forms must too), and the fp32 tail is F.normalize to fp32 precision."""
    w = int_weights(1)
    x = int_items(512, 2, device="cpu")
    h = x.double()
    for l, wl in enumerate(w):
        h = h @ wl.double().T
        assert float(h.abs().max()) < 2 ** 14 and bool((torch.remainder(h, 32) == 0).all())
        if l < 3:
            h = h.clamp(min=0)
    z = int_chain(x, w)
    assert torch.equal(z, h) and float((z != 0).double().mean()) > 0.8
    assert torch.equal(reference(x, w, 0), z)
    xs = x.clone()
    xs[:, ::3] *= 2048.0                          # entries up to 196,608 and layer-1 pre-activations beyond 65504
    zs = int_chain(xs, w)
    assert float(xs.abs().max()) > F16_MAX and torch.equal(reference(xs, w, 0), zs)
    for zz in (z, zs):
        tail = exact_tail(zz)
        torch.testing.assert_close(tail.double(), F.normalize(zz, dim=-1, eps=1e-12), rtol=0, atol=4e-7)


def test_every_shipped_instantiation_has_a_cell():
    """Every enc_mlp_kernel instantiation in the built library is the expected kernel of some cell (cuobjdump, CPU only)."""
    shipped = {k for k in shipped_kernels() if family(k) in FAMILIES}
    covered = {KERNELS[(p, h)] for p, h, _ in instantiation_cells()}
    assert shipped, "no enc_mlp_kernel in the library"
    assert not sorted(shipped - covered), f"shipped instantiations without a cell: {sorted(shipped - covered)}"
    assert not sorted(covered - shipped), f"cells expect kernels the library does not ship: {sorted(covered - shipped)}"


# ---------------------------------------------------------------------------------------------------------------------
# GPU: statistics against the fp64 reference
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("cell", instantiation_cells(), ids=cell_id)
@pytest.mark.parametrize("regime", ["seeded", "trained", "subnormal"])
def test_statistics_against_fp64(ops, regime, cell):
    """Worst ratio measured over all cells (B200): max 0.51, RMS 0.50, share of rows 0.50 (bar / measured)."""
    precise, half_in, normalize = cell
    x, ref = stat_case(regime, normalize)
    image = ops.encoder_pack([w.cuda() for w in regime_weights(regime)])
    z = run_cell(ops, x, image, precise, half_in, normalize)
    s = stats(z, ref, normalize)
    bmax, brms, bwithin = BARS[(regime, precise, normalize)]
    print(f"fp64-stats {regime} {cell_id(cell)}: max {s['max']:.3e} rms {s['rms']:.3e} within {s['within']:.4f} | ratio "
          f"max {s['max'] / bmax:.3g} rms {s['rms'] / brms:.3g} within {bwithin / max(s['within'], 1e-300):.3g}")
    assert s["max"] <= bmax and s["rms"] <= brms and s["within"] >= bwithin, (s, (bmax, brms, bwithin))


@pytest.mark.gpu
@pytest.mark.parametrize("half_in", [0, 1])
@pytest.mark.parametrize("normalize", [0, 1])
def test_precise_silu_is_closer_to_fp64_than_tanh(ops, normalize, half_in):
    """Trained-like weights: activations of O(1), where tanh.approx's error reaches fp16 resolution."""
    regime = "trained"
    x, ref = stat_case(regime, normalize)
    image = ops.encoder_pack([w.cuda() for w in regime_weights(regime)])
    rms = {p: stats(run_cell(ops, x, image, p, half_in, normalize), ref, normalize)["rms"] for p in (0, 1)}
    print(f"fp64-rms {regime} norm{normalize} half{half_in}: precise {rms[1]:.3e} tanh {rms[0]:.3e}")
    assert rms[1] < rms[0], rms


@pytest.mark.gpu
@pytest.mark.parametrize("case,x_exp,w1_exp", [("x", -21, 0), ("h", -13, -8), ("w", -5, -16)])
def test_fp16_subnormal_operands_are_kept(ops, case, x_exp, w1_exp):
    """Integer network at a scale where SiLU is x / 2 to within fp16 rounding: every hidden activation is an fp16
    subnormal, and so are the items (case x) or W1 (case w).  Kept subnormals give z = 2^-3 W4 W3 W2 W1 x exactly,
    flushed ones give 0."""
    w = int_weights(3)
    w[0] = w[0] * 2.0 ** w1_exp
    x = (int_items(4096, 4) / 32.0).clamp_(-1, 1) * 2.0 ** x_exp
    lin = x.double()
    for wl in w:
        lin = lin @ wl.cuda().double().T
    lin = lin / 8.0
    ref = reference(x, w, 0)
    assert torch.equal(ref, lin) == SUBNORMALS_KEPT and float((lin != 0).double().mean()) > 0.5
    image = ops.encoder_pack([wl.cuda() for wl in w])
    for p, h in KERNELS:
        z = run_cell(ops, x, image, p, h, 0)
        print(f"subnormal probe {case} precise{p} half{h}: equal to the linear chain {torch.equal(z.double(), lin)}, "
              f"zero {bool((z == 0).all())}")
        assert torch.equal(z, ref.float()), (case, p, h)


# ---------------------------------------------------------------------------------------------------------------------
# GPU: bit-exact integer network
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def int_net(ops):
    w = int_weights(1)
    return w, ops.encoder_pack([wl.cuda() for wl in w])


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 127, 128, 129, 148 * 128 - 1, 148 * 128 + 1, 1 << 20, (1 << 22) + 61])
def test_integer_network_is_bit_exact(ops, int_net, n):
    """Every row of every instantiation, normalize 0 and 1, with torch.equal.  2^20 rows is the bench's chunk and
    2^22 + 61 its shard (28 or more tiles per CTA)."""
    w, image = int_net
    x = int_items(n, n)
    xh = x.half()
    for normalize in (0, 1):
        want = exact_z(x, w, normalize)
        for p, h in KERNELS:
            z = fwd(ops, xh if h else x, image, p, normalize)
            if not torch.equal(z, want):
                bad = (z != want).any(1).nonzero().view(-1)
                pytest.fail(f"precise{p} half{h} norm{normalize}: {bad.numel()} of {n} rows differ, first {bad[:8].tolist()}")
        del want


@pytest.mark.gpu
@pytest.mark.parametrize("cell", instantiation_cells(), ids=cell_id)
def test_integer_network_saturates_like_satfinite(ops, int_net, cell):
    """Entries and layer-1 pre-activations beyond 65504: x and the hidden activations clamp to +-65504 (fp16 items can
    only hold the clamped catalogue)."""
    precise, half_in, normalize = cell
    w, image = int_net
    x = int_items(148 * 128 + 5, 6)
    x[:, ::3] *= 2048.0
    want = exact_z(x, w, normalize)
    a1 = x.double().clamp(-F16_MAX, F16_MAX) @ w[0].cuda().double().T
    assert float(x.abs().max()) > F16_MAX and float(a1.max()) > F16_MAX
    xin = x.clamp(-F16_MAX, F16_MAX) if half_in else x
    z = run_cell(ops, xin, image, precise, half_in, normalize)
    assert torch.equal(z, want)


# ---------------------------------------------------------------------------------------------------------------------
# GPU: row independence, isolation, bounds
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("half_in", [0, 1])
@pytest.mark.parametrize("precise", [0, 1])
@pytest.mark.parametrize("regime", ["seeded", "trained"])
def test_row_result_does_not_depend_on_the_call(ops, regime, precise, half_in):
    """The same row inside X, X[s:], X.flip(0) and short prefixes sits in another TMEM lane, tile and CTA and under another
    grid size: its z must be bit-identical."""
    n = 148 * 128 * 2 + 61
    image = ops.encoder_pack([w.cuda() for w in regime_weights(regime)])
    x = unit_rows(n, 41).cuda()
    if half_in:
        x = x.half()
    base = fwd(ops, x, image, precise)
    for s in (1, 37, 133):
        assert torch.equal(fwd(ops, x[s:], image, precise), base[s:]), s
    assert torch.equal(fwd(ops, x.flip(0), image, precise), base.flip(0))
    for p in (1, 5, 127, 129, 148 * 128 + 3):
        assert torch.equal(fwd(ops, x[:p], image, precise), base[:p]), p


@pytest.mark.gpu
@pytest.mark.parametrize("half_in", [0, 1])
@pytest.mark.parametrize("precise", [0, 1])
def test_nonfinite_items_stay_in_their_row(ops, precise, half_in):
    """NaN and +-inf entries change only their own row.  fp32 items saturate: an inf entry gives the row of 65504."""
    n = 148 * 128 + 77
    image = ops.encoder_pack([w.cuda() for w in regime_weights("trained")])
    x = unit_rows(n, 43).cuda()
    if half_in:
        x = x.half()
    base = fwd(ops, x, image, precise)
    rows = {0: (3, float("nan")), 200: (700, float("inf")), 128 * 70 + 64: (0, float("-inf")), n - 1: (767, float("nan"))}
    xb, xs = x.clone(), x.clone()
    for r, (c, v) in rows.items():
        xb[r, c] = v
        xs[r, c] = v if v != v else (F16_MAX if v > 0 else -F16_MAX)
    z = fwd(ops, xb, image, precise)
    keep = torch.ones(n, dtype=torch.bool, device="cuda")
    keep[list(rows)] = False
    assert torch.equal(z[keep], base[keep])
    if not half_in:
        sat = fwd(ops, xs, image, precise)
        for r, (_, v) in rows.items():
            if v == v:
                assert torch.equal(z[r], sat[r]), r


@pytest.mark.gpu
@pytest.mark.parametrize("half_in", [0, 1])
@pytest.mark.parametrize("n", [129, 148 * 128 + 77])
def test_reads_and_writes_stay_inside_n_rows(ops, n, half_in):
    """x is a prefix view of a buffer that is NaN past row N, and out= a slice of a larger sentinel buffer: z is
    unchanged and the sentinels are untouched."""
    image = ops.encoder_pack([w.cuda() for w in regime_weights("seeded")])
    x = unit_rows(n, 47).cuda()
    if half_in:
        x = x.half()
    base = fwd(ops, x, image, 1)
    buf = torch.full((n + 300, DIMS[0]), float("nan"), dtype=x.dtype, device="cuda")
    buf[:n] = x
    zbuf = torch.full((n + 256, DIMS[-1]), -7.0, device="cuda")
    out = zbuf[64:64 + n]
    z = fwd(ops, buf[:n], image, 1, out=out)
    assert z.data_ptr() == out.data_ptr() and torch.equal(out, base)
    assert bool((zbuf[:64] == -7.0).all()) and bool((zbuf[64 + n:] == -7.0).all())


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the fp16-catalogue boundary
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("precise", [0, 1])
def test_fp16_items_match_fp32_items_below_65520(ops, precise):
    """Below 65520, x.half() is finite and the fp16 entry gives the fp32 entry's z bit for bit.  From 65520 on, x.half()
    is inf while the fp32 entry saturates the item to +-65504: its z is finite and equals that of the clamped item, which
    x.clamp(-65504, 65504).half() reproduces."""
    n = 512
    image = ops.encoder_pack([w.cuda() for w in regime_weights("seeded")])
    x = unit_rows(n, 53).cuda()
    below = {1: 65504.0, 2: 65519.99, 3: -65519.99, 4: 60000.0}
    above = {5: 65520.0, 6: -65520.0, 7: 1.0e6, 8: float("inf")}
    for r, v in {**below, **above}.items():
        x[r, r * 13] = v
    z32 = fwd(ops, x, image, precise)
    z16 = fwd(ops, x.half(), image, precise)
    keep = torch.ones(n, dtype=torch.bool, device="cuda")
    keep[list(above)] = False
    assert bool(torch.isfinite(x.half()[keep]).all()) and torch.equal(z16[keep], z32[keep])
    assert bool(torch.isinf(x.half()[list(above)]).any(1).all())
    assert bool(torch.isfinite(z32).all())
    xc = x.clamp(-F16_MAX, F16_MAX)
    assert torch.equal(z32, fwd(ops, xc, image, precise))
    assert torch.equal(z32, fwd(ops, xc.half(), image, precise))
