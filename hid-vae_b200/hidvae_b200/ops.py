"""PyTorch-facing operators over the C ABI (include/hidvae_b200.h).

PyTorch is used here for device memory, streams and autograd bookkeeping only; every numeric result comes from
a kernel in libhidvae_b200.so.  Tensors must live on a CUDA device: there is no CPU path.

Mirrors, per function, the reference call sequence it replaces:
  rq_forward / RqFunction     modules/quantize.py:106-148 x L levels + modules/h_rqvae.py:515-523,552,572-574
  encoder_pack / encoder_forward   modules/encoder.py:23-36 (the MLP in front of the quantiser, eval passes)
  tag_heads_pack / _forward   modules/h_rqvae.py:69-99 + :385-389 (eval TagPredictor -> argmax / confidence)
  kmeans_*                    init/kmeans.py:43-61
  uniqueness_loss / count     modules/h_rqvae.py:41-105, :645-648
  semid_dedup / merge_runs    the collision digit of HSemanticIdTokenizer(use_dedup_dim=True)
"""
from __future__ import annotations

import ctypes
from typing import NamedTuple, Optional

import torch
from torch import Tensor

from . import _lib
from ._lib import (HV_ALGO_AUTO, HV_ALGO_SIMT, HV_ALGO_SIMT_DIFF, HV_ALGO_TCGEN05, HV_ALGO_TCGEN05_PREPACKED,
                   HV_MODE_ROTATION_TRICK, HV_MODE_STE, HV_OP_RQ_BACKWARD, HV_OP_RQ_FORWARD, check, lib)

ALGOS = {"auto": HV_ALGO_AUTO, "tcgen05": HV_ALGO_TCGEN05, "simt": HV_ALGO_SIMT, "simt_diff": HV_ALGO_SIMT_DIFF,
         "tcgen05_prepacked": HV_ALGO_TCGEN05_PREPACKED}


def _stream(t: Tensor) -> int:
    return torch.cuda.current_stream(t.device).cuda_stream


def _ptr(t: Optional[Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _require_cuda(*tensors: Tensor) -> None:
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise RuntimeError("hidvae_b200 operators run on CUDA tensors only (there is no CPU fallback); "
                               f"got a tensor on {t.device}")


def _f32c(t: Tensor) -> Tensor:
    if t.dtype != torch.float32:
        t = t.float()
    return t if t.is_contiguous() else t.contiguous()


def _algo(algo) -> int:
    return ALGOS[algo] if isinstance(algo, str) else int(algo)


class RqForwardResult(NamedTuple):
    ids: Tensor                     # [N, L] int64
    emb_out: Optional[Tensor]       # [L, N, D]
    residuals: Optional[Tensor]     # [L, N, D]
    loss: Optional[Tensor]          # [N]
    level_loss: Optional[Tensor]    # [L, N]
    final_residual: Optional[Tensor]  # [N, D]


def workspace_bytes(d: int, k: int, n_levels: int) -> int:
    return int(lib.hv_workspace_bytes(HV_OP_RQ_FORWARD, 0, d, k, n_levels))


def pack_codebooks(codebooks: Tensor) -> Optional[Tensor]:
    """Tensor-core operand image of the effective codebooks [L, K, D] (hv_rq_pack_codebooks), or None when the
    shape has no tcgen05 instantiation.  Pass it as `packed=` to rq_forward to skip the per-call pack launch."""
    _require_cuda(codebooks)
    codebooks = _f32c(codebooks)
    n_levels, k, d = codebooks.shape
    nbytes = workspace_bytes(d, k, n_levels)
    if not nbytes:
        return None
    ws = torch.empty(nbytes, dtype=torch.uint8, device=codebooks.device)
    with torch.cuda.device(codebooks.device):
        check(lib.hv_rq_pack_codebooks(codebooks.data_ptr(), n_levels, k, d, ws.data_ptr(), nbytes, _stream(codebooks)))
    return ws


def rq_forward(x: Tensor, codebooks: Tensor, mode: int = HV_MODE_STE, training: bool = False, beta: float = 0.25,
               want_emb: bool = False, want_residuals: bool = False, want_loss: bool = False,
               want_level_loss: bool = False, want_final_residual: bool = False, algo="auto",
               ids_out: Optional[Tensor] = None, packed: Optional[Tensor] = None) -> RqForwardResult:
    """One launch of the fused L-level quantiser (hv_rq_forward).  x [N, D], codebooks [L, K, D] (effective)."""
    _require_cuda(x, codebooks)
    x = _f32c(x)
    codebooks = _f32c(codebooks)
    if x.dim() != 2 or codebooks.dim() != 3 or x.shape[1] != codebooks.shape[2]:
        raise ValueError(f"rq_forward: x {tuple(x.shape)} and codebooks {tuple(codebooks.shape)} do not agree")
    n, d = x.shape
    n_levels, k, _ = codebooks.shape
    dev = x.device
    ids = ids_out if ids_out is not None else torch.empty((n, n_levels), dtype=torch.int64, device=dev)
    if ids.dtype != torch.int64 or ids.shape != (n, n_levels):
        raise ValueError("rq_forward: ids_out must be int64 [N, L]")
    new = lambda *shape: torch.empty(shape, dtype=torch.float32, device=dev)
    emb = new(n_levels, n, d) if want_emb else None
    res = new(n_levels, n, d) if want_residuals else None
    loss = new(n) if want_loss else None
    level_loss = new(n_levels, n) if want_level_loss else None
    final = new(n, d) if want_final_residual else None
    algo = _algo(algo)
    ws = None
    ws_bytes = 0
    if packed is not None:
        if algo not in (HV_ALGO_AUTO, HV_ALGO_TCGEN05, HV_ALGO_TCGEN05_PREPACKED):
            raise ValueError("rq_forward: `packed` only applies to the tcgen05 algorithm")
        algo, ws, ws_bytes = HV_ALGO_TCGEN05_PREPACKED, packed, packed.numel()
    elif algo in (HV_ALGO_AUTO, HV_ALGO_TCGEN05):
        ws_bytes = workspace_bytes(d, k, n_levels)
        if ws_bytes:
            ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        check(lib.hv_rq_forward(x.data_ptr(), n, d, codebooks.data_ptr(), n_levels, k, int(mode), int(bool(training)),
                                float(beta), ids.data_ptr(), ids.stride(0), ids.stride(1), _ptr(emb), _ptr(res),
                                _ptr(loss), _ptr(level_loss), _ptr(final), algo, _ptr(ws), ws_bytes, _stream(x)))
    return RqForwardResult(ids, emb, res, loss, level_loss, final)


def rq_backward(x: Tensor, codebooks: Tensor, ids: Tensor, mode: int, training: bool, beta: float,
                g_emb: Optional[Tensor], g_loss: Optional[Tensor], g_level_loss: Optional[Tensor],
                use_workspace: bool = True):
    """hv_rq_backward.  g_emb is indexed [L, N, D] (any strides with unit stride in D), g_loss [N] (any stride),
    g_level_loss [L, N].  Returns (g_x [N, D], g_codebooks [L, K, D]).  `use_workspace=False` withholds the
    gradient-replica scratch (large N then scatter-adds straight into g_codebooks; same result up to summation order)."""
    _require_cuda(x, codebooks, ids)
    x = _f32c(x)
    codebooks = _f32c(codebooks)
    n, d = x.shape
    n_levels, k, _ = codebooks.shape
    g_x = torch.empty_like(x)
    g_cb = torch.zeros_like(codebooks)
    ls = rs = 0
    if g_emb is not None:
        if g_emb.dtype != torch.float32:
            g_emb = g_emb.float()
        if (g_emb.stride(2) != 1 and d > 1) or g_emb.stride(0) % 4 or g_emb.stride(1) % 4 or g_emb.data_ptr() % 16:
            g_emb = g_emb.contiguous()
        ls, rs = g_emb.stride(0), g_emb.stride(1)
    gl_stride = 0
    if g_loss is not None:
        if g_loss.dtype != torch.float32:
            g_loss = g_loss.float()
        gl_stride = g_loss.stride(0) if g_loss.dim() else 0
    if g_level_loss is not None:
        g_level_loss = _f32c(g_level_loss)
    ws_bytes = int(lib.hv_workspace_bytes(HV_OP_RQ_BACKWARD, n, d, k, n_levels)) if use_workspace else 0
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=x.device) if ws_bytes else None
    with torch.cuda.device(x.device):
        check(lib.hv_rq_backward(x.data_ptr(), n, d, codebooks.data_ptr(), n_levels, k, int(mode), int(bool(training)),
                                 float(beta), ids.data_ptr(), ids.stride(0), ids.stride(1), _ptr(g_emb), ls, rs,
                                 _ptr(g_loss), gl_stride, _ptr(g_level_loss), g_x.data_ptr(), g_cb.data_ptr(),
                                 _ptr(ws), ws_bytes, _stream(x)))
    return g_x, g_cb


class RqFunction(torch.autograd.Function):
    """Differentiable fused residual quantiser.

    forward(x [N, D], codebooks [L, K, D], mode, training, beta, algo, want_residuals, want_level_loss)
        -> emb_out [L, N, D], residuals [L, N, D] (not differentiable), ids [N, L], loss [N], level_loss [L, N]
        (residuals / level_loss are empty placeholders when not wanted: 4DL + 4L bytes per item less to write)
    backward implements the recursion of SURVEY.md section 8a (autograd of modules/quantize.py:131-148 and
    modules/h_rqvae.py:552); the forward chain is recomputed, only x, codebooks and ids are saved."""

    @staticmethod
    def forward(ctx, x, codebooks, mode, training, beta, algo, want_residuals=True, want_level_loss=True):
        out = rq_forward(x, codebooks, mode, training, beta, want_emb=True, want_residuals=want_residuals, want_loss=True,
                         want_level_loss=want_level_loss, algo=algo)
        ctx.save_for_backward(x, codebooks, out.ids)
        ctx.cfg = (int(mode), bool(training), float(beta))
        residuals = out.residuals if want_residuals else x.new_empty(0)
        level_loss = out.level_loss if want_level_loss else x.new_empty(0)
        ctx.want_level_loss = bool(want_level_loss)
        ctx.mark_non_differentiable(out.ids, residuals)
        return out.emb_out, residuals, out.ids, out.loss, level_loss

    @staticmethod
    def backward(ctx, g_emb, _g_res, _g_ids, g_loss, g_level_loss):
        x, codebooks, ids = ctx.saved_tensors
        mode, training, beta = ctx.cfg
        g_x, g_cb = rq_backward(x, codebooks, ids, mode, training, beta, g_emb, g_loss,
                                g_level_loss if ctx.want_level_loss else None)
        return (g_x if ctx.needs_input_grad[0] else None, g_cb if ctx.needs_input_grad[1] else None,
                None, None, None, None, None, None)


def rq_apply(x: Tensor, codebooks: Tensor, mode: int, training: bool, beta: float, algo="auto",
             want_residuals: bool = True, want_level_loss: bool = True):
    """Autograd entry: returns (emb_out [L,N,D], residuals [L,N,D], ids [N,L], loss [N], level_loss [L,N]); residuals /
    level_loss come back as None when not wanted."""
    emb, res, ids, loss, ll = RqFunction.apply(x, codebooks, int(mode), bool(training), float(beta), algo,
                                               bool(want_residuals), bool(want_level_loss))
    return emb, (res if want_residuals else None), ids, loss, (ll if want_level_loss else None)


def rq_encode(x: Tensor, codebooks: Tensor, algo="auto", ids_out: Optional[Tensor] = None,
              packed: Optional[Tensor] = None) -> Tensor:
    """Encode-only (eval) semantic IDs [N, L] -- modules/tokenizer/h_semids.py:127-130."""
    return rq_forward(x, codebooks, HV_MODE_STE, False, 0.0, algo=algo, ids_out=ids_out, packed=packed).ids


# ------------------------------------------------------------------------------------------------------------------
# fused encoder MLP (modules/encoder.py:23-36) -- inference only: training keeps the PyTorch layers (autograd)
# ------------------------------------------------------------------------------------------------------------------
# ---------------------------------------------------------------------------------------------------------------
# Gumbel-softmax level (training mode of QuantizeForwardMode.GUMBEL_SOFTMAX)
# ---------------------------------------------------------------------------------------------------------------
def gumbel_supported(d: int, k: int) -> bool:
    return bool(lib.hv_gumbel_supported(int(d), int(k)))


def _device_rng(seed, device=None) -> Optional[Tensor]:
    """None for a host seed (a Python int); for a device seed the validated tensor (seed, offset): a CUDA int64 of two
    elements with values in [0, 2^62), on `device` when one is given."""
    if not isinstance(seed, Tensor):
        return None
    if not seed.is_cuda or seed.dtype != torch.int64 or seed.numel() != 2:
        raise ValueError("a device Gumbel seed is a CUDA int64 tensor of two elements (seed, offset); got "
                         f"{seed.dtype} {tuple(seed.shape)} on {seed.device}")
    if device is not None:
        device = torch.device(device)
        if device.type == "cuda" and device.index is None:
            device = torch.device("cuda", torch.cuda.current_device())
        if seed.device != device:
            raise ValueError(f"the device Gumbel seed is on {seed.device}, the operands on {device}")
    return seed.reshape(2).contiguous()


def gumbel_uniforms(n: int, k: int, seed, device=None) -> Tensor:
    """The [N, K] uniforms the fused Gumbel kernels draw for `seed` (recording / reproducing a step): a Python int, or a
    device pair (seed, offset) such as the one `gumbel_apply` saved (`device` then defaults to the pair's)."""
    rng = _device_rng(seed, device)
    out = torch.empty((n, k), dtype=torch.float32, device=device if rng is None else rng.device)
    with torch.cuda.device(out.device):
        if rng is None:
            check(lib.hv_gumbel_uniforms(n, k, int(seed), 0, out.data_ptr(), _stream(out)))
        else:
            check(lib.hv_gumbel_uniforms_devrng(n, k, rng.data_ptr(), out.data_ptr(), _stream(out)))
    return out


class GumbelFunction(torch.autograd.Function):
    """Fused Gumbel-softmax level: forward(x [N, D], codebook [K, D], temperature, beta, uniforms [N, K] | None, seed)
    -> emb_out [N, D], ids [N] (not differentiable), loss [N].  The noise is either the given uniforms (the reference's
    torch.rand draw) or Philox uniforms of `seed`, regenerated in the backward; dist / logits / weights never reach HBM.
    `seed` is a Python int or a CUDA int64 tensor (seed, offset) read by the kernels on the device; the backward reads the
    tensor the forward saved (the last of ctx.saved_tensors)."""

    @staticmethod
    def forward(ctx, x, codebook, temperature, beta, uniforms, seed):
        rng = _device_rng(seed)
        _require_cuda(x, codebook)
        x, codebook = _f32c(x), _f32c(codebook)
        n, d = x.shape
        k = codebook.shape[0]
        if rng is not None and rng.device != x.device:
            raise ValueError(f"the device Gumbel seed is on {rng.device}, x on {x.device}")
        if uniforms is not None:
            _require_cuda(uniforms)
            uniforms = _f32c(uniforms)
            assert uniforms.shape == (n, k)
        emb = torch.empty_like(x)
        ids = torch.empty((n,), dtype=torch.int64, device=x.device)
        loss = torch.empty((n,), dtype=torch.float32, device=x.device)
        lse = torch.empty((n,), dtype=torch.float32, device=x.device)
        with torch.cuda.device(x.device):
            if rng is None:
                check(lib.hv_gumbel_forward(x.data_ptr(), n, d, codebook.data_ptr(), k, float(temperature), float(beta),
                                            _ptr(uniforms), int(seed), 0, emb.data_ptr(), ids.data_ptr(), loss.data_ptr(),
                                            lse.data_ptr(), _stream(x)))
            else:
                check(lib.hv_gumbel_forward_devrng(x.data_ptr(), n, d, codebook.data_ptr(), k, float(temperature), float(beta),
                                                   _ptr(uniforms), rng.data_ptr(), emb.data_ptr(), ids.data_ptr(),
                                                   loss.data_ptr(), lse.data_ptr(), _stream(x)))
        ctx.save_for_backward(x, codebook, emb, lse, uniforms, rng)
        ctx.cfg = (float(temperature), float(beta), None if rng is not None else int(seed))
        ctx.mark_non_differentiable(ids)
        return emb, ids, loss

    @staticmethod
    def backward(ctx, g_emb, _g_ids, g_loss):
        x, codebook, emb, lse, uniforms, rng = ctx.saved_tensors
        temperature, beta, seed = ctx.cfg
        n, d = x.shape
        k = codebook.shape[0]
        g_emb = _f32c(g_emb) if g_emb is not None else None
        g_loss = _f32c(g_loss) if g_loss is not None else None
        g_x = torch.empty_like(x)
        g_cb = torch.zeros_like(codebook)
        with torch.cuda.device(x.device):
            if rng is None:
                check(lib.hv_gumbel_backward(x.data_ptr(), n, d, codebook.data_ptr(), k, temperature, beta, _ptr(uniforms), seed,
                                             0, emb.data_ptr(), lse.data_ptr(), _ptr(g_emb), _ptr(g_loss), g_x.data_ptr(),
                                             g_cb.data_ptr(), _stream(x)))
            else:
                check(lib.hv_gumbel_backward_devrng(x.data_ptr(), n, d, codebook.data_ptr(), k, temperature, beta,
                                                    _ptr(uniforms), rng.data_ptr(), emb.data_ptr(), lse.data_ptr(), _ptr(g_emb),
                                                    _ptr(g_loss), g_x.data_ptr(), g_cb.data_ptr(), _stream(x)))
        return g_x, g_cb, None, None, None, None


def gumbel_apply(x: Tensor, codebook: Tensor, temperature: float, beta: float, uniforms: Optional[Tensor] = None,
                 seed=None):
    """(emb_out [N, D], ids [N], loss [N]) of one Gumbel-softmax level.  Without `uniforms` the noise comes from Philox with
    `seed`: a Python int, or a CUDA int64 tensor (seed, offset) read on the device.  The default draws a fresh seed: eagerly
    from torch's CPU generator (so torch.manual_seed makes a run reproducible); under CUDA-graph capture as a (seed, 0)
    tensor from torch's CUDA generator, so that every replay of the graph draws anew."""
    if seed is None:
        if torch.cuda.is_current_stream_capturing():
            # a host draw would be frozen into the graph; torch's CUDA generator is graph-safe: every replay advances its
            # Philox offset, so every replay draws a new seed
            seed = torch.zeros(2, dtype=torch.int64, device=x.device)
            seed[:1].random_(0, 2 ** 62)
        else:
            seed = int(torch.randint(0, 2 ** 62, (1,)).item())
    elif not isinstance(seed, Tensor):
        seed = int(seed)
    return GumbelFunction.apply(x, codebook, float(temperature), float(beta), uniforms, seed)


def _dims_array(dims):
    return (ctypes.c_int * len(dims))(*[int(v) for v in dims])


def encoder_supported(dims) -> bool:
    """True when the fused kernel has an instantiation for the MLP widths [in, hidden..., out]."""
    return int(lib.hv_encoder_workspace_bytes(len(dims) - 1, _dims_array(dims))) > 0


class EncoderImage(NamedTuple):
    data: Tensor          # uint8: the fp16 tensor-core image of every layer's weights
    dims: tuple           # (in, hidden..., out)


def encoder_pack(weights) -> EncoderImage:
    """fp16 tensor-core image of the Linear weights [out_l, in_l] (hv_encoder_pack_weights).  Pack once per set of
    weights and pass the result to encoder_forward."""
    weights = [_f32c(w.detach()) for w in weights]
    _require_cuda(*weights)
    dims = [weights[0].shape[1]] + [w.shape[0] for w in weights]
    arr = _dims_array(dims)
    nbytes = int(lib.hv_encoder_workspace_bytes(len(weights), arr))
    if not nbytes:
        raise _lib.HidvaeError(_lib.HV_ERR_UNSUPPORTED, f"no fused encoder instantiation for widths {dims}")
    image = torch.empty(nbytes, dtype=torch.uint8, device=weights[0].device)
    ptrs = (ctypes.c_void_p * len(weights))(*[w.data_ptr() for w in weights])
    with torch.cuda.device(image.device):
        check(lib.hv_encoder_pack_weights(ptrs, len(weights), arr, image.data_ptr(), nbytes, _stream(image)))
    return EncoderImage(image, tuple(int(v) for v in dims))


def encoder_forward(x: Tensor, image: EncoderImage, normalize: bool = False, precise_silu: bool = False,
                    out: Optional[Tensor] = None) -> Tensor:
    """z [N, out] = the MLP applied to x [N, in] (hv_encoder_forward / hv_encoder_forward_f16): one fused tcgen05 kernel.
    x is fp32, or fp16 -- a catalogue kept in half precision moves half the bytes; the kernel rounds fp32 items to fp16 before
    the first GEMM anyway, so `x.half()` gives bit-identical z."""
    image, dims = image.data, image.dims
    _require_cuda(x, image)
    half_in = x.dtype == torch.float16
    x = x.contiguous() if half_in else _f32c(x)
    if x.dim() != 2 or x.shape[1] != dims[0]:
        raise ValueError(f"encoder_forward: x {tuple(x.shape)} does not match the encoder input width {dims[0]}")
    n = x.shape[0]
    z = out if out is not None else torch.empty((n, dims[-1]), dtype=torch.float32, device=x.device)
    if z.shape != (n, dims[-1]) or z.dtype != torch.float32 or not z.is_contiguous():
        raise ValueError("encoder_forward: out must be contiguous fp32 [N, out]")
    with torch.cuda.device(x.device):
        fn = lib.hv_encoder_forward_f16 if half_in else lib.hv_encoder_forward
        check(fn(x.data_ptr(), n, len(dims) - 1, _dims_array(dims), image.data_ptr(), image.numel(),
                 int(bool(normalize)), int(bool(precise_silu)), z.data_ptr(), _stream(x)))
    return z


# ------------------------------------------------------------------------------------------------------------------
# tag heads (modules/h_rqvae.py TagPredictor, eval mode) -- inference only: training keeps the PyTorch heads
# ------------------------------------------------------------------------------------------------------------------
def _tag_shape_args(n_levels, d, first_hidden, class_counts, use_norm):
    counts = (ctypes.c_int * len(class_counts))(*[int(c) for c in class_counts])
    return int(n_levels), int(d), int(first_hidden), counts, int(bool(use_norm))


def tag_heads_supported(n_levels: int, d: int, first_hidden: int, class_counts, use_norm: bool) -> bool:
    """True when hv_tag_heads_forward serves this HRqVae shape (len(class_counts) must be n_levels)."""
    if len(class_counts) != n_levels:
        return False
    return int(lib.hv_tag_heads_workspace_bytes(*_tag_shape_args(n_levels, d, first_hidden, class_counts, use_norm), 1,
                                                None)) > 0


class TagHeadsImage(NamedTuple):
    data: Tensor          # uint8: fp16 weight blocks and fp32 biases / LayerNorm parameters of every level
    shape: tuple          # (n_levels, d, first_hidden, class_counts, use_norm)


def tag_heads_pack(params, d: int, first_hidden: int, class_counts, use_norm: bool) -> TagHeadsImage:
    """Image of the tag heads (hv_tag_heads_pack).  `params`: every level's TagPredictor.parameters(), level by level."""
    params = [_f32c(p.detach()) for p in params]
    _require_cuda(*params)
    n_levels = len(class_counts)
    shape = _tag_shape_args(n_levels, d, first_hidden, class_counts, use_norm)
    nbytes = ctypes.c_size_t(0)
    if not int(lib.hv_tag_heads_workspace_bytes(*shape, 1, ctypes.byref(nbytes))):
        raise _lib.HidvaeError(_lib.HV_ERR_UNSUPPORTED, f"no tag-head instantiation for L={n_levels}, D={d}, "
                               f"hidden={first_hidden}, classes={list(class_counts)}")
    image = torch.empty(nbytes.value, dtype=torch.uint8, device=params[0].device)
    ptrs = (ctypes.c_void_p * len(params))(*[p.data_ptr() for p in params])
    with torch.cuda.device(image.device):
        check(lib.hv_tag_heads_pack(ptrs, len(params), *shape, image.data_ptr(), nbytes.value, _stream(image)))
    return TagHeadsImage(image, (n_levels, int(d), int(first_hidden), tuple(int(c) for c in class_counts), bool(use_norm)))


def tag_heads_forward(emb: Tensor, image: TagHeadsImage, pred_out: Optional[Tensor] = None,
                      conf_out: Optional[Tensor] = None, logits_out=None):
    """(pred [N, L] int64, conf [N, L] fp32 or None) of the tag heads on level embeddings emb [L, N, D] fp32 (any strides
    with a contiguous last dimension).  `pred_out` / `conf_out` may be strided [N, L] views -- e.g. the tag columns of an
    id table -- and are written in place; `logits_out` is an optional list of L fp32 [N, C_i] tensors."""
    n_levels, d, first_hidden, counts, use_norm = image.shape
    _require_cuda(emb, image.data)
    if emb.dtype != torch.float32 or emb.dim() != 3 or emb.shape[0] < n_levels or emb.shape[2] != d or emb.stride(2) != 1:
        raise ValueError(f"tag_heads_forward: emb must be fp32 [>= {n_levels}, N, {d}] with a contiguous last dimension, "
                         f"got {emb.dtype} {tuple(emb.shape)}")
    n = emb.shape[1]
    if pred_out is None:
        pred_out = torch.empty((n, n_levels), dtype=torch.int64, device=emb.device)
    for name, t, dt in (("pred_out", pred_out, torch.int64), ("conf_out", conf_out, torch.float32)):
        if t is not None and (t.dtype != dt or t.shape != (n, n_levels) or t.device != emb.device):
            raise ValueError(f"tag_heads_forward: {name} must be {dt} [{n}, {n_levels}] on {emb.device}")
    logit_ptrs = None
    if logits_out is not None:
        for t, c in zip(logits_out, counts):
            if t.dtype != torch.float32 or t.shape != (n, c) or not t.is_contiguous():
                raise ValueError(f"tag_heads_forward: logits_out entries must be contiguous fp32 [{n}, C_i]")
        logit_ptrs = (ctypes.c_void_p * n_levels)(*[t.data_ptr() for t in logits_out])
    shape = _tag_shape_args(n_levels, d, first_hidden, counts, use_norm)
    ws_bytes = int(lib.hv_tag_heads_workspace_bytes(*shape, n, None))
    workspace = torch.empty(ws_bytes, dtype=torch.uint8, device=emb.device)
    with torch.cuda.device(emb.device):
        check(lib.hv_tag_heads_forward(
            emb.data_ptr(), emb.stride(0), emb.stride(1), n, *shape, image.data.data_ptr(), image.data.numel(),
            pred_out.data_ptr(), pred_out.stride(0), pred_out.stride(1),
            _ptr(conf_out), conf_out.stride(0) if conf_out is not None else 0, conf_out.stride(1) if conf_out is not None else 0,
            logit_ptrs, workspace.data_ptr(), ws_bytes, _stream(emb)))
    return pred_out, conf_out


# ------------------------------------------------------------------------------------------------------------------
# k-means (init/kmeans.py)
# ------------------------------------------------------------------------------------------------------------------
def kmeans_assign(x: Tensor, centroids: Tensor, exact_diff_form: bool = True) -> Tensor:
    """argmin_k |x - c_k|^2 -> [N] int64 (init/kmeans.py:44-47).  `exact_diff_form` evaluates sum (x-c)^2 like the
    reference; otherwise the tensor-core GEMM form is used (same near-tie policy as the quantiser)."""
    algo = HV_ALGO_SIMT_DIFF if exact_diff_form else HV_ALGO_AUTO
    return rq_forward(x, centroids.unsqueeze(0), HV_MODE_STE, False, 0.0, algo=algo).ids.view(-1)


def _sort_workspace(n: int, device) -> Optional[Tensor]:
    """Scratch of the key sort behind the segmented k-means update and the sorted uniqueness pass (None for n == 0)."""
    nbytes = int(lib.hv_sort_workspace_bytes(n))
    return torch.empty(nbytes, dtype=torch.uint8, device=device) if nbytes else None


def kmeans_accumulate(x: Tensor, assign: Tensor, k: int, prev_assign: Optional[Tensor] = None):
    """Deterministic per-cluster sums [K, D], counts [K] and the number of changed assignments (0-d int64).
    `assign` and `prev_assign` are int64 [N] with values in [0, k)."""
    if x.dim() != 2:
        raise ValueError("kmeans_accumulate: x must be [N, D]")
    n, d = x.shape
    for name, a in (("assign", assign), ("prev_assign", prev_assign)):
        if a is not None and (a.dtype != torch.int64 or tuple(a.shape) != (n,)):
            raise ValueError(f"kmeans_accumulate: {name} must be int64 [{n}], got {a.dtype} {list(a.shape)}")
    _require_cuda(x, assign, prev_assign)
    x = _f32c(x)
    sums = torch.empty((k, d), dtype=torch.float32, device=x.device)
    counts = torch.empty((k,), dtype=torch.float32, device=x.device)
    changed = torch.empty((), dtype=torch.int64, device=x.device)
    assign = assign.contiguous()
    if prev_assign is not None:
        prev_assign = prev_assign.contiguous()
    ws = _sort_workspace(n, x.device) if k * n > (1 << 24) else None
    with torch.cuda.device(x.device):
        check(lib.hv_kmeans_accumulate(x.data_ptr(), n, d, assign.data_ptr(), _ptr(prev_assign), k, sums.data_ptr(),
                                       counts.data_ptr(), changed.data_ptr(), _ptr(ws), ws.numel() if ws is not None else 0,
                                       _stream(x)))
    return sums, counts, changed


def kmeans_finalize(sums: Tensor, counts: Tensor, centroids: Tensor, reseed_rows: Optional[Tensor] = None) -> Tensor:
    """centroids (in place) <- means / reseeds; returns stats [2] = (max centroid shift, number of empty clusters)."""
    _require_cuda(sums, counts, centroids)
    k, d = centroids.shape
    if not centroids.is_contiguous() or centroids.dtype != torch.float32:
        raise ValueError("kmeans_finalize: centroids must be contiguous fp32 (updated in place)")
    stats = torch.empty((2,), dtype=torch.float32, device=centroids.device)
    if reseed_rows is not None:
        reseed_rows = _f32c(reseed_rows)
    with torch.cuda.device(centroids.device):
        check(lib.hv_kmeans_finalize(sums.data_ptr(), counts.data_ptr(), _ptr(reseed_rows), k, d, centroids.data_ptr(),
                                     stats.data_ptr(), _stream(centroids)))
    return stats


# ------------------------------------------------------------------------------------------------------------------
# uniqueness loss / p_unique_ids (modules/h_rqvae.py:41-105, :645-648)
# ------------------------------------------------------------------------------------------------------------------
def uniq_stats(ids: Tensor, feats: Optional[Tensor], margin: float) -> Tensor:
    """stats [3] double: (sum of hinges over identical pairs i<j, number of such pairs, rows with a later twin)."""
    if ids.dtype != torch.int64 or ids.dim() != 2:
        raise ValueError("uniq_stats: ids must be int64 [rows, width]")
    rows, width = ids.shape
    if feats is not None and (feats.dim() != 2 or feats.shape[0] < rows):
        raise ValueError(f"uniq_stats: feats must be [>= {rows}, D] (one row per id row), got {list(feats.shape)}")
    _require_cuda(ids)
    d = 0
    if feats is not None:
        _require_cuda(feats)
        feats = _f32c(feats)
        d = feats.shape[1]
    stats = torch.empty((3,), dtype=torch.float64, device=ids.device)
    ws = _sort_workspace(rows, ids.device) if rows >= 4096 else None
    with torch.cuda.device(ids.device):
        check(lib.hv_uniq_forward(ids.data_ptr(), rows, width, ids.stride(0), ids.stride(1), _ptr(feats), d,
                                  float(margin), stats.data_ptr(), _ptr(ws), ws.numel() if ws is not None else 0, _stream(ids)))
    return stats


class UniqFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, feats, ids, margin, weight):
        feats_c = _f32c(feats)
        stats = uniq_stats(ids, feats_c, margin)
        ctx.save_for_backward(feats_c, ids, stats)
        ctx.cfg = (float(margin), float(weight))
        pairs = stats[1]
        mean = torch.where(pairs > 0, stats[0] / pairs.clamp(min=1.0), torch.zeros_like(pairs))
        return (weight * mean).to(torch.float32)

    @staticmethod
    def backward(ctx, g_out):
        feats, ids, stats = ctx.saved_tensors
        margin, weight = ctx.cfg
        g_feats = torch.zeros_like(feats)
        g = g_out.contiguous().float().reshape(1)
        rows, width = ids.shape
        ws = _sort_workspace(rows, feats.device) if rows >= 4096 else None
        with torch.cuda.device(feats.device):
            check(lib.hv_uniq_backward(ids.data_ptr(), rows, width, ids.stride(0), ids.stride(1), feats.data_ptr(),
                                       feats.shape[1], margin, weight, stats.data_ptr(), g.data_ptr(),
                                       g_feats.data_ptr(), _ptr(ws), ws.numel() if ws is not None else 0, _stream(feats)))
        return g_feats, None, None, None


def uniqueness_loss(ids: Tensor, feats: Tensor, margin: float, weight: float) -> Tensor:
    """weight * mean_{i<j, ids_i == ids_j} relu(cos(f_i, f_j) - margin); 0 when there is no such pair.
    `ids` is [rows, width]; no host synchronisation (the reference syncs in torch.where, h_rqvae.py:73)."""
    return UniqFunction.apply(feats, ids, float(margin), float(weight))


def count_rows_with_later_twin(ids: Tensor) -> Tensor:
    """0-d double tensor: number of rows that have a LATER identical row; p_unique_ids = 1 - this / rows."""
    return uniq_stats(ids, None, 0.0)[2]


# ------------------------------------------------------------------------------------------------------------------
# semantic-ID collision digit (HSemanticIdTokenizer(use_dedup_dim=True))
# ------------------------------------------------------------------------------------------------------------------
class DedupResult(NamedTuple):
    digits: Tensor      # [rows] int64: earlier rows (and prior rows) with the same tuple; -1 for a row with an id out of range
    run_keys: Tensor    # [rows] int64 capacity: the call's distinct tuple keys, ascending; the first stats[0] are valid
    run_counts: Tensor  # [rows] int64 capacity: rows of the call holding each key
    stats: Tensor       # [3] int64: distinct tuples, largest digit (-1 if none), rows with an id outside [0, 2^bits)


def dedup_bits(codebook_size: int) -> int:
    """Bits of one id in the exact tuple key: ceil(log2 K), at least 1."""
    return max(1, (int(codebook_size) - 1).bit_length())


def dedup_key(ids: Tensor, bits: int) -> Tensor:
    """The kernel's key of every tuple, in torch: sum_c ids[c] << bits * (width - 1 - c) (ids must lie in [0, 2^bits))."""
    width = ids.shape[-1]
    shifts = torch.arange(width - 1, -1, -1, device=ids.device, dtype=torch.int64) * int(bits)
    return (ids.to(torch.int64) << shifts).sum(-1)


def semid_dedup(ids: Tensor, bits: int, prior=None, digits_out: Optional[Tensor] = None) -> DedupResult:
    """Collision digit of every row of `ids` [rows, width] (any strides): the number of earlier rows with the same tuple,
    plus that tuple's count in `prior` = (keys, counts), the ascending keys of tuples seen before these rows and how often
    (e.g. merge_runs of the lower ranks' run lists).  hv_semid_dedup: one stable radix sort of exact keys, no host sync.
    `digits_out` (int64 [rows], any stride, e.g. column L of an [N, L + 1] table) receives the digits in place.
    width * bits must be <= 63 (the key is exact); wider shapes raise ValueError."""
    if ids.dtype != torch.int64 or ids.dim() != 2:
        raise ValueError("semid_dedup: ids must be int64 [rows, width]")
    rows, width = ids.shape
    bits = int(bits)
    if bits < 1 or width < 1 or width * bits > 63:
        raise ValueError(f"semid_dedup: width {width} x {bits} bits does not fit an exact 63-bit key")
    _require_cuda(ids)
    dev = ids.device
    digits = digits_out if digits_out is not None else torch.empty((rows,), dtype=torch.int64, device=dev)
    if digits.dtype != torch.int64 or digits.shape != (rows,) or digits.device != dev:
        raise ValueError("semid_dedup: digits_out must be int64 [rows] on the device of ids")
    prior_keys = prior_counts = None
    n_prior = 0
    if prior is not None:
        prior_keys, prior_counts = prior
        _require_cuda(prior_keys, prior_counts)
        prior_keys, prior_counts = prior_keys.to(torch.int64).contiguous(), prior_counts.to(torch.int64).contiguous()
        n_prior = prior_keys.numel()
        if prior_counts.numel() != n_prior:
            raise ValueError("semid_dedup: prior keys and counts differ in length")
    run_keys = torch.empty((rows,), dtype=torch.int64, device=dev)
    run_counts = torch.empty((rows,), dtype=torch.int64, device=dev)
    stats = torch.empty((3,), dtype=torch.int64, device=dev)
    ws_bytes = int(lib.hv_semid_dedup_workspace_bytes(rows))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev) if ws_bytes else None
    with torch.cuda.device(dev):
        check(lib.hv_semid_dedup(ids.data_ptr(), rows, width, ids.stride(0), ids.stride(1), bits,
                                 _ptr(prior_keys) if n_prior else None, _ptr(prior_counts) if n_prior else None, n_prior,
                                 digits.data_ptr(), digits.stride(0), run_keys.data_ptr(), run_counts.data_ptr(),
                                 stats.data_ptr(), _ptr(ws), ws_bytes, _stream(ids)))
    return DedupResult(digits, run_keys, run_counts, stats)


def merge_runs(runs):
    """[(keys, counts), ...] -> (keys, counts): the union of run lists, ascending, with the counts of equal keys added."""
    runs = list(runs)
    if not runs:
        raise ValueError("merge_runs: no run list given")
    keys = torch.cat([k.reshape(-1).to(torch.int64) for k, _ in runs])
    counts = torch.cat([c.reshape(-1).to(torch.int64) for _, c in runs])
    keys, order = torch.sort(keys)
    merged, inverse = torch.unique_consecutive(keys, return_inverse=True)
    return merged, torch.zeros_like(merged).index_add_(0, inverse, counts[order])
