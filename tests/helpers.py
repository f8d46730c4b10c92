"""Shared helpers of the parity tests: synthetic inputs (SURVEY.md section 8d), the near-tie ID comparison, the
`lib_mod` / `ops` fixtures, and the kernel-name harness of the instantiation-coverage tests."""
import functools
import os
import re
import shutil
import subprocess
from typing import NamedTuple

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import rq as O

NEAR_TIE_REL = 1e-5  # BASELINE.json north_star: ids bit-exact except where the top-2 distance gap is < 1e-5 relative
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "hid-vae_b200", "libhidvae_b200.so")


# ---------------------------------------------------------------------------------------------------------------------
# fixtures (a test module imports the ones it uses)
# ---------------------------------------------------------------------------------------------------------------------
def _load_lib():
    """hidvae_b200._lib, building the library first when it is missing."""
    if not os.path.isfile(LIB):
        import __graft_entry__
        __graft_entry__.build()
    from hidvae_b200 import _lib
    return _lib


@pytest.fixture(scope="module")
def lib_mod():
    return _load_lib()


@pytest.fixture(scope="module")
def ops():
    _load_lib()
    from hidvae_b200 import ops as _ops
    return _ops


# ---------------------------------------------------------------------------------------------------------------------
# kernel names: every hv:: kernel as family<arg,...> (integers, true / false), or family for a plain kernel, both from
# torch.profiler's demangled names and from the mangled symbols cuobjdump lists
# ---------------------------------------------------------------------------------------------------------------------
_DEMANGLED = re.compile(r"(?:void\s+)?hv::(?:(?:\(anonymous namespace\)|\w+)::)*(\w+)(?:<([^<>]*)>)?\(")
_MANGLED_ARGS = re.compile(r"I((?:L[ib]\d+E)+)E")


def family(kernel):
    return kernel.split("<")[0]


def _demangled_arg(a):
    a = a.strip().replace(" ", "")
    m = re.fullmatch(r"\((bool|int)\)(-?\d+)", a)
    if m:
        return ("true" if m.group(2) != "0" else "false") if m.group(1) == "bool" else m.group(2)
    return a


def normalise(demangled):
    """family<a,b,...> or family of a profiler kernel name; None for a kernel outside hv::."""
    m = _DEMANGLED.match(demangled)
    if m is None:
        return None
    return m.group(1) if m.group(2) is None else f"{m.group(1)}<{','.join(map(_demangled_arg, m.group(2).split(',')))}>"


def normalise_symbol(mangled):
    """The same form from a mangled kernel symbol _ZN2hv<len><name>...[I<args>E]E...; None outside hv::.  The nested
    name's components are length-prefixed, the last one is the kernel's; template arguments must be Li<n>E / Lb<n>E."""
    if not mangled.startswith("_ZN2hv"):
        return None
    pos, name = len("_ZN2hv"), None
    while (m := re.match(r"\d+", mangled[pos:])) is not None:
        start = pos + len(m.group())
        pos = start + int(m.group())
        name = mangled[start:pos]
    if mangled[pos] == "E":
        return name
    m = _MANGLED_ARGS.match(mangled, pos)
    assert m is not None, f"{mangled}: template arguments other than int / bool values"
    args = [v if t == "i" else ("true" if v != "0" else "false") for t, v in re.findall(r"L([ib])(\d+)E", m.group(1))]
    return f"{name}<{','.join(args)}>"


@functools.lru_cache(maxsize=None)
def _library_kernels(tool):
    text = subprocess.run([tool, "-symbols", LIB], check=True, capture_output=True, text=True).stdout
    entries = (line.split()[-1] for line in text.splitlines() if "STO_ENTRY" in line)
    return frozenset(n for n in map(normalise_symbol, entries) if n is not None)


def shipped_kernels():
    """Every hv:: kernel of the built library (cuobjdump -symbols, once per session); cub's kernels are left out.  Skips
    the calling test when the library is not built or cuobjdump is missing."""
    tool = shutil.which("cuobjdump") or os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "cuobjdump")
    if not os.path.isfile(LIB):
        pytest.skip(f"{os.path.relpath(LIB, ROOT)} is not built")
    if not os.path.isfile(tool):
        pytest.skip("cuobjdump not found")
    return _library_kernels(tool)


class Launches(NamedTuple):
    names: set        # normalised hv:: kernels that were launched
    kernels: set      # raw names of every CUDA kernel that was launched (copies and memsets left out)

    @property
    def recorded(self):
        """The profiler recorded at least one CUDA kernel."""
        return bool(self.kernels)


def profiled(fn):
    """Run fn() once under torch.profiler (CPU + CUDA activity); returns (fn's result, Launches)."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        result = fn()
        torch.cuda.synchronize()
    kernels = {ev.name for ev in prof.events() if ev.device_type == torch.autograd.DeviceType.CUDA
               and not ev.name.lower().startswith(("memset", "memcpy"))}
    return result, Launches({n for n in map(normalise, kernels) if n is not None}, kernels)


def assert_launched(launches, expected, families):
    """`expected` (a set of kernels) ran, and no other kernel of `families`.  Returns the skip reason when the profiler saw
    no CUDA kernel at all (the caller skips after its numeric checks)."""
    if not launches.recorded:
        return "torch.profiler recorded no CUDA kernel on this machine: kernel-name assertion not possible (numbers checked)"
    seen = {n for n in launches.names if family(n) in families}
    assert seen == set(expected), f"expected exactly {sorted(expected)} of {families}, launched {sorted(seen)}"
    return None


def unit_rows(n, d, seed):
    g = torch.Generator().manual_seed(seed)
    return F.normalize(torch.randn(n, d, generator=g), dim=-1)


def make_codebooks(n_levels, k, d, seed, kind="uniform"):
    """Effective codebooks [L, K, D]: level 0 row-normalised (modules/h_rqvae.py:295), later levels scaled so
    that every level sees residuals of its own magnitude."""
    g = torch.Generator().manual_seed(seed)
    cbs = []
    for l in range(n_levels):
        w = torch.rand(k, d, generator=g) if kind == "uniform" else torch.randn(k, d, generator=g)
        if l == 0:
            w = F.normalize(w, dim=-1)
        else:
            w = (w - w.mean()) * (0.5 ** l) / (d ** 0.5) * 2.0
        cbs.append(w)
    return torch.stack(cbs)


def oracle_levels(x, codebooks, mode, beta, training):
    return O.rq_forward(x, [codebooks[l] for l in range(codebooks.shape[0])], mode, beta, training)


def check_ids(ids_gpu, x, codebooks, mode, beta, training, allow_near_ties=True):
    """Compare [N, L] ids with the oracle level by level.  At every level the oracle is evaluated on the residual
    that follows the GPU's own earlier choices, so a documented near-tie at one level does not turn into spurious
    mismatches downstream.  A row may differ only where the GPU's code is within NEAR_TIE_REL (relative distance
    gap) of the oracle's best.  Returns a bool mask of rows whose ids match the oracle on every level."""
    ids_gpu = ids_gpu.cpu()
    n, n_levels = ids_gpu.shape
    res = x.clone()
    clean = torch.ones(n, dtype=torch.bool)   # rows not (yet) affected by a near-tie
    for l in range(n_levels):
        cb = codebooks[l]
        table = O.squared_l2_table(res, cb)
        top2 = torch.topk(table, 2 if cb.shape[0] > 1 else 1, dim=1, largest=False)
        ids_ref = table.min(dim=1).indices
        differs = ids_gpu[:, l] != ids_ref
        if differs.any():
            rows = torch.nonzero(differs).view(-1)
            # the GPU's choice must be (near-)tied with the oracle's best
            d_best = top2.values[rows, 0]
            d_gpu = table[rows, ids_gpu[rows, l]]
            rel = (d_gpu - d_best).abs() / d_best.abs().clamp(min=1e-30)
            bad = rel >= NEAR_TIE_REL
            assert allow_near_ties and not bad.any(), (
                f"level {l}: {int(bad.sum())} rows differ from the oracle beyond the near-tie allowance; "
                f"worst relative gap {float(rel.max()):.3e} (rows {rows[bad][:8].tolist()})")
            clean = clean & ~differs
        # follow the GPU's own choice so later levels are compared on the same residuals
        e_gpu = cb[ids_gpu[:, l]]
        if training and mode == O.MODE_ROTATION_TRICK:
            emb_out = O.rotation_trick(res / (res.norm(dim=-1, keepdim=True) + 1e-8),
                                       e_gpu / (e_gpu.norm(dim=-1, keepdim=True) + 1e-8), res)
            if emb_out.dim() == 1:
                emb_out = emb_out.unsqueeze(0)
        else:
            emb_out = e_gpu
        res = res - emb_out
    return clean


def npz(golden_dir, name):
    import os
    return np.load(os.path.join(golden_dir, name))


def t(a):
    return torch.from_numpy(np.asarray(a))
