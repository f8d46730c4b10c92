"""Semantic-ID collision digit: hv_semid_dedup / ops.semid_dedup / HSemanticIdTokenizer(use_dedup_dim=True).

    digit[r] = #{ r' < r : ids[r', 0:L] == ids[r, 0:L] }      (plus the tuple's count in a prior list)

Oracles:
  (a) the literal reference loop on the CPU: batches of 512, tril(_get_hits(b, b), -1).sum(-1) + _get_hits(b, cache).sum(-1);
  (b) an O(N log N) torch formulation: inverse from torch.unique(dim=0), stable argsort, position within the group.
A CPU test pins (b) to (a); the GPU tests compare the kernel with (b).  Digits are integers: every comparison is torch.equal.
The argument checks of the C ABI and of the Python wrappers need no GPU and run in the CPU suite.
"""
import ctypes
import os

import pytest
import torch

from helpers import ROOT, lib_mod, ops, profiled

gpu = pytest.mark.gpu


# ---------------------------------------------------------------------------------------------------------------------
# oracles
# ---------------------------------------------------------------------------------------------------------------------
def digits_reference_loop(ids, batch=512):
    """(a): the tokenizer's loop over batches of 512 rows, written with its own _get_hits."""
    from modules.tokenizer.h_semids import HSemanticIdTokenizer
    hits = lambda q, k: HSemanticIdTokenizer._get_hits(None, q, k)
    cache, out = ids[:0], []
    for lo in range(0, ids.shape[0], batch):
        b = ids[lo:lo + batch]
        out.append(torch.tril(hits(b, b), -1).sum(-1) + hits(b, cache).sum(-1))
        cache = torch.cat([cache, b])
    return torch.cat(out) if out else ids.new_zeros(0)


def digits_sorted(ids, bits=None):
    """(b): position of every row inside its group of identical tuples, groups from torch.unique.  With `bits`, rows
    holding an id outside [0, 2^bits) get -1 and are left out of every group."""
    n = ids.shape[0]
    out = torch.full((n,), -1, dtype=torch.int64, device=ids.device)
    valid = torch.ones(n, dtype=torch.bool, device=ids.device)
    if bits is not None:
        valid = ((ids >= 0) & (ids < (1 << bits))).all(-1)
    v = ids[valid]
    if v.shape[0]:
        _, inv = torch.unique(v, dim=0, return_inverse=True)
        order = torch.argsort(inv, stable=True)
        counts = torch.bincount(inv)
        starts = counts.cumsum(0) - counts
        pos = torch.empty_like(order)
        pos[order] = torch.arange(v.shape[0], device=ids.device)
        out[valid] = pos - starts[inv]
    return out


def expected_runs(ops, ids, bits):
    """Distinct keys (ascending) and their counts over the rows whose ids are in range."""
    valid = ((ids >= 0) & (ids < (1 << bits))).all(-1)
    keys = ops.dedup_key(ids[valid], bits)
    return torch.unique(keys, return_counts=True)


# ---------------------------------------------------------------------------------------------------------------------
# CPU: oracle (b) against (a), argument validation
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,width,values", [(0, 3, 4), (1, 3, 4), (1537, 3, 3), (4103, 1, 256), (20000, 3, 5), (9000, 4, 2)])
def test_sorted_oracle_matches_reference_loop(n, width, values):
    g = torch.Generator().manual_seed(n + width)
    ids = torch.randint(0, values, (n, width), generator=g)
    assert torch.equal(digits_sorted(ids), digits_reference_loop(ids))


def test_sorted_oracle_matches_reference_loop_on_identical_rows():
    ids = torch.full((2000, 3), 7, dtype=torch.int64)
    assert torch.equal(digits_sorted(ids), torch.arange(2000))
    assert torch.equal(digits_reference_loop(ids), torch.arange(2000))


def _call(lib_mod, rows=8, width=3, bits=8, ids=1, digits=1, run_keys=1, run_counts=1, stats=1, workspace=1, ws_bytes=1 << 30,
          prior_keys=None, prior_counts=None, n_prior=0):
    p = lambda v: None if v is None else ctypes.c_void_p(v)
    return lib_mod.lib.hv_semid_dedup(p(ids), rows, width, width, 1, bits, p(prior_keys), p(prior_counts), n_prior, p(digits),
                                      width + 1, p(run_keys), p(run_counts), p(stats), p(workspace), ws_bytes, None)


def test_argument_validation_before_any_cuda_call(lib_mod):
    L = lib_mod
    assert _call(L, rows=-1) == L.HV_ERR_BAD_SHAPE and "bad shape" in L.last_error()
    assert _call(L, width=0) == L.HV_ERR_BAD_SHAPE
    assert _call(L, bits=0) == L.HV_ERR_BAD_SHAPE
    assert _call(L, n_prior=-1) == L.HV_ERR_BAD_SHAPE
    assert _call(L, width=8, bits=8) == L.HV_ERR_UNSUPPORTED and "63" in L.last_error()      # 64 bits
    assert _call(L, width=1, bits=64) == L.HV_ERR_UNSUPPORTED
    assert _call(L, width=65, bits=1) == L.HV_ERR_UNSUPPORTED
    assert _call(L, rows=1 << 31) == L.HV_ERR_UNSUPPORTED
    assert _call(L, ids=None) == L.HV_ERR_NULL
    assert _call(L, digits=None) == L.HV_ERR_NULL
    assert _call(L, run_keys=None) == L.HV_ERR_NULL
    assert _call(L, run_counts=None) == L.HV_ERR_NULL
    assert _call(L, stats=None) == L.HV_ERR_NULL
    assert _call(L, n_prior=4) == L.HV_ERR_NULL                                               # prior list without pointers
    assert _call(L, workspace=None) == L.HV_ERR_WORKSPACE
    need = L.lib.hv_semid_dedup_workspace_bytes(8)
    assert _call(L, ws_bytes=need - 1) == L.HV_ERR_WORKSPACE and "workspace" in L.last_error()


def test_workspace_sizes(lib_mod):
    ws = lib_mod.lib.hv_semid_dedup_workspace_bytes
    assert ws(0) == 0 and ws(-1) == 0 and ws(1 << 31) == 0
    assert ws(1) > 0 and ws((1 << 31) - 1) > ws(1 << 22) > 16 * (1 << 22)   # at least the sort's keys and the run tables


def test_python_side_raises_value_error_for_wide_keys(ops):
    with pytest.raises(ValueError, match="63-bit"):
        ops.semid_dedup(torch.zeros(4, 8, dtype=torch.int64), 8)          # 64 bits: rejected before the device is needed
    with pytest.raises(ValueError):
        ops.semid_dedup(torch.zeros(4, 3, dtype=torch.int32), 8)
    assert ops.dedup_bits(256) == 8 and ops.dedup_bits(4096) == 12 and ops.dedup_bits(257) == 9 and ops.dedup_bits(1) == 1
    from modules.tokenizer.h_semids import HSemanticIdTokenizer as T
    kw = dict(input_dim=16, output_dim=8, hidden_dims=[12], n_cat_feats=0)
    with pytest.raises(ValueError, match="63-bit"):
        T(codebook_size=1 << 16, n_layers=4, use_dedup_dim=True, **kw)
    assert T(codebook_size=1 << 16, n_layers=3, use_dedup_dim=True, **kw).dedup_stats is None


def test_merge_runs_adds_counts_of_equal_keys(ops):
    a = (torch.tensor([1, 5, 9]), torch.tensor([2, 1, 4]))
    b = (torch.tensor([0, 5]), torch.tensor([7, 3]))
    c = (torch.tensor([], dtype=torch.int64), torch.tensor([], dtype=torch.int64))
    keys, counts = ops.merge_runs([a, b, c])
    assert keys.tolist() == [0, 1, 5, 9] and counts.tolist() == [7, 2, 4, 4]


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the kernel against oracle (b)
# ---------------------------------------------------------------------------------------------------------------------
SHAPES = [(1, 8), (3, 8), (4, 12), (7, 9)]          # (width, bits); (7, 9) is exactly 63 bits
SMALL_N = [0, 1, 511, 512, 513, 4103, 65536]


def make_ids(kind, n, width, bits, seed, device="cuda"):
    g = torch.Generator(device=device).manual_seed(seed)
    if kind == "distinct":   # an odd multiplier is a bijection mod 2^(width*bits): n distinct keys, unpacked to ids
        assert n <= 1 << (width * bits)
        mask = (1 << (width * bits)) - 1
        keys = (torch.randperm(n, generator=g, device=device) * 0x1E3779B97F4A7C15 + 12345) & mask
        shifts = torch.arange(width - 1, -1, -1, device=device) * bits
        return (keys.unsqueeze(1) >> shifts) & ((1 << bits) - 1)
    if kind == "identical":
        return torch.full((n, width), (1 << bits) - 1, dtype=torch.int64, device=device)
    if kind == "few":        # 2..4 values per column: long runs
        per_col = torch.tensor([2 + c % 3 for c in range(width)], device=device)
        return (torch.rand((n, width), generator=g, device=device) * per_col).long()
    raise ValueError(kind)


def check_against_oracle(ops, ids, bits, res, prior_digits=None):
    ref = digits_sorted(ids, bits)
    if prior_digits is not None:
        ref = ref + prior_digits
    assert torch.equal(res.digits, ref), f"{int((res.digits != ref).sum())} of {ids.shape[0]} digits differ"
    keys, counts = expected_runs(ops, ids, bits)
    n_runs = int(res.stats[0])
    assert n_runs == keys.numel()
    assert torch.equal(res.run_keys[:n_runs], keys) and torch.equal(res.run_counts[:n_runs], counts)
    assert int(res.stats[1]) == (int(ref.max()) if ref.numel() else -1)
    assert int(res.stats[2]) == int(((ids < 0) | (ids >= (1 << bits))).any(-1).sum())


@gpu
@pytest.mark.parametrize("width,bits", SHAPES)
@pytest.mark.parametrize("kind", ["distinct", "identical", "few"])
@pytest.mark.parametrize("n", SMALL_N)
def test_digits_match_oracle(ops, n, kind, width, bits):
    if kind == "distinct" and n > 1 << (width * bits):
        pytest.skip("fewer tuples than rows")
    ids = make_ids(kind, n, width, bits, seed=n * 31 + width)
    res = ops.semid_dedup(ids, bits)
    check_against_oracle(ops, ids, bits, res)
    if kind == "identical":
        assert torch.equal(res.digits, torch.arange(n, device="cuda")) and int(res.stats[0]) == min(n, 1)
    if kind == "distinct":
        assert int(res.stats[1]) == (0 if n else -1) and int(res.stats[0]) == n


@gpu
@pytest.mark.parametrize("kind", ["distinct", "identical", "few"])
@pytest.mark.parametrize("n", [1 << 22, (1 << 25) + 3])
def test_digits_match_oracle_large(ops, n, kind):
    ids = make_ids(kind, n, 3, 8 if kind != "distinct" else 9, seed=n % 1000)
    bits = 8 if kind != "distinct" else 9
    res = ops.semid_dedup(ids, bits)
    check_against_oracle(ops, ids, bits, res)
    if kind == "identical":
        assert torch.equal(res.digits, torch.arange(n, device="cuda"))


@pytest.fixture(scope="module")
def bench_table():
    """The [4 Mi, 3] id table the bench's tokenizer assigns to one GPU's shard of synthetic items."""
    import bench
    tok = bench.make_tokenizer(torch.device("cuda"))
    items = bench.synth_items(bench.ITEMS_PER_GPU, seed=0, device=torch.device("cuda"))
    table = tok.precompute_corpus_ids(items).clone()
    del items
    torch.cuda.empty_cache()
    return table


@gpu
def test_bench_table(ops, bench_table):
    res = ops.semid_dedup(bench_table, 8)
    check_against_oracle(ops, bench_table, 8, res)
    assert int(res.stats[0]) < bench_table.shape[0]     # the bench's catalogue does collide


@gpu
@pytest.mark.parametrize("width,bits", [(3, 8), (4, 12)])
def test_strided_inputs(ops, width, bits):
    n = 70001
    ids = make_ids("few", n, width, bits, seed=3)
    ids[::5] = make_ids("distinct", (n + 4) // 5, width, bits, seed=4)
    ref = digits_sorted(ids, bits)
    table = torch.full((n, width + 1), -7, dtype=torch.int64, device="cuda")
    table[:, :width] = ids
    res = ops.semid_dedup(table[:, :width], bits, digits_out=table[:, width])      # [:, :L] view, digit_stride L + 1
    assert res.digits.data_ptr() == table[:, width].data_ptr()
    assert torch.equal(table[:, width], ref) and torch.equal(table[:, :width], ids)
    store = ids.t().contiguous()                                                   # transposed [L, N] store: col_stride = N
    assert torch.equal(ops.semid_dedup(store.t(), bits).digits, ref)


@gpu
@pytest.mark.parametrize("parts", [2, 3, 8])
@pytest.mark.parametrize("kind", ["few", "bench"])
def test_priors_reproduce_the_whole_table(ops, bench_table, parts, kind):
    """Sharding on one GPU: part p with prior = merge_runs(parts < p) gets the whole table's digits on its rows, and the
    merged runs of all parts are the whole table's runs."""
    ids, bits = (make_ids("few", 100003, 4, 12, seed=8), 12) if kind == "few" else (bench_table, 8)
    whole = ops.semid_dedup(ids, bits)
    bounds = [ids.shape[0] * p // parts for p in range(parts + 1)]
    lists = []
    for p in range(parts):
        part = ids[bounds[p]:bounds[p + 1]]
        alone = ops.semid_dedup(part, bits)
        n = int(alone.stats[0])
        prior = ops.merge_runs(lists) if lists else None
        lists.append((alone.run_keys[:n].clone(), alone.run_counts[:n].clone()))
        res = ops.semid_dedup(part, bits, prior=prior)
        assert torch.equal(res.digits, whole.digits[bounds[p]:bounds[p + 1]]), f"part {p} of {parts}"
    keys, counts = ops.merge_runs(lists)
    n = int(whole.stats[0])
    assert torch.equal(keys, whole.run_keys[:n]) and torch.equal(counts, whole.run_counts[:n])
    assert int(counts.max()) - 1 == int(whole.stats[1])


@gpu
@pytest.mark.parametrize("width,bits", [(3, 8), (7, 9)])
def test_out_of_range_ids(ops, width, bits):
    n = 40000
    ids = make_ids("few", n, width, bits, seed=11)
    ids[:, 0] += (1 << bits) - 3                                  # the largest ids: the all-max tuple is among them
    ids[7::13, width - 1] = 1 << bits                             # too large
    ids[5::29, 0] = -1                                            # negative
    ids[3::31] = (1 << bits) - 1                                  # the all-max tuple, whose key invalid rows share
    ids[2] = -(1 << 40)
    res = ops.semid_dedup(ids, bits)
    check_against_oracle(ops, ids, bits, res)
    bad = ((ids < 0) | (ids >= (1 << bits))).any(-1)
    assert bool((res.digits[bad] == -1).all()) and int(res.stats[2]) == int(bad.sum()) > 0
    assert int(res.stats[0]) == torch.unique(ids[~bad], dim=0).shape[0]
    everything_bad = torch.full((1000, width), 1 << bits, dtype=torch.int64, device="cuda")
    res = ops.semid_dedup(everything_bad, bits)
    assert bool((res.digits == -1).all()) and res.stats.tolist() == [0, -1, 1000]


@gpu
def test_deterministic_and_graph_capturable(ops, bench_table):
    ids, bits = bench_table, 8
    a = ops.semid_dedup(ids, bits)
    b = ops.semid_dedup(ids, bits)
    n = int(a.stats[0])
    assert torch.equal(a.digits, b.digits) and torch.equal(a.stats, b.stats)
    assert torch.equal(a.run_keys[:n], b.run_keys[:n]) and torch.equal(a.run_counts[:n], b.run_counts[:n])
    static_ids = ids.clone()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        ops.semid_dedup(static_ids, bits)                         # warm-up outside the capture
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        g = ops.semid_dedup(static_ids, bits)
    g.digits.fill_(-5)
    g.stats.fill_(-5)
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(g.digits, a.digits) and torch.equal(g.stats, a.stats)
    assert torch.equal(g.run_keys[:n], a.run_keys[:n]) and torch.equal(g.run_counts[:n], a.run_counts[:n])
    static_ids.copy_(make_ids("few", ids.shape[0], 3, 8, seed=21))   # new inputs, same graph
    graph.replay()
    check_against_oracle(ops, static_ids, 8, g)


@gpu
def test_profiler_sees_only_dedup_and_cub_kernels(ops):
    ids = make_ids("few", 1 << 20, 3, 8, seed=5)
    ops.semid_dedup(ids, 8)
    _, launches = profiled(lambda: ops.semid_dedup(ids, 8))
    if not launches.recorded:
        pytest.skip("torch.profiler recorded no CUDA kernel on this machine")
    kernels = launches.kernels
    ours = {k for k in kernels if "dedup_" in k}
    assert {k for k in kernels if k not in ours and "cub::" not in k} == set(), sorted(kernels)
    for name in ("dedup_keys_kernel", "dedup_flags_kernel", "dedup_runs_kernel", "dedup_finish_kernel"):
        assert any(name in k for k in ours), (name, sorted(kernels))
    assert any("RadixSort" in k for k in kernels) and any("Scan" in k for k in kernels)


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the tokenizer
# ---------------------------------------------------------------------------------------------------------------------
def _tokenizers(chunk_items):
    from modules.tokenizer.h_semids import HSemanticIdTokenizer
    kw = dict(input_dim=768, output_dim=32, hidden_dims=[512, 256, 128], codebook_size=256, n_layers=3, n_cat_feats=0,
              hrqvae_codebook_normalize=True, chunk_items=chunk_items, encoder_precision="fused")
    torch.manual_seed(0)
    plain = HSemanticIdTokenizer(**kw).cuda().eval()
    dedup = HSemanticIdTokenizer(use_dedup_dim=True, **kw).cuda().eval()
    dedup.load_state_dict(plain.state_dict())
    return plain, dedup


@gpu
@pytest.mark.parametrize("half", [False, True])
def test_tokenizer_table(half):
    import bench
    n, chunk = 90001, 25000                                       # the chunk does not divide the catalogue
    items = bench.synth_items(n, seed=3, device=torch.device("cuda"))
    if half:
        items = items.half()
    plain, dedup = _tokenizers(chunk)
    base = plain.precompute_corpus_ids(items)
    table = dedup.precompute_corpus_ids(items)
    assert table.shape == (n, 4) == (n, dedup.sem_ids_dim)
    assert torch.equal(table[:, :3], base)
    ref = digits_sorted(base)
    assert torch.equal(table[:, 3], ref)
    assert int(ref.max()) > 0                                      # the catalogue does collide
    assert dedup.dedup_stats == (n, torch.unique(base, dim=0).shape[0], int(ref.max()))
    assert plain.dedup_stats is None


@gpu
def test_tokenizer_cache_consumers():
    import bench
    from data.schemas import SeqBatch
    n = 30000
    items = bench.synth_items(n, seed=4, device=torch.device("cuda"))
    _, tok = _tokenizers(8192)
    table = tok.precompute_corpus_ids(items)
    L = 3
    # every cached row hits, with all L + 1 columns; the next free digit of a tuple misses
    assert bool(tok.exists_prefix(table[:1000]).all())
    probe = table[:1000].clone()
    probe[:, L] = tok.dedup_stats[2] + 1
    assert not bool(tok.exists_prefix(probe).any())
    # the cached branch of forward: token types 0..L, rows of L + 1 ids
    b, s = 4, 6
    ids = torch.randint(0, n, (b, s), generator=torch.Generator().manual_seed(1)).cuda()
    batch = SeqBatch(user_ids=torch.arange(b).cuda(), ids=ids, ids_fut=ids[:, :1], x=torch.zeros(b, s, 768).cuda(),
                     x_fut=torch.zeros(b, 768).cuda(), seq_mask=torch.ones(b, s, dtype=torch.bool).cuda())
    out = tok(batch)
    assert out.sem_ids.shape == (b, (L + 1) * s)
    assert torch.equal(out.token_type_ids[0], torch.arange(L + 1, device="cuda").repeat(s))
    assert torch.equal(out.sem_ids.reshape(b, s, L + 1), table[ids])


@gpu
def test_sharded_digits_on_two_gpus():
    """Each rank's shard holds the global digits before gather_shards, and the gathered table equals the single-process
    table (tools/check_dedup_shards.py under torchrun).  Needs two GPUs on the box."""
    import json
    import subprocess
    import sys
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
                          "127.0.0.1", "--master-port", "29551", os.path.join(ROOT, "tools", "check_dedup_shards.py")],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, (out.stdout[-1500:] + out.stderr[-2500:])
    line = [l for l in out.stdout.splitlines() if l.startswith("{")][-1]
    assert json.loads(line)["ok"] is True
