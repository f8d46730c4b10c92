"""The library's kernels as a whole (CPU only).

Every kernel family in libhidvae_b200.so is either claimed by the instantiation-coverage test of one test file (that test
fails when a shipped instantiation of the family is no cell's expected kernel) or listed in NO_CELL as deliberately left
without instantiation cells.  A kernel of a new family fails here until its author adds cells for it or lists it.

The kernel-name harness of tests/helpers.py is pinned on profiler (demangled) and cuobjdump (mangled) names of every
family the coverage tests check.
"""
import test_gpu_encoder_fp64
import test_gpu_fp64_reference
import test_gpu_kmeans_uniq_fp64
import test_gpu_tag_heads
from helpers import family, normalise, normalise_symbol, shipped_kernels

CLAIMED = {m.__name__: set(m.FAMILIES) for m in (test_gpu_fp64_reference, test_gpu_kmeans_uniq_fp64, test_gpu_encoder_fp64,
                                                 test_gpu_tag_heads)}
NO_CELL = {
    "rq_pack_codebooks_kernel": "writes the operand images the tensor-core forward kernels read",
    "rq_bwd_fold_replicas_kernel": "folds the backward's gradient replicas into the codebook gradient",
    "enc_pack_weights_kernel": "writes the fused encoder's weight image",
    "gumbel_uniforms_kernel": "draws the Gumbel uniforms; test_gpu_gumbel_graph.py pins the draw bit for bit",
    "dedup_keys_kernel": "collision digit: test_gpu_semid_dedup.py checks every dedup_* kernel runs",
    "dedup_flags_kernel": "collision digit",
    "dedup_runs_kernel": "collision digit",
    "dedup_finish_kernel": "collision digit",
    "peer_allreduce_kernel": "multi-GPU gradient all-reduce, checked against NCCL on two GPUs",
}


def test_every_kernel_family_is_claimed_or_listed():
    shipped = {family(k) for k in shipped_kernels()}
    claims = [f for fams in CLAIMED.values() for f in fams] + list(NO_CELL)
    twice = sorted({f for f in claims if claims.count(f) > 1})
    assert not twice, f"families claimed more than once: {twice}"
    unaccounted = sorted(shipped - set(claims))
    assert not unaccounted, f"kernel families with neither a coverage test nor a NO_CELL entry: {unaccounted}"
    stale = sorted(set(claims) - shipped)
    assert not stale, f"claimed or listed families the library does not ship: {stale}"


def test_kernel_name_normalisation():
    demangled = {
        "void hv::(anonymous namespace)::rq_bwd_smem_kernel<(int)32, (int)8, (bool)1, (bool)1, (int)3>"
        "(hv::(anonymous namespace)::RqBwdArgs)": "rq_bwd_smem_kernel<32,8,true,true,3>",
        "void hv::(anonymous namespace)::rq_bwd_kernel<32, false, true, 0>(hv::RqBwdArgs)": "rq_bwd_kernel<32,false,true,0>",
        "void hv::rq_fwd_tc_v11_kernel<false, true>(hv::RqFwdArgs, hv::V11Params)": "rq_fwd_tc_v11_kernel<false,true>",
        "void hv::(anonymous namespace)::rq_fwd_tc_kernel<64, true, 2>(hv::RqFwdArgs, hv::(anonymous namespace)::TcParams)":
            "rq_fwd_tc_kernel<64,true,2>",
        "void hv::(anonymous namespace)::kmeans_segsum_kernel<(int)64>(float const*, long, unsigned long const*, unsigned int "
        "const*, int, float*, float*)": "kmeans_segsum_kernel<64>",
        "void hv::(anonymous namespace)::uniq_kernel<false>(hv::(anonymous namespace)::UniqArgs, double*)": "uniq_kernel<false>",
        "void hv::(anonymous namespace)::uniq_sorted_kernel<(bool)1>(hv::UniqArgs)": "uniq_sorted_kernel<true>",
        "hv::(anonymous namespace)::uniq_keys_kernel(hv::(anonymous namespace)::UniqArgs, unsigned long*, unsigned int*)":
            "uniq_keys_kernel",
        "void hv::(anonymous namespace)::enc_mlp_kernel<(bool)1, (bool)0>(hv::(anonymous namespace)::EncArgs)":
            "enc_mlp_kernel<true,false>",
        "void hv::(anonymous namespace)::enc_mlp_kernel<true, true>(hv::(anonymous namespace)::EncArgs)": "enc_mlp_kernel<true,true>",
        "void hv::(anonymous namespace)::tag_gemm_kernel<(int)2>(hv::(anonymous namespace)::GemmArgs)": "tag_gemm_kernel<2>",
        "void hv::(anonymous namespace)::gumbel_fwd_kernel<32>(hv::(anonymous namespace)::GumbelArgs)": "gumbel_fwd_kernel<32>",
        "void hv::(anonymous namespace)::gumbel_bwd_kernel<(int)64>(hv::(anonymous namespace)::GumbelArgs)":
            "gumbel_bwd_kernel<64>",
        "hv::(anonymous namespace)::gumbel_uniforms_kernel(hv::(anonymous namespace)::GumbelArgs, float*)":
            "gumbel_uniforms_kernel",
        "void at::native::vectorized_elementwise_kernel<4, float>(int)": None,
        "void cub::DeviceRadixSortOnesweepKernel<int>(int)": None,
    }
    for name, want in demangled.items():
        assert normalise(name) == want, name
    mangled = {
        "_ZN2hv12_GLOBAL__N_118rq_bwd_smem_kernelILi32ELi8ELb1ELb1ELi3EEEvNS0_9RqBwdArgsE": "rq_bwd_smem_kernel<32,8,true,true,3>",
        "_ZN2hv12_GLOBAL__N_113rq_bwd_kernelILi4ELb0ELb0ELi0EEEvNS0_9RqBwdArgsE": "rq_bwd_kernel<4,false,false,0>",
        "_ZN2hv48_GLOBAL__N__9de15e25_15_rq_fwd_tc_v4_cu_81c2742d16rq_fwd_tc_kernelILi64ELb1ELi2EEEvNS_9RqFwdArgsENS0_8TcParamsE":
            "rq_fwd_tc_kernel<64,true,2>",
        "_ZN2hv41_GLOBAL__N__b0c6ceb8_9_kmeans_cu_900813ab20kmeans_segsum_kernelILi64EEEvPKflPKmPKjiPfS8_":
            "kmeans_segsum_kernel<64>",
        "_ZN2hv39_GLOBAL__N__bdcb109d_7_uniq_cu_e4a9325011uniq_kernelILb0EEEvNS0_8UniqArgsEPdPKdfPKfPf": "uniq_kernel<false>",
        "_ZN2hv39_GLOBAL__N__bdcb109d_7_uniq_cu_e4a9325016uniq_keys_kernelENS0_8UniqArgsEPmPj": "uniq_keys_kernel",
        "_ZN2hv43_GLOBAL__N__053ced98_10_enc_mlp_cu_09e2636814enc_mlp_kernelILb0ELb1EEEvNS0_7EncArgsE": "enc_mlp_kernel<false,true>",
        "_ZN2hv45_GLOBAL__N__72aa8d43_12_tag_heads_cu_8688409515tag_gemm_kernelILi2EEEvNS0_8GemmArgsE": "tag_gemm_kernel<2>",
        "_ZN2hv41_GLOBAL__N__337d5d23_9_gumbel_cu_e442257d17gumbel_fwd_kernelILi32EEEvNS0_10GumbelArgsE": "gumbel_fwd_kernel<32>",
        "_ZN2hv41_GLOBAL__N__337d5d23_9_gumbel_cu_e442257d17gumbel_bwd_kernelILi64EEEvNS0_10GumbelArgsE": "gumbel_bwd_kernel<64>",
        "_ZN2hv41_GLOBAL__N__337d5d23_9_gumbel_cu_e442257d22gumbel_uniforms_kernelENS0_10GumbelArgsEPf": "gumbel_uniforms_kernel",
        "_ZN3cub18CUB_200802_SM_100011EmptyKernelIvEEvv": None,
    }
    for name, want in mangled.items():
        assert normalise_symbol(name) == want, name
