"""Every __global__ kernel of the library has a test.

The kernels the fit dispatch tables select (dmf_inst_body.cuh) are the fit universe of tests/plan_probe.cu: test_kernel_matrix.py
runs every entry of it against the oracle.  Every other kernel must be listed in KERNEL_TESTS with the tests that call it; the
test checks that each listed test function exists.  A new kernel without a test fails here."""
import ast
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "demethify_b200", "csrc")

KERNEL_TESTS = {
    "wls_moments_kernel": ["tests/test_gpu_aux_kernels.py::test_wls_moments_bitwise_vs_exact",
                           "tests/test_kernel_matrix.py::test_wls_each_storage_pair"],
    "wls_nnls_kernel": ["tests/test_gpu_aux_kernels.py::test_wls_nnls_vs_exact",
                        "tests/test_gpu_aux_kernels.py::test_wls_nnls_iteration_limit_is_an_error"],
    "resid_gram_kernel": ["tests/test_gpu_aux_kernels.py::test_resid_gram_bitwise_vs_exact",
                          "tests/test_gpu_aux_kernels.py::test_resid_gram_floor_componentwise"],
    "resid_project_kernel": ["tests/test_gpu_aux_kernels.py::test_resid_project_bitwise_vs_exact"],
    "nndsvd_apply_kernel": ["tests/test_gpu_aux_kernels.py::test_nndsvd_apply_and_split_vs_rule"],
    "nndsvd_split_kernel": ["tests/test_gpu_aux_kernels.py::test_nndsvd_apply_and_split_vs_rule"],
    "percentile_kernel": ["tests/test_gpu_aux_kernels.py::test_percentile_bitwise_vs_numpy",
                          "tests/test_gpu_aux_kernels.py::test_percentile_special_values"],
    "labels_kernel": ["tests/test_gpu_aux_kernels.py::test_consensus_bitwise_vs_numpy"],
    "consensus_kernel": ["tests/test_gpu_aux_kernels.py::test_consensus_bitwise_vs_numpy"],
    "legacy_streams_kernel": ["tests/test_gpu_rng.py::test_uniform_and_state_match_numpy", "tests/test_gpu_rng.py::test_randint_matches_numpy"],
    "pack_u16_kernel": ["tests/test_kernel_matrix.py::test_pack_weights_boundaries"],
    "gather_rows_kernel": ["tests/test_kernel_matrix.py::test_gather_rows_bit_exact"],
    "set_step_state_kernel": ["tests/test_gpu_steps.py::test_set_step_state_checks_and_writes_only_its_scalars"],
    "finalize_cost_kernel": ["tests/test_gpu_sharded.py::test_sharded_mode_single_rank_vs_oracle"],
    "u_commit_kernel": ["tests/test_gpu_sharded_stream.py::test_sharded_stream_single_rank"],
    "alpha_commit_kernel": ["tests/test_gpu_sharded_stream.py::test_sharded_stream_single_rank"],
    # multi-GPU only: the ranks spin-wait on each other's peer buffers, so one GPU cannot run it
    "peer_allreduce_kernel": ["tools/sharded_check.py"],
}


def _strip_comments(src):
    return re.sub(r"//[^\n]*|/\*.*?\*/", "", src, flags=re.S)


def global_kernels():
    """Names of every __global__ function in the library's sources."""
    names = set()
    for f in sorted(os.listdir(CSRC)):
        if f.endswith((".cu", ".cuh", ".h")):
            src = _strip_comments(open(os.path.join(CSRC, f)).read())
            for m in re.finditer(r"__global__\s+void\s+(?:__launch_bounds__\s*\((?:[^()]|\([^()]*\))*\)\s*)?(\w+)\s*\(", src):
                names.add(m.group(1))
    return names


def fit_universe_kernels():
    """Kernels the fit dispatch tables of dmf_inst_body.cuh can return: the fit universe of plan_probe."""
    src = _strip_comments(open(os.path.join(CSRC, "dmf_inst_body.cuh")).read())
    return set(re.findall(r"\b(\w+_kernel)\s*<", src))


def test_kernel_scan_finds_the_known_kernels():
    ks = global_kernels()
    assert {"wls_moments_kernel", "percentile_kernel", "resid_gram_kernel", "fused_outer_kernel", "labels_kernel"} <= ks
    assert {"cost_kernel", "rowgram_kernel", "fused_outer_kernel", "wls_moments_kernel"} <= fit_universe_kernels() <= ks


def test_every_kernel_has_a_test():
    ks = global_kernels()
    missing = sorted(ks - fit_universe_kernels() - set(KERNEL_TESTS))
    assert not missing, f"kernels with no test: {missing} (add them to KERNEL_TESTS)"
    assert set(KERNEL_TESTS) <= ks, f"KERNEL_TESTS names kernels that no longer exist: {sorted(set(KERNEL_TESTS) - ks)}"


def test_listed_tests_exist():
    for kernel, ids in KERNEL_TESTS.items():
        assert ids, kernel
        for node in ids:
            path, _, name = node.partition("::")
            full = os.path.join(ROOT, path)
            assert os.path.exists(full), (kernel, node)
            if not name:
                assert kernel == "peer_allreduce_kernel", f"{kernel}: only the multi-GPU kernel may point at a script"
                continue
            tree = ast.parse(open(full).read())
            funcs = {n.name for n in ast.walk(tree) if isinstance(n, (ast.FunctionDef, ast.AsyncFunctionDef))}
            assert name in funcs, f"{kernel}: {node} does not exist"
