"""Every kernel compiled into libcss_b200.so is launched and checked by some test (no GPU needed to check the list).

The compiled set comes from `cuobjdump -sass` (demangled by c++filt, return type and parameter list dropped, as the profiler's
names are in tests/test_gpu_kernel_matrix.py).  It must equal the kernels that module's cases declare, plus COVERED_ELSEWHERE:
kernels with a single dispatch that an existing test drives and checks exactly.  A new instantiation without a test fails
here on any machine with the CUDA toolkit; an instantiation that nothing can reach should be deleted, not listed.
"""
import ast
import os
import re
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

COVERED_ELSEWHERE = {
    "atl_forward_kernel<19>": "tests/test_gpu_atl.py::test_atl_against_reference_golden",
    "atl_backward_kernel<19>": "tests/test_gpu_atl.py::test_atl_against_reference_golden",
    "atl_forward_kernel<21>": "tests/test_gpu_atl.py::test_atl_against_reference_golden",
    "atl_backward_kernel<21>": "tests/test_gpu_atl.py::test_atl_against_reference_golden",
    "aug_image_front_kernel": "tests/test_gpu_aug_image.py::test_batch_transform_2_vs_pil_chain",
    "aug_image_back_kernel": "tests/test_gpu_aug_image.py::test_batch_transform_2_vs_pil_chain",
    "aug_index_kernel": "tests/test_gpu_aug.py::test_transform_maps_vs_reference",
    "aug_maps_kernel<float>": "tests/test_gpu_aug.py::test_transform_maps_vs_reference",
    "aug_maps_kernel<long>": "tests/test_gpu_aug.py::test_transform_maps_vs_reference",
    "cut_mix_kernel": "tests/test_gpu_aug.py::test_generate_cut_gather_drop_in_vs_reference",
    "ohem_forward_kernel<19>": "tests/test_gpu_ohem.py::test_cityscapes_full_size",
    "ohem_backward_kernel<19>": "tests/test_gpu_ohem.py::test_cityscapes_full_size",
    "ohem_forward_kernel<21>": "tests/test_gpu_ohem.py::test_other_class_counts",
    "ohem_backward_kernel<21>": "tests/test_gpu_ohem.py::test_other_class_counts",
    "ohem_forward_kernel<0>": "tests/test_gpu_ohem.py::test_other_class_counts",
    "ohem_backward_kernel<0>": "tests/test_gpu_ohem.py::test_other_class_counts",
    "ohem_hist_kernel<0>": "tests/test_gpu_ohem.py::test_cityscapes_full_size",
    "ohem_hist_kernel<1>": "tests/test_gpu_ohem.py::test_cityscapes_full_size",
    "ohem_hist_kernel<2>": "tests/test_gpu_ohem.py::test_cityscapes_full_size",
    "ohem_scan_kernel<0>": "tests/test_gpu_ohem.py::test_cityscapes_full_size",
    "ohem_scan_kernel<1>": "tests/test_gpu_ohem.py::test_cityscapes_full_size",
    "ohem_scan_kernel<2>": "tests/test_gpu_ohem.py::test_cityscapes_full_size",
    "ohem_select_sum_kernel": "tests/test_gpu_ohem.py::test_cityscapes_full_size",
    "ohem_finalize_kernel": "tests/test_gpu_ohem.py::test_cityscapes_full_size",
    "grad_scatter_kernel": "tests/test_gpu_grad.py::test_grad_scatter_matches_numpy",
    "rows_verify_kernel<float>": "tests/test_gpu_ddp.py::test_rows_cache_never_serves_stale_rows",
    "sample_kernel": "tests/test_gpu_loss.py::test_contrast_loss_against_oracle_device_draws",
    "stats_allreduce_kernel<2>": "tests/test_gpu_dist.py::test_peer_memory_allreduce_world2",
    "threshold_glue_kernel": "tests/test_gpu_stage12.py::test_threshold_glue_exact_against_oracle",
}


def normalise(name):
    name = re.sub(r"^void\s+", "", name.strip())
    return name.split("(", 1)[0].strip()


def compiled_kernels():
    from css_b200 import build
    lib = build.build()
    sass = subprocess.run(["cuobjdump", "-sass", lib], capture_output=True, text=True, check=True).stdout
    mangled = re.findall(r"Function : (\S+)", sass)
    assert mangled, "cuobjdump listed no kernels"
    demangled = subprocess.run(["c++filt"], input="\n".join(mangled), capture_output=True, text=True, check=True).stdout
    return [normalise(n) for n in demangled.splitlines()]


def test_normalise_matches_the_matrix_module():
    from tests import test_gpu_kernel_matrix as M
    name = "void rep_pass_kernel<7, false, float, false>(float const*, float const*, int, int)"
    assert normalise(name) == M.normalise(name) == "rep_pass_kernel<7, false, float, false>"


def test_every_compiled_kernel_is_tested():
    if shutil.which("cuobjdump") is None or shutil.which("c++filt") is None:
        pytest.skip("cuobjdump / c++filt not available")
    from tests import test_gpu_kernel_matrix as M
    compiled = compiled_kernels()
    assert len(compiled) == len(set(compiled)), "two kernels normalise to the same name"
    declared = M.declared_kernels()
    assert not declared & set(COVERED_ELSEWHERE), f"listed twice: {sorted(declared & set(COVERED_ELSEWHERE))}"
    expected = declared | set(COVERED_ELSEWHERE)
    untested = sorted(set(compiled) - expected)
    assert not untested, f"compiled kernels no test launches: {untested}"
    gone = sorted(expected - set(compiled))
    assert not gone, f"tests declare kernels that are no longer compiled: {gone}"


def test_covered_elsewhere_names_existing_tests():
    for kernel, node in COVERED_ELSEWHERE.items():
        path, func = node.split("::")
        full = os.path.join(ROOT, path)
        assert os.path.isfile(full), f"{kernel}: {path} does not exist"
        tree = ast.parse(open(full).read())
        names = {n.name for n in tree.body if isinstance(n, ast.FunctionDef)}
        assert func in names, f"{kernel}: {node} does not exist"
