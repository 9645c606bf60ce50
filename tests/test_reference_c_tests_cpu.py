"""The reference's own C-API test programs for this path — cpp/tests/c_api/{pagerank,bfs,sssp,extract_paths,katz,hits,
weakly_connected_components,eigenvector_centrality,degrees}_test.c — replayed case by case (tests/c_api_replay.py, from the
cases recorded in tests/golden/reference_golden.json) against the CPU emulation build of the library: every golden vector
and error contract those programs check, through the real C ABI.  tests/test_reference_c_tests_gpu.py replays the same
cases against the CUDA library."""
import os
import sys

import pytest

from tests.c_api_replay import run_program

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

EXPECTED = {
    "pagerank": ["test_pagerank", "test_pagerank_with_transpose", "test_pagerank_4", "test_pagerank_4_with_transpose",
                 "test_pagerank_non_convergence", "test_personalized_pagerank", "test_personalized_pagerank_non_convergence"],
    "bfs": ["test_bfs", "test_bfs_with_transpose", "test_bfs_exceptions"],
    "sssp": ["test_sssp", "test_sssp_with_transpose", "test_sssp_with_transpose_double"],
    "extract_paths": ["test_bfs_with_extract_paths", "test_bfs_with_extract_paths_with_transpose"],
    "katz": ["test_katz"],
    "hits": ["test_hits", "test_hits_with_transpose", "test_hits_with_initial", "test_hits_bigger", "test_hits_bigger_normalized",
             "test_hits_bigger_unnormalized"],
    "weakly_connected_components": ["test_weakly_connected_components", "test_weakly_connected_components_transpose"],
    "eigenvector_centrality": ["test_eigenvector_centrality", "test_eigenvector_centrality_3971"],
    "degrees": ["test_degrees", "test_degrees_symmetric", "test_in_degrees", "test_out_degrees", "test_degrees_subset",
                "test_degrees_symmetric_subset", "test_in_degrees_subset", "test_out_degrees_subset"],
}


def check_program(lib_path, golden, name):
    """every case of the program passes, and the cases are the ones the program runs"""
    results = run_program(lib_path, golden["c_api_programs"][name])
    assert [case for case, _ in results] == EXPECTED[name]
    failed = [f"{case}: {why}" for case, why in results if why is not None]
    assert not failed, "\n".join(failed)


@pytest.fixture(scope="module")
def emu_lib():
    sys.path.insert(0, os.path.join(ROOT, "emu"))
    import build_emu
    try:
        return build_emu.build()
    except Exception as e:
        pytest.skip(f"emulation build unavailable: {e}")


@pytest.mark.parametrize("name", ["pagerank", "bfs", "sssp", "extract_paths", "katz", "hits", "weakly_connected_components", "eigenvector_centrality", "degrees"])
def test_reference_c_test_program(emu_lib, golden, name):
    check_program(emu_lib, golden, name)
