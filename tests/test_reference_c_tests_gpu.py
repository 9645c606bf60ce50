"""The reference's own C-API test programs (cpp/tests/c_api/{pagerank,bfs,sssp,extract_paths,katz,hits,
weakly_connected_components}_test.c) replayed case by case against the CUDA library on the B200 (tests/c_api_replay.py).
(eigenvector_centrality_test.c and degrees_test.c: tests/test_zz_late_additions_gpu.py.)"""
import pytest

from cugraph_b200.build import LIB
from tests.test_reference_c_tests_cpu import check_program

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("name", ["pagerank", "bfs", "sssp", "extract_paths", "katz", "hits", "weakly_connected_components"])
def test_reference_c_test_program_on_gpu(golden, name):
    check_program(LIB, golden, name)
