"""GPU tests of eigenvector centrality and the degree functions, the entry points added last.  The file name sorts last on
purpose: under `pytest -x` the longer-standing GPU tests run first."""
import numpy as np
import pytest

from cugraph_b200.build import LIB
from tests.test_reference_c_tests_cpu import check_program
from tests.test_siblings_gpu import _graph

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("name", ["eigenvector_centrality", "degrees"])
def test_reference_c_test_program_on_gpu(golden, name):
    check_program(LIB, golden, name)


def test_eigenvector_centrality_gpu():
    import oracle
    plc, h, g, ids, s, d, _ = _graph()
    verts, vals = plc.eigenvector_centrality(h, g, 1e-7, 1000, False)
    ref, _ = oracle.eigenvector(s, d, ids.size, None, epsilon=1e-7, max_iterations=1000)
    got = np.zeros(ids.size)
    got[np.searchsorted(ids, verts.cpu().numpy())] = vals.cpu().numpy()
    np.testing.assert_allclose(got, ref, rtol=2e-3, atol=1e-8)


def test_degrees_gpu():
    plc, h, g, ids, s, d, _ = _graph()
    v, din, dout = plc.degrees(h, g, None, False)
    vi = np.searchsorted(ids, v.cpu().numpy())
    assert np.array_equal(din.cpu().numpy(), np.bincount(d, minlength=ids.size)[vi])
    assert np.array_equal(dout.cpu().numpy(), np.bincount(s, minlength=ids.size)[vi])
