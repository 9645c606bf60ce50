"""What the reference's own pylibcugraph tests for this path check — python/pylibcugraph/pylibcugraph/tests/{test_pagerank,
test_sssp,test_graph_sg,test_katz_centrality,test_connected_components,test_rmat,test_structure,test_utils,test_version,
test_eigenvector_centrality}.py — restated against this repository's pylibcugraph mirror on the CPU emulation build
(tests/emu_py.py): the same calls, arguments and tolerances, with every expected value read from
tests/golden/reference_golden.json (written from the reference's fixtures by tests/golden/make_golden.py).  Left out, as
before: test_SGGraph_create_from_cudf (needs cudf) and test_scc (strongly connected components are not part of this build;
their argument checks are kept)."""
import itertools
import types

import numpy as np
import pytest


@pytest.fixture(scope="module")
def surface():
    pytest.importorskip("torch")
    from tests.emu_py import emulated_python_surface
    try:
        cm = emulated_python_surface()
        L = cm.__enter__()
    except Exception as e:  # no host compiler
        pytest.skip(f"emulation build unavailable: {e}")
    yield L
    cm.__exit__(None, None, None)


def _t(x, dtype):
    import torch
    return torch.as_tensor(np.asarray(x, dtype=dtype))


def _sg_graph(plc, src, dst, w, transposed):
    """conftest.py create_SGGraph"""
    h = plc.ResourceHandle()
    g = plc.SGGraph(resource_handle=h, graph_properties=plc.GraphProperties(is_symmetric=False, is_multigraph=False),
                    src_or_offset_array=_t(src, np.int32), dst_or_index_array=_t(dst, np.int32),
                    weight_array=_t(w, np.float32), store_transposed=transposed, renumber=False, do_expensive_check=False)
    return g, h


def _check_pagerank(plc, golden):
    for name, d in golden["pylibcugraph"].items():
        p = d["pagerank"]
        g, h = _sg_graph(plc, d["src"], d["dst"], d["weights"], True)
        verts, vals = plc.pagerank(h, g, None, None, None, None, p["alpha"], p["epsilon"], p["max_iterations"], False)
        assert sum(range(len(p["vertices"]))) == sum(p["vertices"])
        assert verts.dtype == _t([], np.int32).dtype and vals.dtype == _t([], np.float32).dtype, name
        for i, (v, x) in enumerate(zip(verts.tolist(), vals.tolist())):
            assert x == pytest.approx(p["values"][v], p["rel_tol"]), f"{name}: pagerank index {i}"


def _check_sssp(plc, golden):
    for name, d in golden["pylibcugraph"].items():
        s = d["sssp"]
        g, h = _sg_graph(plc, d["src"], d["dst"], d["weights"], False)
        verts, dist, pred = plc.sssp(h, g, s["source"], s["cutoff"], True, False)
        assert verts.dtype == _t([], np.int32).dtype and dist.dtype == _t([], np.float32).dtype, name
        assert pred.dtype == _t([], np.int32).dtype, name
        for i, (v, a, p) in enumerate(zip(verts.tolist(), dist.tolist(), pred.tolist())):
            e = s["distances"][v]
            if a <= 3.4e38 or e <= 3.4e38:      # unreachable vertices carry the float maximum
                assert a == pytest.approx(e, 1e-4), f"{name}: distance index {i}"
            if s["predecessors_checked"]:    # equally short paths make karate / dolphins predecessors ambiguous
                assert p == s["predecessors"][v], f"{name}: predecessor index {i}"


def _check_graph_sg(plc, golden):
    gp = plc.GraphProperties()
    assert gp.is_symmetric is False and gp.is_multigraph is False
    for attr in ("is_symmetric", "is_multigraph"):
        setattr(gp, attr, True)
        assert getattr(gp, attr) is True
        setattr(gp, attr, 0)
        assert getattr(gp, attr) is False
        with pytest.raises(TypeError):
            setattr(gp, attr, "foo")
    gp = plc.GraphProperties(is_symmetric=True, is_multigraph=True)
    assert gp.is_symmetric is True and gp.is_multigraph is True
    gp = plc.GraphProperties(is_multigraph=True, is_symmetric=False)
    assert gp.is_symmetric is False and gp.is_multigraph is True
    with pytest.raises(TypeError):
        plc.GraphProperties(is_symmetric="foo", is_multigraph=False)
    with pytest.raises(TypeError):
        plc.GraphProperties(is_multigraph=[])

    rh = plc.ResourceHandle()
    del rh
    for d in golden["pylibcugraph"].values():
        g, _ = _sg_graph(plc, d["src"], d["dst"], d["weights"], False)
        del g
    for name, d in golden["pylibcugraph_invalid_graphs"].items():
        with pytest.raises(ValueError):
            _sg_graph(plc, d["src"], d["dst"], d["weights"], False)


def _check_centralities(plc, golden):
    for algo, a in golden["pylibcugraph_centralities"].items():
        h = plc.ResourceHandle()
        g = plc.SGGraph(resource_handle=h, graph_properties=plc.GraphProperties(is_symmetric=False, is_multigraph=False),
                        src_or_offset_array=_t(a["src"], np.int32), dst_or_index_array=_t(a["dst"], np.int32),
                        weight_array=_t(a["weights"], np.float32), store_transposed=False, renumber=False,
                        do_expensive_check=True)
        if algo == "katz":
            verts, vals = plc.katz_centrality(h, g, None, a["alpha"], a["beta"], a["epsilon"], a["max_iterations"],
                                              do_expensive_check=False)
        else:
            verts, vals = plc.eigenvector_centrality(h, g, a["epsilon"], a["max_iterations"], do_expensive_check=False)
        for i, (v, x) in enumerate(zip(verts.tolist(), vals.tolist())):
            assert x == pytest.approx(a["values"][v], a["rel_tol"]), f"{algo}: vertex index {i}"


def _symmetric_csr(adjacency=None, src=None, dst=None):
    """test_connected_components.py: the input as a scipy CSR matrix (edge lists with unit weights), symmetrised"""
    from scipy.sparse import coo_matrix, csr_matrix
    if adjacency is not None:
        csr = csr_matrix(adjacency)
    else:
        n = len(set(src) | set(dst))
        csr = coo_matrix((np.ones(len(src)), (src, dst)), shape=(n, n), dtype=np.float32).tocsr()
    rows, cols = csr.nonzero()
    csr[cols, rows] = csr[rows, cols]
    return csr


def _check_connected_components(plc, golden):
    import torch
    from scipy.sparse import csr_matrix
    assert callable(plc.weakly_connected_components) and callable(plc.strongly_connected_components)
    for name, d in golden["pylibcugraph_wcc"].items():
        csr = _symmetric_csr(d.get("adjacency"), d.get("src"), d.get("dst"))
        labels = torch.zeros(csr.shape[0], dtype=torch.int32)
        plc.weakly_connected_components(None, None, _t(csr.indptr, np.int32), _t(csr.indices, np.int32),
                                        _t(csr.data, np.float32), labels, False)
        comps = {}
        for v, lab in enumerate(labels.tolist()):
            comps.setdefault(lab, []).append(v)
        assert sorted(comps.values()) == sorted(d["components"]), name

    adjacency = golden["pylibcugraph_wcc"]["graph1"]["adjacency"]
    for api_name in ("weakly_connected_components", "strongly_connected_components"):
        api = getattr(plc, api_name)
        cai, lst = _t(range(8), np.int32), list(range(8))
        for args in ((cai, lst, cai), (lst, cai, cai), (cai, cai, lst)):   # test_non_CAI_input
            with pytest.raises(TypeError):
                api(None, None, args[0], args[1], None, args[2], False)
        csr = _symmetric_csr(adjacency) if api_name == "weakly_connected_components" else csr_matrix(adjacency)
        n = csr.shape[0]
        for off, idx, lab in ((np.int32, np.int32, np.int64), (np.int64, np.int32, np.int32),
                              (np.int32, np.float32, np.int32)):                 # test_bad_dtypes
            with pytest.raises(TypeError):
                api(None, None, _t(csr.indptr, off), _t(csr.indices, idx), None, _t(np.zeros(n), lab), False)

    for api_name, symmetric in (("weakly_connected_components", True), ("strongly_connected_components", False)):
        api = getattr(plc, api_name)                                            # test_invalid_input_{wcc,scc}
        csr = _symmetric_csr(adjacency) if symmetric else csr_matrix(adjacency)
        h = plc.ResourceHandle()
        with pytest.raises(TypeError):
            api(h, None, csr.indptr, csr.indices, None, None, False)
        off, idx = _t(csr.indptr, np.int32), _t(csr.indices, np.int32)
        G = plc.SGGraph(h, plc.GraphProperties(is_symmetric=symmetric, is_multigraph=False), off, idx, None,
                        store_transposed=False, renumber=False, do_expensive_check=True, input_array_format="CSR")
        with pytest.raises(TypeError):
            api(h, G, off, idx, None, None, True)


def _check_rmat(plc):
    """test_rmat.py: every combination of its parameters, and its check_results"""
    for scale, num_edges, clip_and_flip, scramble, weights, types_, ids in itertools.product(
            [2, 4, 8], [4, 16, 32], *[[False, True]] * 5):
        src, dst, wgt, eids, etypes = plc.generate_rmat_edgelist(
            resource_handle=plc.ResourceHandle(), random_state=42, scale=scale, num_edges=num_edges, a=0.57, b=0.19,
            c=0.19, clip_and_flip=clip_and_flip, scramble_vertex_ids=scramble, include_edge_weights=weights,
            minimum_weight=0, maximum_weight=1, dtype=np.float32, include_edge_ids=ids, include_edge_types=types_,
            min_edge_type_value=2, max_edge_type_value=5, multi_gpu=False)
        assert (wgt is not None) if weights else True
        assert (eids is not None) if ids else True
        assert (etypes is not None) if types_ else True
        assert len(src) == len(dst) == num_edges
        assert len(np.union1d(np.asarray(src.tolist()), np.asarray(dst.tolist()))) <= 2 ** scale


def _check_structure(plc):
    """test_structure.py: unequal id widths are widened to 64 bits with a UserWarning"""
    srcs = _t([0, 1, 1, 2, 2, 2, 3, 4, 1, 3, 4, 0, 1, 3, 5, 5], np.int32)
    dsts = _t([1, 3, 4, 0, 1, 3, 5, 5, 0, 1, 1, 2, 2, 2, 3, 4], np.int32)
    weights = _t(np.ones(16), np.float32)
    msg = ("The graph requires 'src_or_offset_array', 'dst_or_index_array' 'vertices_array' and 'edge_id_array' to match. "
           "Those will be widened to 64-bit.")
    props = plc.GraphProperties(is_symmetric=True, is_multigraph=False)
    for vdtype, eids in ((np.int64, None), (np.int32, _t(range(16), np.int64))):
        with pytest.warns(UserWarning, match=msg):
            plc.SGGraph(resource_handle=plc.ResourceHandle(), graph_properties=props, src_or_offset_array=srcs,
                        dst_or_index_array=dsts, weight_array=weights, edge_id_array=eids, store_transposed=False,
                        renumber=True, vertices_array=_t(range(6), vdtype))


def _check_utils_and_version(plc):
    from cugraph_b200.pylibcugraph.utilities.api_tools import experimental_warning_wrapper

    def EXPERIMENTAL__func(a, b):
        return a - b

    class EXPERIMENTAL__klass:
        def __init__(self, a, b):
            self.r = a - b

    with pytest.warns(PendingDeprecationWarning):
        assert 1 == experimental_warning_wrapper(EXPERIMENTAL__func)(3, 2)
    exp_klass = experimental_warning_wrapper(EXPERIMENTAL__klass)
    with pytest.warns(PendingDeprecationWarning):
        k = exp_klass(3, 2)
        assert 1 == k.r and isinstance(k, exp_klass) and k.__class__.__name__ == "klass"
    with pytest.raises(TypeError):
        experimental_warning_wrapper(types.ModuleType("modname"))
    assert isinstance(plc.__git_commit__, str)
    assert isinstance(plc.__version__, str) and len(plc.__version__) > 0


def test_reference_pylibcugraph_tests(surface, golden):
    from cugraph_b200 import pylibcugraph as plc
    _check_pagerank(plc, golden)
    _check_sssp(plc, golden)
    _check_graph_sg(plc, golden)
    _check_centralities(plc, golden)
    _check_connected_components(plc, golden)
    _check_rmat(plc)
    _check_structure(plc)
    _check_utils_and_version(plc)
