"""The reference's C-API test programs for this path (cpp/tests/c_api/{pagerank,bfs,sssp,extract_paths,katz,hits,
weakly_connected_components,eigenvector_centrality,degrees}_test.c) replayed from their recorded cases
(tests/golden/reference_golden.json "c_api_programs", written by tests/golden/make_golden.py).  Each generic_* routine
of those programs is restated here over ctypes: the same C-ABI calls with the same arguments, inputs copied in and results
copied out through the ABI's own device-array functions (so the same code drives the CPU emulation build and the CUDA
library), and the same checks and tolerances (nearlyEqual: |a - b| <= max(|a|, |b|) * 0.001, test_utils.cpp:42-57)."""
import ctypes as C

import numpy as np

INT32, INT64, FLOAT32, FLOAT64 = 2, 3, 8, 9
SUCCESS, INVALID_INPUT = 0, 4
EPSILON = 0.001
P, PP = C.c_void_p, C.POINTER(C.c_void_p)
_NP = {INT32: np.int32, INT64: np.int64, FLOAT32: np.float32, FLOAT64: np.float64}
_TID = {np.dtype(v): k for k, v in _NP.items()}


class CaseFailed(AssertionError):
    pass


class _Props(C.Structure):
    _fields_ = [("is_symmetric", C.c_int), ("is_multigraph", C.c_int)]


_SIGS = {
    "cugraph_create_resource_handle": (P, [P]),
    "cugraph_free_resource_handle": (None, [P]),
    "cugraph_error_message": (C.c_char_p, [P]),
    "cugraph_type_erased_device_array_create": (C.c_int, [P, C.c_size_t, C.c_int, PP, PP]),
    "cugraph_type_erased_device_array_free": (None, [P]),
    "cugraph_type_erased_device_array_view": (P, [P]),
    "cugraph_type_erased_device_array_view_free": (None, [P]),
    "cugraph_type_erased_device_array_view_size": (C.c_size_t, [P]),
    "cugraph_type_erased_device_array_view_type": (C.c_int, [P]),
    "cugraph_type_erased_device_array_view_copy_from_host": (C.c_int, [P, P, P, PP]),
    "cugraph_type_erased_device_array_view_copy_to_host": (C.c_int, [P, P, P, PP]),
    "cugraph_graph_create_with_times_sg": (C.c_int, [P, C.POINTER(_Props)] + [P] * 8 + [C.c_int] * 6 + [PP, PP]),
    "cugraph_graph_free": (None, [P]),
    "cugraph_pagerank": (C.c_int, [P, P, P, P, P, P, C.c_double, C.c_double, C.c_size_t, C.c_int, PP, PP]),
    "cugraph_pagerank_allow_nonconvergence": (C.c_int, [P, P, P, P, P, P, C.c_double, C.c_double, C.c_size_t, C.c_int,
                                                        PP, PP]),
    "cugraph_personalized_pagerank": (C.c_int, [P, P, P, P, P, P, P, P, C.c_double, C.c_double, C.c_size_t, C.c_int,
                                                PP, PP]),
    "cugraph_personalized_pagerank_allow_nonconvergence": (C.c_int, [P, P, P, P, P, P, P, P, C.c_double, C.c_double,
                                                                     C.c_size_t, C.c_int, PP, PP]),
    "cugraph_katz_centrality": (C.c_int, [P, P, P, C.c_double, C.c_double, C.c_double, C.c_size_t, C.c_int, PP, PP]),
    "cugraph_eigenvector_centrality": (C.c_int, [P, P, C.c_double, C.c_size_t, C.c_int, PP, PP]),
    "cugraph_centrality_result_get_vertices": (P, [P]),
    "cugraph_centrality_result_get_values": (P, [P]),
    "cugraph_centrality_result_free": (None, [P]),
    "cugraph_hits": (C.c_int, [P, P, C.c_double, C.c_size_t, P, P, C.c_int, C.c_int, PP, PP]),
    "cugraph_hits_result_get_vertices": (P, [P]),
    "cugraph_hits_result_get_hubs": (P, [P]),
    "cugraph_hits_result_get_authorities": (P, [P]),
    "cugraph_hits_result_free": (None, [P]),
    "cugraph_bfs": (C.c_int, [P, P, P, C.c_int, C.c_size_t, C.c_int, C.c_int, PP, PP]),
    "cugraph_sssp": (C.c_int, [P, P, C.c_size_t, C.c_double, C.c_int, C.c_int, PP, PP]),
    "cugraph_paths_result_get_vertices": (P, [P]),
    "cugraph_paths_result_get_distances": (P, [P]),
    "cugraph_paths_result_get_predecessors": (P, [P]),
    "cugraph_paths_result_free": (None, [P]),
    "cugraph_extract_paths": (C.c_int, [P, P, P, P, P, PP, PP]),
    "cugraph_extract_paths_result_get_max_path_length": (C.c_size_t, [P]),
    "cugraph_extract_paths_result_get_paths": (P, [P]),
    "cugraph_extract_paths_result_free": (None, [P]),
    "cugraph_weakly_connected_components": (C.c_int, [P, P, C.c_int, PP, PP]),
    "cugraph_labeling_result_get_vertices": (P, [P]),
    "cugraph_labeling_result_get_labels": (P, [P]),
    "cugraph_labeling_result_free": (None, [P]),
    "cugraph_degrees": (C.c_int, [P, P, P, C.c_int, PP, PP]),
    "cugraph_in_degrees": (C.c_int, [P, P, P, C.c_int, PP, PP]),
    "cugraph_out_degrees": (C.c_int, [P, P, P, C.c_int, PP, PP]),
    "cugraph_degrees_result_get_vertices": (P, [P]),
    "cugraph_degrees_result_get_in_degrees": (P, [P]),
    "cugraph_degrees_result_get_out_degrees": (P, [P]),
    "cugraph_degrees_result_free": (None, [P]),
}


def _check(ok, what):
    if not ok:
        raise CaseFailed(what)


def _nearly_equal(a, b, dtype=np.float32):
    a, b = dtype(a), dtype(b)
    return bool(abs(a - b) <= max(abs(a), abs(b)) * dtype(EPSILON))


def _host(values, dtype):
    """a C array literal of the recorded case as a host array (FLT_MAX / DBL_MAX spelled by name)"""
    big = {"FLT_MAX": np.finfo(np.float32).max, "DBL_MAX": np.finfo(np.float64).max}
    return np.ascontiguousarray([big.get(v, v) if isinstance(v, str) else v for v in values], dtype=dtype)


class Session:
    """One resource handle on one build of the library; the device arrays it creates live until close()."""

    def __init__(self, lib_path):
        L = C.CDLL(lib_path)
        for name, (res, args) in _SIGS.items():
            fn = getattr(L, name)
            fn.restype, fn.argtypes = res, args
        self.L = L
        self.h = L.cugraph_create_resource_handle(None)
        assert self.h, "resource handle creation failed"
        self._arrays = []

    def close(self):
        for a in self._arrays:
            self.L.cugraph_type_erased_device_array_free(a)
        self._arrays = []
        self.L.cugraph_free_resource_handle(self.h)

    def ok(self, code, err, what, expect=SUCCESS):
        if code != expect:
            msg = self.L.cugraph_error_message(err) if err.value else b""
            raise CaseFailed(f"{what} returned {code}, expected {expect}: {msg.decode(errors='replace')}")

    def device(self, host):
        """cugraph_type_erased_device_array_create + _view_copy_from_host of a host array: the view"""
        arr, err = P(), P()
        self.ok(self.L.cugraph_type_erased_device_array_create(self.h, host.size, _TID[host.dtype], C.byref(arr), C.byref(err)),
                err, "cugraph_type_erased_device_array_create")
        self._arrays.append(arr)
        view = self.L.cugraph_type_erased_device_array_view(arr)
        self.ok(self.L.cugraph_type_erased_device_array_view_copy_from_host(self.h, view, host.ctypes.data, C.byref(err)),
                err, "copy_from_host")
        return view

    def host(self, view):
        """cugraph_type_erased_device_array_view_copy_to_host of a result view; None for a NULL view"""
        if not view:
            return None
        n = self.L.cugraph_type_erased_device_array_view_size(view)
        out = np.empty(n, dtype=_NP[self.L.cugraph_type_erased_device_array_view_type(view)])
        err = P()
        if n:
            self.ok(self.L.cugraph_type_erased_device_array_view_copy_to_host(self.h, out.ctypes.data, view, C.byref(err)),
                    err, "copy_to_host")
        self.L.cugraph_type_erased_device_array_view_free(view)
        return out

    def graph(self, src, dst, wgt, store_transposed, renumber=False, is_symmetric=False, wdtype=np.float32):
        """test_utils.cpp create_test_graph / create_test_graph_double: is_multigraph FALSE, no drop / symmetrize, no
        expensive check"""
        views = [self.device(_host(src, np.int32)), self.device(_host(dst, np.int32)), self.device(_host(wgt, wdtype))]
        g, err = P(), P()
        code = self.L.cugraph_graph_create_with_times_sg(
            self.h, C.byref(_Props(int(is_symmetric), 0)), None, *views, None, None, None, None,
            int(store_transposed), int(renumber), 0, 0, 0, 0, C.byref(g), C.byref(err))
        self.ok(code, err, "create_test_graph")
        return g


def _centrality_check(s, res, expected, num_vertices):
    verts = s.host(s.L.cugraph_centrality_result_get_vertices(res))
    vals = s.host(s.L.cugraph_centrality_result_get_values(res))
    s.L.cugraph_centrality_result_free(res)
    _check(verts.size >= num_vertices, f"{verts.size} result rows for {num_vertices} vertices")
    for i in range(num_vertices):
        _check(_nearly_equal(expected[verts[i]], vals[i]), f"vertex {verts[i]}: {vals[i]} != {expected[verts[i]]}")


def _pagerank(s, a, allow_nonconvergence=False, personalized=False):
    g = s.graph(a["h_src"], a["h_dst"], a["h_wgt"], a["store_transposed"])
    res, err = P(), P()
    fn = "cugraph_personalized_pagerank" if personalized else "cugraph_pagerank"
    fn += "_allow_nonconvergence" if allow_nonconvergence else ""
    pers = []
    if personalized:
        n = a["num_personalization_vertices"]
        pers = [s.device(_host(a["h_personalization_vertices"][:n], np.int32)),
                s.device(_host(a["h_personalization_values"][:n], np.float32))]
    code = getattr(s.L, fn)(s.h, g, None, None, None, None, *pers, a["alpha"], a["epsilon"], a["max_iterations"], 0,
                            C.byref(res), C.byref(err))
    s.ok(code, err, fn)
    _centrality_check(s, res, _host(a["h_result"], np.float32), a["num_vertices"])
    s.L.cugraph_graph_free(g)


def _katz(s, a):
    g = s.graph(a["h_src"], a["h_dst"], a["h_wgt"], a["store_transposed"])
    res, err = P(), P()
    s.ok(s.L.cugraph_katz_centrality(s.h, g, None, a["alpha"], a["beta"], a["epsilon"], a["max_iterations"], 0,
                                     C.byref(res), C.byref(err)), err, "cugraph_katz_centrality")
    _centrality_check(s, res, _host(a["h_result"], np.float32), a["num_vertices"])
    s.L.cugraph_graph_free(g)


def _eigenvector(s, a):
    g = s.graph(a["h_src"], a["h_dst"], a["h_wgt"], a["store_transposed"])
    res, err = P(), P()
    s.ok(s.L.cugraph_eigenvector_centrality(s.h, g, a["epsilon"], a["max_iterations"], 0, C.byref(res), C.byref(err)),
         err, "cugraph_eigenvector_centrality")
    _centrality_check(s, res, _host(a["h_result"], np.float32), a["num_vertices"])
    s.L.cugraph_graph_free(g)


def _hits(s, a):
    g = s.graph(a["h_src"], a["h_dst"], a["h_wgt"], a["store_transposed"], a["renumber"])
    init = [None, None]
    if a["h_initial_vertices"] is not None:
        n = a["num_initial_vertices"]
        init = [s.device(_host(a["h_initial_vertices"][:n], np.int32)), s.device(_host(a["h_initial_hubs"][:n], np.float32))]
    res, err = P(), P()
    s.ok(s.L.cugraph_hits(s.h, g, a["epsilon"], a["max_iterations"], *init, int(a["normalize"]), 0, C.byref(res),
                          C.byref(err)), err, "cugraph_hits")
    verts = s.host(s.L.cugraph_hits_result_get_vertices(res))
    hubs = s.host(s.L.cugraph_hits_result_get_hubs(res))
    auth = s.host(s.L.cugraph_hits_result_get_authorities(res))
    s.L.cugraph_hits_result_free(res)
    exp_h, exp_a = _host(a["h_result_hubs"], np.float32), _host(a["h_result_authorities"], np.float32)
    _check(verts.size >= a["num_vertices"], f"{verts.size} result rows for {a['num_vertices']} vertices")
    for i in range(a["num_vertices"]):
        _check(_nearly_equal(exp_h[verts[i]], hubs[i]), f"hub of vertex {verts[i]}: {hubs[i]} != {exp_h[verts[i]]}")
        _check(_nearly_equal(exp_a[verts[i]], auth[i]), f"authority of vertex {verts[i]}: {auth[i]} != {exp_a[verts[i]]}")
    s.L.cugraph_graph_free(g)


def _bfs_paths(s, g, seeds_view, depth_limit):
    res, err = P(), P()
    s.ok(s.L.cugraph_bfs(s.h, g, seeds_view, 0, depth_limit, 1, 0, C.byref(res), C.byref(err)), err, "cugraph_bfs")
    return res


def _bfs(s, a):
    g = s.graph(a["h_src"], a["h_dst"], a["h_wgt"], a["store_transposed"])
    res = _bfs_paths(s, g, s.device(_host(a["h_seeds"][:a["num_seeds"]], np.int32)), a["depth_limit"])
    verts = s.host(s.L.cugraph_paths_result_get_vertices(res))
    dist = s.host(s.L.cugraph_paths_result_get_distances(res))
    pred = s.host(s.L.cugraph_paths_result_get_predecessors(res))
    s.L.cugraph_paths_result_free(res)
    _check(verts.size >= a["num_vertices"], f"{verts.size} result rows for {a['num_vertices']} vertices")
    for i in range(a["num_vertices"]):
        v = verts[i]
        _check(a["expected_distances"][v] == dist[i], f"distance of vertex {v}: {dist[i]}")
        _check(a["expected_predecessors"][v] == pred[i], f"predecessor of vertex {v}: {pred[i]}")
    s.L.cugraph_graph_free(g)


def _bfs_exceptions(s, loc):
    """bfs_test.c test_bfs_exceptions: INT64 seeds on an INT32 graph are rejected with CUGRAPH_INVALID_INPUT"""
    g = s.graph(loc["src"], loc["dst"], loc["wgt"], False)
    seeds = s.device(_host(loc["seeds"][:loc["num_seeds"]], np.int64))
    res, err = P(), P()
    s.ok(s.L.cugraph_bfs(s.h, g, seeds, 0, loc["depth_limit"], 1, 0, C.byref(res), C.byref(err)), err, "cugraph_bfs",
         expect=INVALID_INPUT)
    s.L.cugraph_graph_free(g)


def _sssp(s, a, dtype=np.float32):
    g = s.graph(a["h_src"], a["h_dst"], a["h_wgt"], a["store_transposed"], wdtype=dtype)
    res, err = P(), P()
    s.ok(s.L.cugraph_sssp(s.h, g, a["source"], a["cutoff"], 1, 0, C.byref(res), C.byref(err)), err, "cugraph_sssp")
    verts = s.host(s.L.cugraph_paths_result_get_vertices(res))
    dist = s.host(s.L.cugraph_paths_result_get_distances(res))
    pred = s.host(s.L.cugraph_paths_result_get_predecessors(res))
    s.L.cugraph_paths_result_free(res)
    exp_d = _host(a["expected_distances"], dtype)
    _check(verts.size >= a["num_vertices"], f"{verts.size} result rows for {a['num_vertices']} vertices")
    for i in range(a["num_vertices"]):
        v = verts[i]
        _check(_nearly_equal(exp_d[v], dist[i], dtype), f"distance of vertex {v}: {dist[i]} != {exp_d[v]}")
        _check(a["expected_predecessors"][v] == pred[i], f"predecessor of vertex {v}: {pred[i]}")
    s.L.cugraph_graph_free(g)


def _extract_paths(s, a):
    g = s.graph(a["h_src"], a["h_dst"], a["h_wgt"], a["store_transposed"])
    seeds = s.device(_host(a["h_seeds"][:a["num_seeds"]], np.int32))
    dests = s.device(_host(a["h_destinations"][:a["num_destinations"]], np.int32))
    paths = _bfs_paths(s, g, seeds, a["depth_limit"])
    res, err = P(), P()
    s.ok(s.L.cugraph_extract_paths(s.h, g, seeds, paths, dests, C.byref(res), C.byref(err)), err, "cugraph_extract_paths")
    length = s.L.cugraph_extract_paths_result_get_max_path_length(res)
    _check(length == a["expected_max_path_length"], f"max path length {length}")
    got = s.host(s.L.cugraph_extract_paths_result_get_paths(res))
    for i in range(got.size):
        _check(a["expected_paths"][i] == got[i], f"paths[{i}] = {got[i]}")
    s.L.cugraph_extract_paths_result_free(res)
    s.L.cugraph_paths_result_free(paths)
    s.L.cugraph_graph_free(g)


def _wcc(s, a):
    g = s.graph(a["h_src"], a["h_dst"], a["h_wgt"], a["store_transposed"], is_symmetric=True)
    res, err = P(), P()
    s.ok(s.L.cugraph_weakly_connected_components(s.h, g, 0, C.byref(res), C.byref(err)), err,
         "cugraph_weakly_connected_components")
    verts = s.host(s.L.cugraph_labeling_result_get_vertices(res))
    labels = s.host(s.L.cugraph_labeling_result_get_labels(res))
    s.L.cugraph_labeling_result_free(res)
    n, expected = a["num_vertices"], a["h_result"]
    _check(verts.size >= n, f"{verts.size} result rows for {n} vertices")
    label_of = {}                                   # expected component -> the label of its first vertex in the result
    for i in range(n):
        label_of.setdefault(expected[verts[i]], labels[i])
    for i in range(n):
        _check(labels[i] == label_of[expected[verts[i]]], f"vertex {verts[i]} labelled {labels[i]}")
    s.L.cugraph_graph_free(g)


def _degrees(s, a):
    g = s.graph(a["h_src"], a["h_dst"], a["h_wgt"], a["store_transposed"], is_symmetric=a["is_symmetric"])
    subset = None
    if a["h_vertices"] is not None:
        subset = s.device(_host(a["h_vertices"][:a["num_vertices_to_compute"]], np.int32))
    fn = ("cugraph_degrees" if a["in_degrees"] and a["out_degrees"] else
          "cugraph_in_degrees" if a["in_degrees"] else "cugraph_out_degrees")
    res, err = P(), P()
    s.ok(getattr(s.L, fn)(s.h, g, subset, 0, C.byref(res), C.byref(err)), err, fn)
    verts = s.host(s.L.cugraph_degrees_result_get_vertices(res))
    ins = s.host(s.L.cugraph_degrees_result_get_in_degrees(res))
    outs = s.host(s.L.cugraph_degrees_result_get_out_degrees(res))
    s.L.cugraph_degrees_result_free(res)
    want = a["num_vertices_to_compute"] if subset is not None else a["num_vertices"]
    _check(verts.size == want, f"{verts.size} result rows, expected {want}")
    for i in range(verts.size):
        v = verts[i]
        if a["h_in_degrees"] is not None:
            _check(ins is not None and ins[i] == a["h_in_degrees"][v], f"in degree of vertex {v}")
        if a["h_out_degrees"] is not None:
            _check(outs is not None and outs[i] == a["h_out_degrees"][v], f"out degree of vertex {v}")
    s.L.cugraph_graph_free(g)


GENERICS = {
    "generic_pagerank_test": _pagerank,
    "generic_pagerank_nonconverging_test": lambda s, a: _pagerank(s, a, allow_nonconvergence=True),
    "generic_personalized_pagerank_test": lambda s, a: _pagerank(s, a, personalized=True),
    "generic_personalized_pagerank_nonconverging_test": lambda s, a: _pagerank(s, a, True, True),
    "generic_bfs_test": _bfs,
    "generic_sssp_test": _sssp,
    "generic_sssp_test_double": lambda s, a: _sssp(s, a, np.float64),
    "generic_bfs_test_with_extract_paths": _extract_paths,
    "generic_katz_test": _katz,
    "generic_hits_test": _hits,
    "generic_wcc_test": _wcc,
    "generic_eigenvector_centrality_test": _eigenvector,
    "generic_degrees_test": _degrees,
}
STANDALONE = {"test_bfs_exceptions": _bfs_exceptions}


def run_program(lib_path, cases):
    """Every recorded case of one program against the library at lib_path, in order: [(test name, None or failure)]"""
    s = Session(lib_path)
    out = []
    try:
        for case in cases:
            try:
                if "generic" in case:
                    GENERICS[case["generic"]](s, case["args"])
                else:
                    STANDALONE[case["name"]](s, case["locals"])
                out.append((case["name"], None))
            except CaseFailed as e:
                out.append((case["name"], str(e)))
    finally:
        s.close()
    return out
