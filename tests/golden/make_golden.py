#!/usr/bin/env python
"""Generate tests/golden/reference_golden.json from the reference's own test fixtures (run where a checkout of
the reference is available, named by $CUGRAPH_REFERENCE; the tests only ever read the committed JSON).

Sources of truth (all read, none copied as source):
  * python/pylibcugraph/pylibcugraph/tests/test_pagerank.py  `_test_data`  (karate/dolphins/Simple_1/2)
  * python/pylibcugraph/pylibcugraph/tests/test_sssp.py      `_test_data`
  * python/pylibcugraph/pylibcugraph/tests/conftest.py       Simple_1 / Simple_2 / invalid edge lists
  * python/pylibcugraph/pylibcugraph/tests/test_{katz_centrality,eigenvector_centrality,connected_components}.py
                                                             expected values (transcribed below with file:line)
  * datasets/{karate,dolphins,toy_graph,toy_graph_undirected,karate-disjoint-sequential}.csv   edge lists
  * cpp/tests/c_api/{pagerank,bfs,sssp}_test.c               6-/4-vertex golden arrays (transcribed
    below with file:line, they are C array literals)
  * cpp/tests/c_api/{pagerank,bfs,sssp,extract_paths,katz,hits,weakly_connected_components,eigenvector_centrality,
    degrees}_test.c                                          every case's array literals and scalars (parsed)
The pylibcugraph test modules import cupy; a numpy shim stands in for it here.
"""
import importlib.util
import json
import os
import re
import sys
import types

import numpy as np

REF = os.environ["CUGRAPH_REFERENCE"]
OUT = os.path.dirname(os.path.abspath(__file__))


def _load_with_cupy_shim(path, name):
    shim = types.ModuleType("cupy")
    shim.asarray = lambda x, dtype=None: np.asarray(list(x) if isinstance(x, range) else x, dtype=dtype)
    sys.modules["cupy"] = shim
    if "pytest" not in sys.modules:
        import pytest  # noqa: F401
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def _csv(path):
    rows = [l.split() for l in open(path) if l.strip()]
    return ([int(r[0]) for r in rows], [int(r[1]) for r in rows], [float(r[2]) for r in rows])


C_PROGRAMS = ["pagerank", "bfs", "sssp", "extract_paths", "katz", "hits", "weakly_connected_components",
              "eigenvector_centrality", "degrees"]


def _c_value(tok, arrays, scalars):
    tok = tok.strip()
    if tok in arrays:
        return arrays[tok]
    if tok in scalars:
        return scalars[tok]
    if tok in ("TRUE", "FALSE"):
        return tok == "TRUE"
    if tok == "NULL":
        return None
    if tok in ("FLT_MAX", "DBL_MAX"):
        return tok
    tok = tok.rstrip("fd") if re.fullmatch(r"[-+0-9.eE]+[fd]", tok) else tok
    return float(tok) if re.search(r"[.eE]", tok) else int(tok)


def _c_program_cases(path):
    """The cases of one cpp/tests/c_api/*_test.c program, in the order its main() runs them: for each test function the
    generic_* routine it returns into and that routine's arguments by parameter name (the host arrays and scalars the
    test declares).  A test that does not delegate to a generic_* routine is recorded with the arrays and scalars it
    declares."""
    src = re.sub(r"/\*.*?\*/|//[^\n]*", "", open(path).read(), flags=re.S)
    params = {}
    for name, plist in re.findall(r"int\s+(generic_\w+)\s*\(([^)]*)\)\s*\{", src):
        params[name] = [re.findall(r"\w+", p)[-1] for p in plist.split(",")]
    bodies = dict(re.findall(r"int\s+(test_\w+)\s*\([^)]*\)\s*\{(.*?)\n\}", src, flags=re.S))
    cases = []
    for test in re.findall(r"RUN_TEST\((\w+)\)", src):
        body = bodies[test]
        arrays = {n: [_c_value(x, {}, {}) for x in v.replace("\n", " ").split(",") if x.strip()]
                  for n, v in re.findall(r"\w+\s+(\w+)\[\]\s*=\s*\{([^}]*)\};", body)}
        scalars = {n: _c_value(v, {}, {}) for n, v in
                   re.findall(r"(?:size_t|double|float|bool_t|int|vertex_t|weight_t|edge_t)\s+(\w+)\s*=\s*([^;{]+);", body)}
        call = re.search(r"return\s+(generic_\w+)\s*\((.*?)\);", body, flags=re.S)
        case = {"name": test}
        if call:
            args = [_c_value(a, arrays, scalars) for a in call.group(2).split(",")]
            case["generic"] = call.group(1)
            case["args"] = dict(zip(params[call.group(1)], args))
        else:
            case["locals"] = dict(arrays, **scalars)
        cases.append(case)
    return cases


def main():
    tdir = os.path.join(REF, "python/pylibcugraph/pylibcugraph/tests")
    pr = _load_with_cupy_shim(os.path.join(tdir, "test_pagerank.py"), "ref_test_pagerank")
    ss = _load_with_cupy_shim(os.path.join(tdir, "test_sssp.py"), "ref_test_sssp")
    graphs = {
        "karate.csv": _csv(os.path.join(REF, "datasets/karate.csv")),
        "dolphins.csv": _csv(os.path.join(REF, "datasets/dolphins.csv")),
        # conftest.py:38-52
        "Simple_1": ([0, 1, 2], [1, 2, 3], [1.0, 1.0, 1.0]),
        "Simple_2": ([0, 1, 1, 2, 2, 2, 3, 4], [1, 3, 4, 0, 1, 3, 5, 5],
                     [0.1, 2.1, 1.1, 5.1, 3.1, 4.1, 7.2, 3.2]),
    }
    out = {"_source": "generated by tests/golden/make_golden.py from the reference's test fixtures",
           "pylibcugraph": {}}
    for name, (s, d, w) in graphs.items():
        ent = {"src": s, "dst": d, "weights": w,
               "pagerank": {"alpha": pr._alpha, "epsilon": pr._epsilon,
                            "max_iterations": pr._max_iterations, "rel_tol": 1e-4,
                            "vertices": np.asarray(pr._test_data[name][0]).tolist(),
                            "values": [float(x) for x in np.asarray(pr._test_data[name][1], dtype=np.float64)]},
               "sssp": {"source": int(ss._test_data[name]["start_vertex"]), "cutoff": 999999999,
                        "distances": [float(x) for x in np.asarray(ss._test_data[name]["distance"], dtype=np.float64)],
                        "predecessors": np.asarray(ss._test_data[name]["predecessor"]).tolist(),
                        "predecessors_checked": name not in ("karate.csv", "dolphins.csv")}}
        out["pylibcugraph"][name] = ent

    # test_katz_centrality.py:11,89-95 (datasets/toy_graph_undirected.csv) and test_eigenvector_centrality.py:16,85-90
    # (datasets/toy_graph.csv)
    ks, kd, kw = _csv(os.path.join(REF, "datasets/toy_graph_undirected.csv"))
    es, ed, ew = _csv(os.path.join(REF, "datasets/toy_graph.csv"))
    out["pylibcugraph_centralities"] = {
        "katz": {"src": ks, "dst": kd, "weights": kw, "rel_tol": 1e-4,
                 "alpha": 0.01, "beta": 1.0, "epsilon": 1e-6, "max_iterations": 1000,
                 "values": [0.410614, 0.403211, 0.390689, 0.415175, 0.395125, 0.433226]},
        "eigenvector": {"src": es, "dst": ed, "weights": ew, "rel_tol": 1e-4, "epsilon": 1e-6, "max_iterations": 200,
                        "values": [0.236325, 0.292055, 0.458457, 0.60533, 0.190498, 0.495942]},
    }
    # test_connected_components.py:19-149: inputs (dense adjacency or an edge-list file) and the expected weak components
    ks, kd, _ = _csv(os.path.join(REF, "datasets/karate-disjoint-sequential.csv"))
    dolphins = graphs["dolphins.csv"]
    out["pylibcugraph_wcc"] = {
        "graph1": {"adjacency": [[0, 1, 1, 0, 0], [0, 0, 1, 0, 0], [0, 0, 0, 0, 0], [0, 0, 0, 0, 1], [0, 0, 0, 0, 0]],
                   "components": [[0, 1, 2], [3, 4]]},
        "graph2": {"adjacency": [[0, 1, 1, 0, 0], [1, 0, 1, 0, 0], [1, 1, 0, 0, 0], [0, 0, 0, 0, 1], [0, 0, 0, 1, 0]],
                   "components": [[0, 1, 2], [3, 4]]},
        "karate-disjoint-sequential": {"src": ks, "dst": kd, "components": [list(range(34)), [34, 35, 36]]},
        "dolphins": {"src": dolphins[0], "dst": dolphins[1], "components": [list(range(62))]},
    }
    # conftest.py:25-37: edge lists SGGraph must reject with ValueError
    out["pylibcugraph_invalid_graphs"] = {
        "InvalidNumWeights_1": {"src": [0, 1, 2], "dst": [1, 2, 3], "weights": [1.0, 1.0, 1.0, 1.0]},
        "InvalidNumVerts_1": {"src": [1, 2], "dst": [1, 2, 3], "weights": [1.0, 1.0, 1.0]},
    }

    g6 = {"src": [0, 1, 1, 2, 2, 2, 3, 4], "dst": [1, 3, 4, 0, 1, 3, 5, 5],
          "weights": [0.1, 2.1, 1.1, 5.1, 3.1, 4.1, 7.2, 3.2], "num_vertices": 6}
    g4 = {"src": [0, 1, 2], "dst": [1, 2, 3], "weights": [1.0, 1.0, 1.0], "num_vertices": 4}
    out["c_api"] = {
        # cpp/tests/c_api/pagerank_test.c:385-401 (and :404-423 with store_transposed=FALSE)
        "pagerank_6": dict(g6, alpha=0.95, epsilon=1e-4, max_iterations=20, rel_tol=1e-3,
                           values=[0.0915528, 0.168382, 0.0656831, 0.191468, 0.120677, 0.362237]),
        # pagerank_test.c:463-480 (allow_nonconvergence, 2 iterations)
        "pagerank_6_nonconverged": dict(g6, alpha=0.95, epsilon=1e-4, max_iterations=2, rel_tol=1e-3,
                                        values=[0.0776471, 0.167637, 0.0639699, 0.220202, 0.140046, 0.330498]),
        # pagerank_test.c:425-460
        "pagerank_4": dict(g4, alpha=0.85, epsilon=1e-6, max_iterations=500, rel_tol=1e-3,
                           values=[0.11615584790706635, 0.21488840878009796, 0.29881080985069275,
                                   0.37014490365982056]),
        # pagerank_test.c:482-510
        "personalized_pagerank_4": dict(g4, alpha=0.85, epsilon=1e-6, max_iterations=500, rel_tol=1e-3,
                                        personalization_vertices=[0, 1, 2, 3],
                                        personalization_values=[0.1, 0.2, 0.3, 0.4],
                                        values=[0.0559233, 0.159381, 0.303244, 0.481451]),
        # pagerank_test.c:512-540 (1 iteration, allow_nonconvergence)
        "personalized_pagerank_4_nonconverged": dict(g4, alpha=0.85, epsilon=1e-6, max_iterations=1,
                                                     rel_tol=1e-3,
                                                     personalization_vertices=[0, 1, 2, 3],
                                                     personalization_values=[0.1, 0.2, 0.3, 0.4],
                                                     values=[0.03625, 0.285, 0.32125, 0.3575]),
        # cpp/tests/c_api/bfs_test.c:160-209 (seed 0, depth_limit 10)
        "bfs_6": dict(g6, sources=[0], depth_limit=10,
                      distances=[0, 1, 2147483647, 2, 2, 3], predecessors=[-1, 0, -1, 1, 1, 3]),
        # cpp/tests/c_api/sssp_test.c:167-225 (source 0; float and double variants)
        "sssp_6": dict(g6, source=0, cutoff=10.0,
                       distances=[0.0, 0.1, "MAX", 2.2, 1.2, 4.4], predecessors=[-1, 0, -1, 1, 1, 4]),
    }
    # cpp/tests/c_api/<program>_test.c: every case of the C-API test programs, with the arguments of the generic_* routine
    # it runs (inputs, parameters and expected results)
    out["c_api_programs"] = {p: _c_program_cases(os.path.join(REF, "cpp/tests/c_api", f"{p}_test.c")) for p in C_PROGRAMS}
    with open(os.path.join(OUT, "reference_golden.json"), "w") as f:
        json.dump(out, f, indent=1)
    print("wrote", os.path.join(OUT, "reference_golden.json"))


if __name__ == "__main__":
    main()
