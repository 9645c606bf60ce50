"""The Python surface on the CPU: cugraph_b200.pylibcugraph wrappers, bench.py's single-GPU and reference arms
driven through the emulation build of the library (tests/emu_py.py).  Catches Python-level mistakes in the wrappers and
the measurement scripts before they reach the GPU box; says nothing about timing or stream ordering."""
import argparse
import importlib.util
import io
import json
import os
import sys

import numpy as np
import pytest

import oracle
from oracle.rmat import rmat_edgelist as rmat_np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def surface():
    torch = pytest.importorskip("torch")  # noqa: F841
    from tests.emu_py import emulated_python_surface
    try:
        cm = emulated_python_surface()
        L = cm.__enter__()
    except Exception as e:  # no host compiler
        pytest.skip(f"emulation build unavailable: {e}")
    yield L
    cm.__exit__(None, None, None)


def _load(path, name):
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_wrappers_match_oracle(surface):
    import torch
    from cugraph_b200 import pylibcugraph as plc
    scale = 9
    V = 1 << scale
    s, d = rmat_np(scale, 16 << scale, seed=3)
    h = plc.ResourceHandle()
    verts_all = torch.arange(V, dtype=torch.int32)
    g = plc.SGGraph(h, plc.GraphProperties(is_multigraph=True), torch.as_tensor(s), torch.as_tensor(d),
                    store_transposed=True, renumber=True, vertices_array=verts_all)
    v, p, conv = plc.pagerank(h, g, None, None, None, None, 0.85, 0.0, 20, False, fail_on_nonconvergence=False)
    ref, _, _ = oracle.pagerank(s, d, V, None, alpha=0.85, epsilon=0.0, max_iterations=20)
    got = np.zeros(V)
    got[v.numpy()] = p.numpy()
    np.testing.assert_allclose(got, ref, rtol=1e-5, atol=1e-12)
    assert conv is False or conv == 0
    s2, d2 = np.concatenate([s, d]), np.concatenate([d, s])
    w = np.random.default_rng(0).random(s.shape[0]).astype(np.float32)
    w2 = np.concatenate([w, w])
    g2 = plc.SGGraph(h, plc.GraphProperties(is_symmetric=True, is_multigraph=True), torch.as_tensor(s2), torch.as_tensor(d2),
                     weight_array=torch.as_tensor(w2), renumber=True, vertices_array=verts_all)
    src = int(s[0])
    dist, pred, bv = plc.bfs(h, g2, torch.tensor([src], dtype=torch.int32), True, 0, True, False)
    rd, _ = oracle.bfs(s2, d2, V, [src])
    gd = np.zeros(V, dtype=np.int32)
    gd[bv.numpy()] = dist.numpy()
    assert np.array_equal(gd, rd)
    sv, sd, sp = plc.sssp(h, g2, src, float("inf"), True, False)
    rs, _ = oracle.sssp(s2, d2, w2, V, src)
    gs = np.zeros(V)
    gs[sv.numpy()] = sd.numpy()
    assert np.array_equal(gs, rs)


def test_bench_single_gpu_arm(surface, monkeypatch, capsys, tmp_path):
    """bench.run_single end to end at a toy scale: one JSON line with every key of the result, including the BFS / SSSP
    numbers as flat keys of `config` and the CPU port + NetworkX baselines; --dump-outputs writes the last timed step's
    PageRank result."""
    monkeypatch.setenv("CUGRAPH_B200_SWEEP_MIN_EDGES", "0")
    monkeypatch.setenv("CUGRAPH_B200_BENCH_BFS_SOURCES", "3")
    monkeypatch.setenv("CUGRAPH_B200_BENCH_SSSP_SOURCES", "2")
    bench = _load(os.path.join(ROOT, "bench.py"), "bench_under_test")
    args = argparse.Namespace(gpus=1, steps=2, warmup=1, impl="b200", scale=10, cpu_sample_scale=10,
                              dump_outputs=str(tmp_path / "dump"))
    bench.run_single(args)
    line = [ln for ln in capsys.readouterr().out.splitlines() if ln.startswith("{")][-1]
    out = json.loads(line)
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "clocks", "e2e", "gpu_launches", "roofline", "cpu_baseline",
                "timing"):
        assert key in out, key
    assert "RMAT-10" in out["metric"]
    assert out["value"] > 0 and out["gpu_launches"] > 0 and out["steps"] == 2
    assert out["e2e"]["value"] is not None and out["e2e"]["value"] > 0, out["e2e"]
    assert out["e2e"]["h2d_bytes_per_step"] == 2 * 4 * (16 << 10)
    assert out["roofline"]["bound"] == "hbm" and out["roofline"]["achieved"] > 0 and 0 < out["roofline"]["frac"]
    assert out["cpu_baseline"]["kind"] == "port" and out["cpu_baseline"]["value"] > 0 and out["cpu_baseline"]["cores"] >= 1
    assert out["cpu_baseline"]["networkx_mteps"] > 0 and out["config"]["networkx_mteps"] == out["cpu_baseline"]["networkx_mteps"]
    cfg = out["config"]
    assert "traversal_error" not in cfg, cfg.get("traversal_error")
    assert cfg["traversal_checks_ok"] is True
    assert cfg["bfs_sources"] == 3 and cfg["sssp_sources"] == 2
    for k in ("bfs_harmonic_mteps", "bfs_mean_mteps", "bfs_ms_per_source", "sssp_harmonic_mteps", "sssp_mean_mteps", "sssp_ms_per_source"):
        assert cfg[k] > 0, k
    verts = np.load(tmp_path / "dump" / "pagerank_vertices.npy")
    scores = np.load(tmp_path / "dump" / "pagerank_scores.npy")
    assert verts.dtype == np.float64 and scores.dtype == np.float32
    assert verts.size == scores.size == cfg["num_vertices"] and (np.diff(verts) > 0).all()
    assert abs(float(scores.astype(np.float64).sum()) - 1.0) < 1e-4


def test_bench_reference_arm(capsys):
    """--impl reference: the CPU port on the benchmark configuration (here a toy scale), same keys, same_config fields"""
    bench = _load(os.path.join(ROOT, "bench.py"), "bench_ref_under_test")
    args = argparse.Namespace(gpus=1, steps=2, warmup=1, impl="reference", scale=10, cpu_sample_scale=10)
    bench.run_reference(args)
    out = json.loads([ln for ln in capsys.readouterr().out.splitlines() if ln.startswith("{")][-1])
    assert out["impl"] == "reference" and out["value"] > 0 and out["dtype"] == "f32"
    assert out["config"]["workload"] == "pagerank_rmat10_ef16_100it" and out["config"]["iterations_timed_per_step"] == 100
    assert out["cpu_baseline"]["kind"] == "port" and out["cpu_baseline"]["value"] == out["value"]
    assert out["e2e"] == {"value": out["value"], "unit": "MTEPS", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_graft_entry_smoke(surface, capsys):
    """__graft_entry__.smoke() itself (scale-12 PageRank + BFS + SSSP against the oracle), kernels emulated"""
    entry = _load(os.path.join(ROOT, "__graft_entry__.py"), "graft_entry_under_test")
    entry.smoke()
    assert "smoke ok" in capsys.readouterr().out


def test_user_level_api(surface):
    """cugraph_b200.api (the shape of the reference's `cugraph` package: Graph.from_pandas_edgelist + functions returning one row
    per vertex) against the oracle: directed PageRank / Katz / HITS, undirected BFS / SSSP / components"""
    import pandas as pd
    from cugraph_b200 import api
    r = np.random.default_rng(5)
    V, E = 400, 3000
    s = (r.integers(0, V, E) * r.random(E) ** 1.5).astype(np.int64)
    d = r.integers(0, V, E).astype(np.int64)
    w = (r.random(E) + 0.25).astype(np.float32)
    pdf = pd.DataFrame({"src": s, "dst": d, "wgt": w})
    ids, inv = np.unique(np.concatenate([s, d]), return_inverse=True)
    si, di = inv[:E], inv[E:]

    def by_id(df, col):
        out = np.zeros(ids.size)
        out[np.searchsorted(ids, df["vertex"].to_numpy())] = df[col].to_numpy()
        return out

    G = api.Graph(directed=True).from_pandas_edgelist(pdf, source="src", destination="dst")
    df = api.pagerank(G, alpha=0.85, max_iter=200, tol=1e-7)
    ref, _, _ = oracle.pagerank(si, di, ids.size, None, alpha=0.85, epsilon=1e-7, max_iterations=200)
    np.testing.assert_allclose(by_id(df, "pagerank"), ref, rtol=2e-5)
    df, conv = api.pagerank(G, max_iter=3, tol=1e-12, fail_on_nonconvergence=False)
    assert conv is False and list(df.columns) == ["vertex", "pagerank"]
    alpha = 0.5 / np.bincount(di).max()
    dk = api.katz_centrality(G, alpha=alpha, beta=1.0, max_iter=300, tol=1e-5)
    rk, _ = oracle.katz(si, di, ids.size, None, alpha=alpha, beta=1.0, epsilon=1e-5, dtype=np.float32)
    np.testing.assert_allclose(by_id(dk, "katz_centrality"), rk, rtol=5e-5)
    dh = api.hits(G, max_iter=500, tol=1e-7)
    rh, ra, _, _ = oracle.hits(si, di, ids.size, epsilon=1e-7)
    np.testing.assert_allclose(by_id(dh, "hubs"), rh, rtol=5e-3, atol=1e-8)
    np.testing.assert_allclose(by_id(dh, "authorities"), ra, rtol=5e-3, atol=1e-8)

    # undirected: symmetrised (and de-duplicated, minimum weight) at creation
    GU = api.Graph(directed=False).from_pandas_edgelist(pdf, source="src", destination="dst", edge_attr="wgt")
    keep = si != di
    a, b = np.minimum(si, di)[keep], np.maximum(si, di)[keep]
    start = int(ids[np.bincount(np.concatenate([a, b])).argmax()])
    db = api.bfs(GU, start=start)
    us, ud = np.concatenate([a, b, si[~keep]]), np.concatenate([b, a, di[~keep]])
    rd, _ = oracle.bfs(us.astype(np.int32), ud.astype(np.int32), ids.size, [int(np.searchsorted(ids, start))])
    rd = np.asarray(rd, dtype=np.int64)
    imax = np.iinfo(np.int32).max
    got = by_id(db, "distance").astype(np.int64)
    assert np.array_equal(got[rd < imax], rd[rd < imax]) and set(db.columns) == {"vertex", "distance", "predecessor"}
    dc = api.weakly_connected_components(GU)
    comp = oracle.wcc(us, ud, ids.size)
    pairs = set(zip(comp.tolist(), by_id(dc, "labels").astype(np.int64).tolist()))
    assert len(pairs) == len(set(comp.tolist()))
    ds = api.sssp(GU, source=start)
    assert set(ds.columns) == {"vertex", "distance", "predecessor"} and float(by_id(ds, "distance")[np.searchsorted(ids, start)]) == 0.0
    with pytest.raises(RuntimeError):
        api.sssp(api.Graph(directed=False).from_pandas_edgelist(pdf, source="src", destination="dst"), source=start)
    # mirror-level extras: eigenvector centrality and the degree functions
    import torch
    from cugraph_b200 import pylibcugraph as plc
    de = api.eigenvector_centrality(G, max_iter=1000, tol=1e-7)
    re_, _ = oracle.eigenvector(si, di, ids.size, None, epsilon=1e-7, max_iterations=1000)
    np.testing.assert_allclose(by_id(de, "eigenvector_centrality"), re_, rtol=5e-3, atol=1e-7)
    h, g = G._plc_graph(True)
    v, din, dout = plc.degrees(h, g, None, False)
    vi = np.searchsorted(ids, v.numpy())
    assert np.array_equal(din.numpy(), np.bincount(di, minlength=ids.size)[vi]) and np.array_equal(dout.numpy(), np.bincount(si, minlength=ids.size)[vi])
    some = torch.as_tensor(ids[:5].copy())
    v2, din2 = plc.in_degrees(h, g, some, False)
    assert v2.numpy().tolist() == ids[:5].tolist() and din2.numpy().tolist() == np.bincount(di, minlength=ids.size)[:5].tolist()
    v3, dout3 = plc.out_degrees(h, g, some, False)
    assert dout3.numpy().tolist() == np.bincount(si, minlength=ids.size)[:5].tolist()
