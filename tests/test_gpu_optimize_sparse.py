"""spg_graph_optimize on its block-sparse path (BSR assembly + block-Jacobi PCG): forced onto small graphs with the
SPG_OPT_DENSE_MAX_DIMS hook and compared with the dense Cholesky path, and taken without the hook on a graph beyond the
dense limit."""
import numpy as np
import pytest

import datasets
import kld_harness as K
from sparsifyposegraph_b200 import records as R, synth

pytestmark = pytest.mark.gpu

HOOK = "SPG_OPT_DENSE_MAX_DIMS"


@pytest.fixture(scope="module")
def ctx():
    from sparsifyposegraph_b200 import capi
    c = capi.Context(0)
    yield c
    c.close()


def perturbed_grid(rows, cols, dim, seed=5):
    """Noise-free grid with every estimate but vertex 0's moved: the optimum is chi2 = 0 at the ground truth."""
    from sparsifyposegraph_b200 import capi
    poses, edges, meas, info = synth.make_grid_graph(rows, cols, dim=dim, sigma_t=0.0, sigma_r=0.0)
    g = synth.fill_graph(capi.Graph(dim=dim), poses, edges, meas, info)
    rng = np.random.default_rng(seed)
    for i in range(1, len(poses)):
        p = poses[i].copy()
        p[:2] += rng.normal(0, 0.05, 2)
        g.set_vertex_pose(i, p)
    return g, poses


def oracle_gradient_norm(oracle, g, fixed=(0,)):
    """|J^T Omega e| over the free vertices, from the oracle's errors and Jacobians (pose edges only)."""
    poses = K.poses_of(g)
    acc = {}
    for e in g.edges():
        a, b = int(e["v"][0]), int(e["v"][1])
        err = oracle.edge_error(g.dim, e["meas"], poses[a], poses[b])
        Ji, Jj = oracle.edge_jacobians(g.dim, e["meas"], poses[a], poses[b])
        acc[a] = acc.get(a, 0) + Ji.T @ e["info"] @ err
        acc[b] = acc.get(b, 0) + Jj.T @ e["info"] @ err
    return float(np.sqrt(sum(float(v @ v) for k, v in acc.items() if k not in fixed)))


def poses_array(g):
    return np.array([g.vertex_pose(int(v)) for v in g.vertex_ids()])


@pytest.mark.parametrize("dim", [3, 6])
def test_sparse_path_recovers_noise_free_grid(ctx, monkeypatch, dim):
    g, poses = perturbed_grid(8, 9, dim)
    assert g.chi2(ctx) > 1.0
    monkeypatch.setenv(HOOK, "0")
    st = g.optimize(ctx)
    print(st)
    assert st["solver"] == 1 and st["cg_iterations"] > 0 and st["cg_max_rel_residual"] <= 1e-6
    assert st["chi2_final"] < 1e-12 * max(st["chi2_initial"], 1.0) and st["dimensions"] == dim * (len(poses) - 1)
    for i in range(1, len(poses)):
        assert np.allclose(g.vertex_pose(i), poses[i], atol=1e-7)


def test_hook_is_read_on_every_call(ctx, monkeypatch):
    """The same graph goes dense without the hook, sparse with it, dense again once it is removed."""
    g, _ = perturbed_grid(8, 9, 3)
    monkeypatch.delenv(HOOK, raising=False)
    assert g.optimize(ctx, max_iterations=1)["solver"] == 0
    monkeypatch.setenv(HOOK, "100")
    assert g.optimize(ctx, max_iterations=1)["solver"] == 1
    monkeypatch.setenv(HOOK, "1000")          # the graph has 213 dimensions
    assert g.optimize(ctx, max_iterations=1)["solver"] == 0
    monkeypatch.delenv(HOOK)
    st = g.optimize(ctx, max_iterations=1)
    assert st["solver"] == 0 and st["cg_iterations"] == 0 and st["cg_max_rel_residual"] == 0


@pytest.mark.parametrize("name", ["intel", "sphere"])
def test_sparse_matches_dense_on_datasets(ctx, oracle, monkeypatch, name):
    from sparsifyposegraph_b200 import capi
    dense, sparse = capi.Graph(datasets.path(name)), capi.Graph(datasets.path(name))
    g0 = oracle_gradient_norm(oracle, sparse)
    monkeypatch.delenv(HOOK, raising=False)
    sd = dense.optimize(ctx)
    monkeypatch.setenv(HOOK, "0")
    ss = sparse.optimize(ctx)
    print(name, "dense", sd, "sparse", ss)
    assert sd["solver"] == 0 and ss["solver"] == 1
    assert abs(ss["chi2_final"] - sd["chi2_final"]) <= 1e-6 * sd["chi2_final"]
    assert abs(sparse.chi2(ctx) - ss["chi2_final"]) <= 1e-9 * ss["chi2_final"]
    assert oracle_gradient_norm(oracle, sparse) <= 1e-5 * g0


def sparsified(ctx, which_graph, topology, algorithm):
    from sparsifyposegraph_b200 import capi
    if which_graph == "intel":
        g = capi.Graph(datasets.path("intel"))
    else:  # small SE2 grid with noise
        g = synth.fill_graph(capi.Graph(dim=3), *synth.make_grid_graph(10, 10, dim=3))
    which = capi.decimate_global(g.max_vertex_id, g.max_vertex_id, 2)
    st = g.marginalize(ctx, which, capi.make_opts(topology, R.LIN_GLOBAL), algorithm)
    assert st["n_failed"] == 0
    return g


@pytest.mark.parametrize("which_graph,topology,algorithm,kind", [("intel", R.TOPO_TREE, R.ALG_GLC, 1),
                                                                 ("grid", R.TOPO_CLIQUEY_SUBGRAPH, R.ALG_NFR, 2)],
                         ids=["intel-glc-tree", "grid-nfr-clsubgr"])
def test_sparse_matches_dense_with_glc_and_multi_factors(ctx, monkeypatch, which_graph, topology, algorithm, kind):
    """GLC and MULTI factors couple all their vertices: the clique patterns of the BSR and the GLC / MULTI assembly under
    the BSR policy. Stationarity: a dense re-optimisation from either result finds nothing left to gain."""
    dense, sparse = (sparsified(ctx, which_graph, topology, algorithm) for _ in range(2))
    assert any(e["kind"] == kind for e in sparse.edges())
    monkeypatch.delenv(HOOK, raising=False)
    sd = dense.optimize(ctx)
    monkeypatch.setenv(HOOK, "0")
    ss = sparse.optimize(ctx)
    print(which_graph, "dense", sd, "sparse", ss)
    assert sd["solver"] == 0 and ss["solver"] == 1
    assert abs(ss["chi2_final"] - sd["chi2_final"]) <= 1e-6 * sd["chi2_final"]
    monkeypatch.delenv(HOOK)
    for g in (dense, sparse):
        again = g.optimize(ctx)
        assert again["chi2_initial"] - again["chi2_final"] <= 1e-8 * again["chi2_initial"]


def test_sparse_keeps_pinned_vertices(ctx, monkeypatch):
    """Many vertices pinned, as the delta-chi2 baseline re-optimisation does: their poses come back bit for bit, and the
    free ones land where the dense path puts them."""
    from sparsifyposegraph_b200 import capi
    dense, sparse = capi.Graph(datasets.path("intel")), capi.Graph(datasets.path("intel"))
    ids = sparse.vertex_ids()
    pinned = [int(v) for v in ids[::7]]
    before = {v: sparse.vertex_pose(v).copy() for v in pinned}
    monkeypatch.delenv(HOOK, raising=False)
    sd = dense.optimize(ctx, fixed=pinned)
    monkeypatch.setenv(HOOK, "0")
    ss = sparse.optimize(ctx, fixed=pinned)
    print("dense", sd, "sparse", ss)
    assert ss["solver"] == 1 and ss["dimensions"] == sd["dimensions"] == 3 * (len(ids) - len(pinned))
    for v in pinned:
        assert np.array_equal(sparse.vertex_pose(v), before[v])
    assert abs(ss["chi2_final"] - sd["chi2_final"]) <= 1e-6 * sd["chi2_final"]
    assert np.allclose(poses_array(sparse), poses_array(dense), atol=1e-6)


def test_sparse_path_beyond_the_dense_limit(ctx, monkeypatch):
    """205 x 205 SE2 poses, 126 072 free dimensions: n^2 * 8 bytes is above the 120 GB the dense path takes, so the call
    goes sparse without the hook (before the sparse path it was refused with SPG_ERR_UNSUPPORTED)."""
    monkeypatch.delenv(HOOK, raising=False)
    g, poses = perturbed_grid(205, 205, 3)
    st = g.optimize(ctx)
    print(st)
    assert st["dimensions"] == 3 * (205 * 205 - 1) and st["dimensions"] ** 2 * 8 > 120e9
    assert st["solver"] == 1
    assert st["chi2_final"] < 1e-12 * st["chi2_initial"]
    got = poses_array(g)
    assert np.allclose(got, poses[np.array(g.vertex_ids())], atol=1e-7)
