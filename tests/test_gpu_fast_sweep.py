"""fast_kernel's CTA-wide variants (G = 0: one blanket per CTA of up to 4 or 8 warps, SE3 blankets of 9 ... 23 vertices,
SE2 of 10 ... 23) against blanket_kernel alone (SPG_NO_FAST=1, same binary), and the blankets such a CTA refuses in
its block sweeps: they must leave through the device-side retry list and come back exactly as blanket_kernel alone
reports them."""
import numpy as np
import pytest

from sparsifyposegraph_b200 import records as R
from sparsifyposegraph_b200 import synth

pytestmark = pytest.mark.gpu

REL_FRO = 1e-9


def rel(a, b):
    nb = np.linalg.norm(b)
    return np.linalg.norm(a - b) / (nb if nb > 0 else 1.0)


@pytest.fixture(scope="module")
def ctx():
    from sparsifyposegraph_b200 import capi
    c = capi.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def ctx_general():
    """blanket_kernel only (the variable is read when the context is created)"""
    import os
    from sparsifyposegraph_b200 import capi
    old = os.environ.get("SPG_NO_FAST")
    os.environ["SPG_NO_FAST"] = "1"
    try:
        c = capi.Context(0)
    finally:
        if old is None:
            del os.environ["SPG_NO_FAST"]
        else:
            os.environ["SPG_NO_FAST"] = old
    yield c
    c.close()


def run(c, dim, records, rec_off, out_off):
    from sparsifyposegraph_b200 import capi
    l0 = c.launches
    out = c.remove_round(dim, R.ALG_NFR, capi.make_opts(R.TOPO_TREE, R.LIN_GLOBAL), records, rec_off, out_off)[0].copy()
    return out, c.launches - l0, c.last_retry_count


@pytest.mark.parametrize("dim,n", [(6, n) for n in range(9, 24)] + [(3, n) for n in (10, 12, 16, 20, 23)])
def test_cta_sweep_matches_blanket_kernel(ctx, ctx_general, dim, n):
    blk = synth.make_blankets(n, 48, dim=dim, variant="ring", seed=7000 + 10 * n + dim)
    nk = R.n_kept_of(blk["records"], blk["rec_off"])
    out_off = R.out_offsets(dim, R.ALG_NFR, R.TOPO_TREE, 1.0, nk)
    got, fast_launches, retried = run(ctx, dim, blk["records"], blk["rec_off"], out_off)
    ref, general_launches, _ = run(ctx_general, dim, blk["records"], blk["rec_off"], out_off)
    assert fast_launches > general_launches      # fast_kernel ran (the retry launch of blanket_kernel follows it)
    assert retried == 0
    worst_x = worst_kld = 0.0
    for b in range(blk["B"]):
        g = R.parse_out(got, out_off, b, dim, R.ALG_NFR, R.TOPO_TREE, n - 1)
        r = R.parse_out(ref, out_off, b, dim, R.ALG_NFR, R.TOPO_TREE, n - 1)
        assert g["status"] == r["status"] == 0, (b, g["status"], r["status"])
        assert [e["v"] for e in g["edges"]] == [e["v"] for e in r["edges"]], b
        worst_kld = max(worst_kld, abs(g["kld"] - r["kld"]) / max(abs(r["kld"]), 1e-3))
        for eg, er in zip(g["edges"], r["edges"]):
            assert np.allclose(eg["meas"], er["meas"], atol=1e-12)
            worst_x = max(worst_x, rel(eg["info"], er["info"]))
    assert worst_x <= REL_FRO, worst_x
    assert worst_kld <= 1e-6, worst_kld


def se3_edge(rng, poses, i, j, info=None):
    z = synth.se3_compose(synth.se3_compose(synth.se3_inverse(poses[i]), poses[j]), synth.se3_exp_small(rng, (), 0.05, 0.02))
    return {"kind": 0, "v": [i, j], "meas": z, "info": synth.random_info(rng, (), 6) if info is None else info}


def crafted_blanket(rng, n, kind):
    """n vertices, star + ring. 'ok': regular. 'c': an edge of information -100 I between two kept vertices makes
    Lambda_t + I indefinite (non-positive pivot in the C sweep). 'g': kept vertex 5 has only edges of zero information:
    its Lambda_t blocks are exactly zero, C = (Lambda_t + I)^-1 is fine and the anchored G sweep meets a zero pivot.
    'weak': kept vertex 5 hangs on the removed vertex by a 3e-6 I edge only: G = Lambda_rr^-1 is large and guard (i)
    (||G||_F <= 1e5) refuses."""
    poses = synth.random_poses(rng, (n,), 6)
    nk = n - 1
    edges = []
    for i in range(1, n):
        info = None
        if kind == "g" and i == 5:
            info = np.zeros((6, 6))
        if kind == "weak" and i == 5:
            info = 3e-6 * np.eye(6)
        edges.append(se3_edge(rng, poses, 0, i, info))
    for i in range(nk):
        a, b = 1 + i, 1 + (i + 1) % nk
        if kind == "weak" and 5 in (a, b):
            continue
        info = None
        if kind == "g" and 5 in (a, b):
            info = np.zeros((6, 6))
        if kind == "c" and (a, b) == (2, 3):
            info = -100.0 * np.eye(6)
        edges.append(se3_edge(rng, poses, a, b, info))
    return R.pack_blanket(6, list(range(100, 100 + n)), poses, edges)


@pytest.mark.parametrize("n", [12, 18])
def test_sweep_refusals_go_through_the_retry_list(ctx, ctx_general, n):
    rng = np.random.default_rng(300 + n)
    kinds = (["ok"] * 5 + ["c", "g", "weak"]) * 6
    recs = [crafted_blanket(rng, n, kind) for kind in kinds]
    records, rec_off = R.concat_records(recs)
    out_off = R.out_offsets(6, R.ALG_NFR, R.TOPO_TREE, 1.0, [n - 1] * len(recs))
    got, fast_launches, retried = run(ctx, 6, records, rec_off, out_off)
    ref, general_launches, _ = run(ctx_general, 6, records, rec_off, out_off)
    assert fast_launches > general_launches
    assert retried == sum(kind != "ok" for kind in kinds)
    for b, kind in enumerate(kinds):
        g = R.parse_out(got, out_off, b, 6, R.ALG_NFR, R.TOPO_TREE, n - 1)
        r = R.parse_out(ref, out_off, b, 6, R.ALG_NFR, R.TOPO_TREE, n - 1)
        if kind == "ok":
            assert g["status"] == r["status"] == 0, b
            assert [e["v"] for e in g["edges"]] == [e["v"] for e in r["edges"]], b
            for eg, er in zip(g["edges"], r["edges"]):
                assert rel(eg["info"], er["info"]) <= REL_FRO, b
        else:   # re-run by blanket_kernel: its record, word for word
            assert np.array_equal(got[out_off[b]:out_off[b + 1]], ref[out_off[b]:out_off[b + 1]]), (b, kind)
            if kind == "c":
                assert g["status"] == 2, (b, g["status"])     # SPG_BLANKET_NOT_PD_CHOWLIU
