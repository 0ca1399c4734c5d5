"""fast_kernel's 4-warp variant (SE3 blankets of 9 ... 16 vertices) on blankets with so many edges that their Jacobians
do not fit the shared memory at once: the assembly runs in several chunks of edges, and each thread keeps its partial
block in thread-local memory while the next chunk's Jacobians are formed. Checked against blanket_kernel alone."""
import numpy as np
import pytest

from sparsifyposegraph_b200 import records as R
from sparsifyposegraph_b200 import synth
from test_gpu_fast_sweep import REL_FRO, ctx, ctx_general, rel, run, se3_edge  # noqa: F401 (fixtures)

pytestmark = pytest.mark.gpu


def dense_blanket(rng, n, chords):
    """star + ring over the n - 1 kept vertices + `chords` further kept pairs (all of them for chords < 0)"""
    poses = synth.random_poses(rng, (n,), 6)
    nk = n - 1
    edges = [se3_edge(rng, poses, 0, i) for i in range(1, n)]
    ring = {(1 + i, 1 + (i + 1) % nk) for i in range(nk)}
    edges += [se3_edge(rng, poses, a, b) for a, b in sorted(ring)]
    others = [(a, b) for a in range(1, n) for b in range(a + 1, n) if (a, b) not in ring and (b, a) not in ring]
    if chords >= 0:
        others = [others[i] for i in sorted(rng.choice(len(others), chords, replace=False))]
    edges += [se3_edge(rng, poses, a, b) for a, b in others]
    return R.pack_blanket(6, list(range(100, 100 + n)), poses, edges)


# 12: C and G swept side by side; 16: one after the other. 66 / 120 / 44 edges: several assembly chunks each
@pytest.mark.parametrize("n,chords", [(12, -1), (16, -1), (16, 14)])
def test_chunked_assembly_matches_blanket_kernel(ctx, ctx_general, n, chords):
    rng = np.random.default_rng(500 + n + chords)
    recs = [dense_blanket(rng, n, chords) for _ in range(24)]
    records, rec_off = R.concat_records(recs)
    out_off = R.out_offsets(6, R.ALG_NFR, R.TOPO_TREE, 1.0, [n - 1] * len(recs))
    got, fast_launches, retried = run(ctx, 6, records, rec_off, out_off)
    ref, general_launches, _ = run(ctx_general, 6, records, rec_off, out_off)
    assert fast_launches > general_launches
    assert retried == 0
    worst_x = worst_kld = 0.0
    for b in range(len(recs)):
        g = R.parse_out(got, out_off, b, 6, R.ALG_NFR, R.TOPO_TREE, n - 1)
        r = R.parse_out(ref, out_off, b, 6, R.ALG_NFR, R.TOPO_TREE, n - 1)
        assert g["status"] == r["status"] == 0, (b, g["status"], r["status"])
        assert [e["v"] for e in g["edges"]] == [e["v"] for e in r["edges"]], b
        worst_kld = max(worst_kld, abs(g["kld"] - r["kld"]) / max(abs(r["kld"]), 1e-3))
        for eg, er in zip(g["edges"], r["edges"]):
            assert np.allclose(eg["meas"], er["meas"], atol=1e-12)
            worst_x = max(worst_x, rel(eg["info"], er["info"]))
    assert worst_x <= REL_FRO, worst_x
    assert worst_kld <= 1e-6, worst_kld
