"""fast_kernel with the C and anchored G block sweeps side by side (CTA-wide variants whose CTA holds nk^2 threads):
one device round of mixed SE3 blanket sizes under one bucket bound, so that a single fused launch meets nk = 2 (serial
order), small nk and the full nk = 11, against blanket_kernel alone (SPG_NO_FAST=1, same binary)."""
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


def mixed_round(sizes, per_size, seed):
    """per_size ring blankets of every size, shuffled into one round"""
    rng = np.random.default_rng(seed)
    recs = []
    for n in sizes:
        blk = synth.make_blankets(n, per_size, dim=6, variant="ring", seed=seed + n)
        recs += [blk["records"][blk["rec_off"][b]:blk["rec_off"][b + 1]] for b in range(per_size)]
    order = rng.permutation(len(recs))
    records, rec_off = R.concat_records([recs[i] for i in order])
    return records, rec_off


def run_device(c, records, rec_off, out_off, max_nv, max_e):
    import torch
    from sparsifyposegraph_b200 import capi
    d_rec = torch.from_numpy(records.view(np.int64)).cuda()
    d_rec_off = torch.from_numpy(rec_off).cuda()
    d_out_off = torch.from_numpy(out_off).cuda()
    d_out = torch.zeros(int(out_off[-1]), dtype=torch.int64, device="cuda")
    l0 = c.launches
    c.remove_round_device(6, R.ALG_NFR, capi.make_opts(R.TOPO_TREE, R.LIN_GLOBAL), len(rec_off) - 1, d_rec.data_ptr(),
                          d_rec_off.data_ptr(), d_out_off.data_ptr(), d_out.data_ptr(), max_nv, max_e)
    c.sync()
    return d_out.cpu().numpy().view(np.uint64), c.launches - l0, c.last_retry_count


def test_fused_launch_of_mixed_sizes_matches_blanket_kernel(ctx, ctx_general):
    sizes = (3, 7, 9, 12)
    records, rec_off = mixed_round(sizes, 24, 8100)
    nk = R.n_kept_of(records, rec_off)
    out_off = R.out_offsets(6, R.ALG_NFR, R.TOPO_TREE, 1.0, nk)
    max_nv, max_e = 12, 22   # 12-vertex ring: 11 star + 11 ring edges
    got, fast_launches, retried = run_device(ctx, records, rec_off, out_off, max_nv, max_e)
    ref, general_launches, _ = run_device(ctx_general, records, rec_off, out_off, max_nv, max_e)
    assert fast_launches > general_launches      # fast_kernel ran (the retry launch of blanket_kernel follows it)
    assert retried == 0
    worst_x = worst_kld = 0.0
    for b in range(len(nk)):
        g = R.parse_out(got, out_off, b, 6, R.ALG_NFR, R.TOPO_TREE, int(nk[b]))
        r = R.parse_out(ref, out_off, b, 6, R.ALG_NFR, R.TOPO_TREE, int(nk[b]))
        assert g["status"] == r["status"] == 0, (b, g["status"], r["status"])
        assert [e["v"] for e in g["edges"]] == [e["v"] for e in r["edges"]], b
        worst_kld = max(worst_kld, abs(g["kld"] - r["kld"]) / max(abs(r["kld"]), 1e-3))
        for eg, er in zip(g["edges"], r["edges"]):
            assert np.allclose(eg["meas"], er["meas"], atol=1e-12)
            worst_x = max(worst_x, rel(eg["info"], er["info"]))
    assert worst_x <= REL_FRO, worst_x
    assert worst_kld <= 1e-6, worst_kld
