"""The SELL plan's list of hub rows (rows with more than 24 partial sums, summed by a whole warp
in the step kernel's epilogue): it must name exactly the hub rows of every CTA's epilogue range,
and the features must match the oracle when one CTA holds more hub rows than it has warps."""
import numpy as np
import pytest
import scipy.sparse as sp
import torch

import efficient_gnn_b200 as egnn
from oracle import wats_oracle as orc
from test_gpu_parity import check_parts

pytestmark = pytest.mark.gpu

EPI_WARP_ROW = 24          # kSellEpiWarpRow (sell.cuh)


def hub_lists(plan):
    """Per CTA: the plan's hub rows, and the rows of its epilogue range with > 24 partial sums."""
    n_cta = plan.n_cta
    bufs = plan._keepalive
    hub = bufs["hub"].cpu().numpy()
    ranges = bufs["cta_info"].cpu().numpy()[2 * n_cta + 64: 3 * n_cta + 65]
    parts = np.diff(bufs["rv_ptr"].cpu().numpy())
    assert hub.size == n_cta + 1 + plan.n_hub and hub[0] == 0 and hub[n_cta] == plan.n_hub
    got = [hub[n_cta + 1 + hub[g]: n_cta + 1 + hub[g + 1]] for g in range(n_cta)]
    want = [ranges[g] + np.flatnonzero(parts[ranges[g]: ranges[g + 1]] > EPI_WARP_ROW) for g in range(n_cta)]
    return got, want


def hub_graph(n=60000, n_hub=100, hub_deg=6500, seed=0):
    """A ring plus n_hub consecutive rows linked to hub_deg random columns each (symmetrised):
    every such row has more than 24 partial sums, and since the epilogue ranges are cut by cost
    the CTA at the front holds more of them than it has warps."""
    rng = np.random.default_rng(seed)
    i = np.arange(n)
    rows = [i, (i + 1) % n]
    cols = [(i + 1) % n, i]
    for h in range(n_hub):
        c = rng.choice(n, hub_deg, replace=False)
        rows += [np.full(hub_deg, h), c]
        cols += [c, np.full(hub_deg, h)]
    r, c = np.concatenate(rows), np.concatenate(cols)
    adj = sp.csr_matrix((np.ones(r.size, np.float32), (r, c)), shape=(n, n))
    adj.data[:] = 1.0
    adj.sort_indices()
    return adj


def test_plan_lists_the_hub_rows_of_every_epilogue_range():
    adj = hub_graph()
    g = egnn.CsrGraph(torch.from_numpy(adj.indptr.astype(np.int32)).cuda(),
                      torch.from_numpy(adj.indices.astype(np.int32)).cuda(), None, adj.shape[0])
    plan = g.sell_plan(force=True)
    got, want = hub_lists(plan)
    for a, b in zip(got, want):
        assert np.array_equal(a, b)
    assert max(len(a) for a in got) > 32, "the graph no longer puts more hub rows than warps in one CTA"
    res = egnn.graph_wavelet_features(g, k=4, s=[0.8, 1.6], return_parts=True, _use_sell=True)
    p = orc.wavelet_parts(adj, k=4, s=[0.8, 1.6])
    check_parts(res, p["T"], p["S"], p["H"], "hub-heavy sell")
    again = egnn.graph_wavelet_features(g, k=4, s=[0.8, 1.6], return_parts=True, _use_sell=True)
    for a, b in zip(res.orders, again.orders):
        assert torch.equal(a, b)
