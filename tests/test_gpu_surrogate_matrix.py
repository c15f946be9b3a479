"""Every instantiation of the structure-gradient surrogate (``csrc/surrogate.cuh``) against the
float64 reference, element-wise.

One evaluation of ``SparseGCNSurrogate`` launches ``gcn_propagate_kernel<HAS_VALS>`` (Z1; also the
second propagation of ``all_logits``, with null bias and null degree output),
``gcn_target_logits_kernel<HAS_VALS>``, ``gcn_grad_row_kernel`` and ``gcn_grad_col_kernel<HAS_VALS>``:
7 instantiations.  The reference is ``tests/surrogate_reference.GcnReference`` (float64, scipy
sparse) on the float32 arrays the kernels receive (``sur.xw``, ``b1``, ``W2``, ``b2``, the device CSR).

* ``TABLE``: one row per (graph, hidden width H, classes C, target).  H in {4, 8, 36, 64, 100, 124,
  128} (1 ... 32 float4 chunks: fewer than the 8 lanes per node of the row kernel, H not a multiple
  of 32, a full warp); C in {1, 2, 7, 8, 9, 41}; target rows of 0, 1, 3, 31, 32, 33, 257, 2100 and
  25 000 entries (the hub, on a graph of 200 003 nodes: beyond the reference's 20 000-node cap);
  binary and weighted graphs; n = 3001 (not a multiple of 8 or 32) and n = 1 with and without a
  self loop; clamped targets and clamped neighbours (an empty row, and a weighted row whose dyadic
  weights cancel to exactly 0).  Every case (``check_case``) checks
  - Z1 and the raw degrees (``sur.propagate()``), the logits and the context (H2[t], raw deg_t,
    a_tt) against float64;
  - row and column ``t`` of ``dLoss/dA`` for the linear loss ``<u, logits>`` (one KL loss per
    graph besides): norm-wise <= 1e-5 and element-wise ratio <= 1 at the 5e-2 floor, the ratio
    at the 1e-3 floor printed beside them;
  - the argmax of ``flip_scores`` equals the float64 argmax whenever the float64 top-two gap
    exceeds twice the norm-wise bar;
  - a second call (and a second propagation) returns the same bits.
  ReLU ties (``|Z1_64|`` within the float32 rounding bound of 0) take the kernel's sign; the count
  is printed.  Values that are identically zero in float64 while their float32 terms are not (H2
  of a row whose entries flips cancel, the row gradient of a one-node graph) are held to the
  rounding bound of their terms instead (``check_or_zero``).
* Flips: the full 64-entry list (removals, additions, a re-weighting that hits one stored entry
  twice, a diagonal flip, flips into the rows of the target's neighbours) and 65 refused, a
  flipped partner as the target, the base graph afterwards (the propagate cache), a flip that
  removes the target's last edge, and (binary graph: +-1 flips sum exactly) flips that empty a
  three-entry row.
* ``test_every_surrogate_instantiation_runs``: each row launches the instantiations it names
  (``torch.profiler``), and the table launches all 7.
* A bias at an odd float offset into a flat buffer gives the bits of an aligned one; the C ABI
  refuses a misaligned bias pointer.
"""
import re
import zlib

import numpy as np
import pytest
import scipy.sparse as sp
import torch
import torch.nn.functional as F

import efficient_gnn_b200 as egnn
from efficient_gnn_b200 import _cabi
from helpers import elementwise_ratio, rel_max_err
from models_for_tests import DenseGCN
from surrogate_reference import GcnReference
from test_gpu_adjoint_matrix import _pattern, _profiled_kernels

pytestmark = pytest.mark.gpu

NFEAT = 16
EMPTY, ZERO_SUM, LOOP = 10, 20, 18            # an empty row; dyadic weights summing to 0; a self loop
ROW_LEN = {EMPTY: 0, 11: 1, 12: 3, 13: 31, 14: 32, 15: 33, 16: 257, 17: 2100}
HUB, HUB_LEN = 7, 25_000
EPS32 = 2.0 ** -24


# ---- graphs ------------------------------------------------------------------------------------
def build_graph(name):
    """Seeded scipy CSR (float32).  "mid_*": 3001 nodes, ~8 entries per row (symmetric binary or
    directed weighted 0.5-2), rows ROW_LEN[t] entries long (those of 3 or more entries include the
    clamped nodes EMPTY and ZERO_SUM), row LOOP with a stored self loop; in "mid_w" row ZERO_SUM is
    0.5 (self loop), 0.25, -0.75, in "mid_bin" it is empty.  "hub_*": 200 003 nodes, ~5 entries per
    row, row HUB of HUB_LEN entries, row EMPTY empty.  "one_*": a single node."""
    if name.startswith("one"):
        val = {"one_empty": [], "one_loop": [1.0], "one_w": [0.5]}[name]
        return sp.csr_matrix((np.asarray(val, np.float32), np.zeros(len(val), np.int32),
                              np.asarray([0, len(val)], np.int32)), shape=(1, 1))
    rng = np.random.default_rng(zlib.crc32(name.encode()))
    weighted = name.endswith("_w")
    n, deg = (200_003, 5) if name.startswith("hub") else (3001, 8)
    a = _pattern(rng, n, deg, directed=weighted)
    special = list(ROW_LEN) + [ZERO_SUM, LOOP] if name.startswith("mid") else [HUB, EMPTY]
    keep = ~np.isin(a.row, special)
    r, c = [a.row[keep]], [a.col[keep]]
    lens = dict(ROW_LEN) if name.startswith("mid") else {HUB: HUB_LEN}
    for t, length in lens.items():
        fixed = [EMPTY, ZERO_SUM] if length >= 3 else []
        cols = rng.choice(np.arange(100, n), length - len(fixed), replace=False)
        r.append(np.full(length, t)); c.append(np.concatenate([fixed, cols]).astype(np.int64))
    if name.startswith("mid"):
        r.append(np.full(21, LOOP)); c.append(np.concatenate([[LOOP], rng.choice(np.arange(100, n), 20, False)]))
    r, c = np.concatenate(r), np.concatenate(c)
    a = sp.csr_matrix((np.ones(r.size, np.float32), (r, c)), shape=(n, n))
    a.sum_duplicates()
    a.data[:] = 1.0
    if weighted:
        a.data = rng.uniform(0.5, 2.0, a.nnz).astype(np.float32)
    if weighted and name.startswith("mid"):
        a = a.tolil()
        a[ZERO_SUM, [ZERO_SUM, 1, 2]] = [0.5, 0.25, -0.75]
        a = a.tocsr()
    a.sort_indices()
    return a


_GRAPHS, _SURROGATES = {}, {}


def graph(name):
    if name not in _GRAPHS:
        _GRAPHS[name] = build_graph(name)
    return _GRAPHS[name]


def surrogate(name, h, c):
    """(surrogate, device CSR as scipy) for a seeded DenseGCN of hidden width h and c classes."""
    key = (name, h, c)
    if key not in _SURROGATES:
        if len(_SURROGATES) > 8:
            _SURROGATES.clear()
        adj = graph(name)
        n = adj.shape[0]
        x = torch.randn(n, NFEAT, generator=torch.Generator().manual_seed(h * 100 + c))
        torch.manual_seed(h * 7 + c)
        gcn = DenseGCN(NFEAT, c, nhid=h).cuda().eval()
        sur = egnn.SparseGCNSurrogate(gcn, x.cuda(), adj)
        _SURROGATES[key] = (sur, sur.graph.to_scipy())
    return _SURROGATES[key]


# ---- one case ----------------------------------------------------------------------------------
def check(tag, got, ref, tol=1e-5):
    got = np.asarray(got, np.float64)
    err = rel_max_err(got, ref)
    r5 = elementwise_ratio(got, ref, tol)
    r3 = elementwise_ratio(got, ref, tol, floor=1e-3)
    print(f"\n[{tag}] rel {err:.2e}, elementwise_ratio x{r5:.2f} (floor 5e-2), x{r3:.2f} (floor 1e-3)")
    assert np.all(np.isfinite(got)), f"{tag}: non-finite"
    assert err <= tol, f"{tag}: rel max err {err:.3e}"
    assert r5 <= 1.0, f"{tag}: elementwise ratio {r5:.2f} at the 5e-2 floor"


def check_or_zero(tag, got, ref, terms, k):
    """``check``, or, where the float64 value is identically zero while its float32 terms are not
    (``surrogate_reference``: H2 of a row cancelled by flips, the row gradient of a one-node
    graph), the rounding bound of a float32 evaluation of k terms: |got| <= k 2^-24 sum|terms|."""
    terms = np.asarray(terms, np.float64)
    if np.abs(ref).max() > 1e-12 * terms.max():
        return check(tag, got, ref)
    worst = float((np.abs(np.asarray(got, np.float64)) / (k * EPS32 * terms + 1e-300)).max())
    print(f"\n[{tag}] identically zero: |got| at most x{worst:.2f} of its rounding bound ({k} terms)")
    assert worst <= 1.0, f"{tag}: {worst:.2f} of the rounding bound"


def kl_to_uniform(out):
    logp = F.log_softmax(out, dim=1)
    return F.kl_div(logp, torch.full_like(logp, 1.0 / logp.shape[1]), reduction="batchmean")


def gradient(sur, t, deltas, loss):
    """(logits as numpy, the StructureGradient, u = dLoss/dlogits as float64) for one loss of the
    target's logits: "linear" is <u, logits> with a seeded u, "kl" the KL divergence to uniform."""
    out = sur.target_logits(t, deltas)
    if loss == "linear":
        u = torch.tensor(np.random.default_rng(t).standard_normal(sur.n_classes).astype(np.float32), device="cuda")
        value = (out * u).sum()
    else:
        o = out.detach().requires_grad_(True)
        u = torch.autograd.grad(kl_to_uniform(o), o)[0].reshape(-1)
        value = kl_to_uniform(out)
    sg = sur.structure_gradient(value)
    return out.detach().cpu().numpy()[0], sg, u.cpu().numpy().astype(np.float64)


def check_case(tag, sur, adj, t, deltas=None, kl=False, fresh=True):
    """``fresh``: drop the propagate cache first; False reads Z1 through the cache, keyed by the
    delta list, as the attack does."""
    if fresh:
        sur._state = None
    z1_t, deg_t = sur.propagate(deltas)
    z1, deg = z1_t.cpu().numpy(), deg_t.cpu().numpy()
    ref = GcnReference(adj, sur.xw.cpu().numpy(), sur.b1.cpu().numpy(), sur.w2.cpu().numpy(), sur.b2.cpu().numpy(),
                       deltas, z1_kernel=z1)
    print(f"\n[{tag}] ReLU ties: {ref.ties}, deg_t {ref.deg_raw[t]:g}, clamped {bool(ref.clamped[t])}")
    check(f"{tag} Z1", z1, ref.z1)
    check(f"{tag} deg", deg, ref.deg_raw)
    logits, ctx = sur._target_logits(t, deltas)
    ctx = ctx.cpu().numpy()
    h = sur.h
    check(f"{tag} logits", logits.cpu().numpy(), ref.logits(t))
    if deltas is None:                                 # the target's own row (the hub: a 25 000-term sum)
        check(f"{tag} Z1[t]", z1[t], ref.z1[t])
    h2_terms, count = ref.h2_terms(t)
    check_or_zero(f"{tag} H2[t]", ctx[:h], ref.h2(t), h2_terms, count + 4)
    assert abs(ctx[128] - ref.deg_raw[t]) <= 1e-6 * max(1.0, abs(ref.deg_raw[t])), (ctx[128], ref.deg_raw[t])
    assert abs(ctx[129] - ref.a_tt(t)) <= 1e-6 * max(1.0, abs(ref.a_tt(t))), (ctx[129], ref.a_tt(t))
    assert (ctx[128] == 0) == ref.clamped[t]
    for loss in ("linear", "kl") if kl else ("linear",):
        out, sg, u = gradient(sur, t, deltas, loss)
        row, col = sg.row.cpu().numpy(), sg.col.cpu().numpy()
        row_ref, col_ref = ref.structure_grad(t, u)
        row_terms, col_terms = ref.structure_grad_terms(t, u)
        k = 2 * h + sur.n_classes + 8                 # v: C-term sums; two H-term dot products; 3 more ops
        check_or_zero(f"{tag} {loss} row", row, row_ref, row_terms, k)
        check_or_zero(f"{tag} {loss} column", col, col_ref, col_terms, k)
        # the attack's choice of flip (calib_fga.py:880-881)
        adj_row = torch.tensor(ref.a.getrow(t).toarray().ravel(), dtype=torch.float32, device="cuda")
        score = sg.flip_scores(adj_row).cpu().numpy()
        score_ref = ref.flip_scores(row_ref, col_ref, t)
        top2 = np.sort(score_ref)[-2:] if score_ref.size > 1 else None
        if top2 is None or top2[1] - top2[0] > 2e-5 * np.abs(score_ref).max():
            assert int(np.argmax(score)) == int(np.argmax(score_ref)), f"{tag}: flip choice"
        # repeatability: the same bits from a second evaluation and a second propagation
        out2, sg2, _ = gradient(sur, t, deltas, loss)
        assert np.array_equal(out, out2), f"{tag}: logits differ between calls"
        assert torch.equal(sg.row, sg2.row), f"{tag}: row differs between calls"
        assert torch.equal(sg.col, sg2.col), f"{tag}: column differs between calls"
    sur._state = None
    z1_again, deg_again = sur.propagate(deltas)
    assert torch.equal(z1_t, z1_again) and torch.equal(deg_t, deg_again), f"{tag}: propagate differs between calls"


# ---- the case table ----------------------------------------------------------------------------
# (graph, H, C, target, KL loss as well).  Binary graphs launch propagate<0>, target_logits<0>,
# grad_row, grad_col<0>; weighted ones the <1> instantiations and grad_row.
TABLE = [
    ("mid_bin", 4, 1, 11, False),
    ("mid_bin", 8, 2, 12, True),
    ("mid_bin", 36, 7, 13, False),
    ("mid_bin", 64, 8, 14, False),
    ("mid_bin", 100, 9, 15, False),
    ("mid_bin", 124, 41, 16, False),
    ("mid_bin", 128, 7, 17, False),
    ("mid_bin", 64, 7, EMPTY, False),
    ("mid_bin", 36, 9, LOOP, False),
    ("mid_w", 4, 2, 16, False),
    ("mid_w", 8, 1, 17, False),
    ("mid_w", 36, 41, 11, True),
    ("mid_w", 64, 9, 12, False),
    ("mid_w", 100, 8, 13, False),
    ("mid_w", 124, 7, 14, False),
    ("mid_w", 128, 9, 15, False),
    ("mid_w", 64, 2, ZERO_SUM, False),
    ("mid_w", 100, 7, EMPTY, False),
    ("mid_w", 8, 7, LOOP, False),
    ("hub_bin", 64, 7, HUB, True),
    ("hub_bin", 64, 7, 123_456, False),
    ("hub_w", 128, 41, HUB, True),
    ("hub_w", 36, 8, EMPTY, False),
    ("one_empty", 8, 2, 0, True),
    ("one_loop", 4, 1, 0, False),
    ("one_w", 124, 7, 0, True),
]


def expected_kernels(name):
    b = int(name.endswith("_w"))
    return {f"propagate<{b}>", f"target_logits<{b}>", "grad_row", f"grad_col<{b}>"}


def case_id(c):
    return f"{c[0]}-H{c[1]}-C{c[2]}-t{c[3]}"


@pytest.mark.parametrize("case", TABLE, ids=[case_id(c) for c in TABLE])
def test_surrogate_matrix_vs_float64(case):
    name, h, c, t, kl = case
    sur, adj = surrogate(name, h, c)
    want = {HUB: HUB_LEN, LOOP: 21, ZERO_SUM: 3}.get(t, ROW_LEN.get(t))
    if not name.startswith("one") and want is not None:
        assert adj[t].nnz == want, (t, adj[t].nnz)
    check_case(case_id(case), sur, adj, t, kl=kl)


@pytest.mark.parametrize("name", ["mid_bin", "mid_w", "one_loop", "one_empty"])
def test_all_logits(name):
    sur, adj = surrogate(name, 36, 7)
    ref = GcnReference(adj, sur.xw.cpu().numpy(), sur.b1.cpu().numpy(), sur.w2.cpu().numpy(), sur.b2.cpu().numpy(),
                       z1_kernel=sur.propagate()[0].cpu().numpy())
    with torch.no_grad():
        got = sur.all_logits().cpu().numpy()
    check(f"{name} all_logits", got, ref.all_logits())


# ---- flips -------------------------------------------------------------------------------------
class Flips:
    """A delta list built against the current values of the perturbed adjacency."""

    def __init__(self, adj):
        self.a = adj.todok()
        self.rows, self.cols, self.vals = [], [], []

    def add(self, i, j, dv):
        self.rows.append(int(i)); self.cols.append(int(j)); self.vals.append(float(dv))
        self.a[i, j] = float(np.float32(self.a[i, j] + dv))

    def set(self, i, j, value):
        self.add(i, j, float(value) - float(self.a[i, j]))

    def deltas(self):
        return list(self.rows), list(self.cols), list(self.vals)


def sixty_four_flips(adj, t, rng):
    """64 flips around target t: its diagonal, four stored entries removed (and their mirrors when
    stored), one stored entry hit twice (removed, then re-added at 0.5: three contributions to one
    column), entries into the rows of two neighbours, then new symmetric edges t <-> j."""
    fl = Flips(adj)
    n = adj.shape[0]
    stored = [int(j) for j in adj[t].indices if j != t]
    fl.set(t, t, 0.75)
    for i in stored[2:6]:
        fl.set(t, i, 0.0)
        if adj[i, t] != 0:
            fl.set(i, t, 0.0)
    twice = stored[6]
    fl.add(t, twice, -float(adj[t, twice]))
    fl.add(t, twice, 0.5)
    for i in stored[7:9]:                        # neighbours: their degree and Z1 change
        for k in rng.choice(np.arange(200, n), 3, replace=False):
            fl.set(i, k, 1.0 - float(fl.a[i, k]))
    partners = []
    while len(fl.rows) < 64:
        j = int(rng.integers(200, n))
        if fl.a[t, j] != 0 or j in partners:
            continue
        partners.append(j)
        fl.set(t, j, 1.0)
        if len(fl.rows) < 64:
            fl.set(j, t, 1.0)
    assert len(fl.rows) == 64
    return fl, partners, twice


@pytest.mark.parametrize("name", ["mid_bin", "mid_w"])
def test_sixty_four_flips(name):
    sur, adj = surrogate(name, 64, 7)
    t = 15
    fl, partners, twice = sixty_four_flips(adj, t, np.random.default_rng(3))
    deltas = fl.deltas()
    assert sum(1 for r, c in zip(*deltas[:2]) if (r, c) == (t, twice)) == 2 and adj[t, twice] != 0
    check_case(f"{name} 64 flips t={t}", sur, adj, t, deltas, kl=True)
    too_many = (deltas[0] + [t], deltas[1] + [partners[0]], deltas[2] + [1.0])
    with pytest.raises(egnn.EgnnError):
        sur.target_logits(t, too_many)
    check_case(f"{name} 64 flips, partner {partners[0]}", sur, adj, partners[0], deltas, fresh=False)
    check_case(f"{name} base graph after flips", sur, adj, t, fresh=False)


@pytest.mark.parametrize("name", ["mid_bin", "mid_w"])
def test_flip_removes_last_edge(name):
    sur, adj = surrogate(name, 8, 9)
    t = 11
    (only,) = adj[t].indices
    fl = Flips(adj)
    fl.set(t, only, 0.0)
    fl.set(only, t, 1.0)
    check_case(f"{name} last edge of {t} removed", sur, adj, t, fl.deltas(), kl=True)


def test_flips_empty_a_row():
    """Binary graph: +-1 flips cancel exactly in any order, so the emptied row is clamped in
    float32 as in float64 (weighted rows are emptied one exact removal at a time above)."""
    sur, adj = surrogate("mid_bin", 100, 2)
    t = 12
    fl = Flips(adj)
    for j in adj[t].indices:
        fl.set(t, j, 0.0)
    fl.set(13, t, 1.0)
    check_case(f"mid_bin row {t} emptied", sur, adj, t, fl.deltas())
    check_case(f"mid_bin row {t} emptied, t=13", sur, adj, 13, fl.deltas())


# ---- which kernels run -------------------------------------------------------------------------
_KERNEL = re.compile(r"gcn_(propagate|target_logits|grad_row|grad_col)_kernel(?:<([^>]*)>)?")


def gcn_keys(names):
    """Normalised ``propagate<1>`` / ``grad_row`` keys of the surrogate kernels among kernel names,
    whichever way the demangler spells the template argument."""
    out = set()
    for name in names:
        m = _KERNEL.search(name)
        if not m:
            continue
        if m.group(2) is None:
            out.add(m.group(1))
            continue
        a = re.sub(r"^\((?:bool|int)\)", "", m.group(2).strip())
        a = {"true": "1", "false": "0"}.get(a, a)
        out.add(f"{m.group(1)}<{a}>")
    return out


ALL_SEVEN = {"propagate<0>", "propagate<1>", "target_logits<0>", "target_logits<1>", "grad_row",
             "grad_col<0>", "grad_col<1>"}


def test_every_surrogate_instantiation_runs():
    probe = _profiled_kernels(lambda: torch.ones(1 << 16, device="cuda").mul_(2.0))
    if not probe:
        pytest.skip("torch.profiler records no CUDA kernel here (CUPTI unavailable): coverage not measurable")
    assert gcn_keys(["void egnn::gcn_grad_col_kernel<(bool)1>(int const*)", "egnn::gcn_grad_row_kernel(float const*)",
                     "void egnn::gcn_propagate_kernel<false>(int const*)"]) == \
        {"grad_col<1>", "grad_row", "propagate<0>"}
    launched = set()
    for case in TABLE:
        name, h, c, t, _kl = case
        sur, _adj = surrogate(name, h, c)

        def run():
            sur._state = None
            out = sur.target_logits(t)
            sur.structure_gradient((out * 1.0).sum())
        got = gcn_keys(_profiled_kernels(run))
        assert got == expected_kernels(name), f"{case_id(case)}: launched {sorted(got)}"
        launched |= got
    for name in ("mid_bin", "mid_w"):                 # the second propagation: null bias, null degrees
        sur, _adj = surrogate(name, 36, 7)
        sur.propagate()
        with torch.no_grad():
            got = gcn_keys(_profiled_kernels(sur.all_logits))
        assert got == {f"propagate<{int(name.endswith('_w'))}>"}, got
    print(f"\n[coverage] {len(launched & ALL_SEVEN)} of {len(ALL_SEVEN)} surrogate instantiations launched")
    assert launched == ALL_SEVEN, f"missing {sorted(ALL_SEVEN - launched)}"


# ---- alignment ---------------------------------------------------------------------------------
def test_bias_at_an_odd_offset_into_a_flat_buffer():
    """A model whose parameters are views into one flat buffer: the hidden bias starts one float
    past a 16-byte boundary.  The surrogate copies it to an aligned buffer (same bits as a model
    with an ordinary bias); the C ABI refuses the misaligned pointer itself."""
    adj = graph("mid_w")
    h, c = 36, 7
    x = torch.randn(adj.shape[0], NFEAT, generator=torch.Generator().manual_seed(1)).cuda()
    torch.manual_seed(2)
    plain = DenseGCN(NFEAT, c, nhid=h).cuda().eval()
    flat = torch.zeros(1 + h, device="cuda")
    flat[1:] = plain.gc1.bias.detach()
    odd = DenseGCN(NFEAT, c, nhid=h).cuda().eval()
    odd.load_state_dict(plain.state_dict())
    odd.gc1.bias.data = flat[1:]
    assert odd.gc1.bias.data_ptr() % 16 == 4
    results = []
    for gcn in (plain, odd):
        sur = egnn.SparseGCNSurrogate(gcn, x, adj)
        assert sur.b1.data_ptr() % 16 == 0
        out = sur.target_logits(16)
        sg = sur.structure_gradient((out * 1.0).sum())
        results.append((sur.propagate()[0].clone(), out.detach().clone(), sg.row.clone(), sg.col.clone()))
    for a, b in zip(*results):
        assert torch.equal(a, b)
    g = sur.graph
    y = torch.empty(g.n, h, device="cuda")
    rc = sur.lib.egnn_gcn_propagate(_cabi.ptr(g.rowptr), _cabi.ptr(g.colidx), _cabi.ptr(g.vals), _cabi.ptr(sur.xw),
                                    _cabi.ptr(odd.gc1.bias), _cabi.ptr(y), None, g.n, h, None, None, None, 0,
                                    _cabi.current_stream())
    assert rc == -1 and b"aligned" in sur.lib.egnn_last_error()
