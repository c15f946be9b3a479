"""SURVEY 8c's downstream recipe, literally: the REFERENCE's own ``WATS`` class
(calibration/WATS.py:76-170, imported unmodified from oracle/_ref) is
constructed twice on the same device with the same seeds - once untouched
(scipy path on the host), once with ``calibration.WATS.graph_wavelet_features``
monkey-patched to the CUDA builder, exactly the one-line change INTEGRATION.md
asks a maintainer to make - and evaluated as
benchmark_calibration_methods.py:100-127 does (accuracy, mean max-probability,
the reference's ``calculate_average_ece``): equal to 4 decimals.

Running the reference's class needs its modules (``oracle/_ref``, or a checkout
named by ``EGNN_REFERENCE_ROOT``).  Without them the same comparison runs
against the outputs of the reference's class stored in ``tests/golden``."""
import os

import numpy as np
import pytest
import scipy.sparse as sp
import torch

import efficient_gnn_b200 as egnn
from efficient_gnn_b200 import synth
from oracle import ref_shim
from oracle import wats_oracle as orc
from helpers import GOLDEN
from models_for_tests import FixedLogits

pytestmark = pytest.mark.gpu


def evaluate(ece_mod, model, x, y, adj, test_mask):
    """benchmark_calibration_methods.py:100-127 (evaluate_calibration) without the prints."""
    model.eval()
    with torch.no_grad():
        probs = model(x, adj).exp()
        tp, tl = probs[test_mask], y[test_mask]
        acc = (torch.argmax(tp, dim=1) == tl).float().mean().item()
        conf = torch.max(tp, dim=1)[0].mean().item()
        ece = ece_mod.calculate_average_ece(tp.cpu().numpy(), tl.cpu().numpy(), tp.shape[1], logits=False)
    return acc, conf, float(ece)


def build(wats_mod, model_mod, shape, self_loops, use_gcn):
    sh = synth.SHAPES[shape]
    rp, ci, n = synth.synth_csr(shape, self_loops=self_loops)
    adj_csr = sp.csr_matrix((np.ones(ci.numel(), np.float32), ci.numpy(), rp.numpy()), shape=(n, n))
    adj = torch.tensor(adj_csr.toarray(), dtype=torch.float32)
    y, logits, val, test = synth.synth_labels(sh.n, sh.n_classes, seed=42)
    x = torch.randn(sh.n, 16, generator=torch.Generator().manual_seed(7))
    torch.manual_seed(42)                       # benchmark_calibration_methods.py:166-167
    torch.cuda.manual_seed_all(42)
    np.random.seed(42)
    base = model_mod.CompatibleGCN(16, nclass=sh.n_classes) if use_gcn else FixedLogits(logits)
    cal = wats_mod.WATS(base, x, y, adj, val)   # the reference constructor: features + calib_train
    return cal, x.cuda(), y.cuda(), adj.cuda(), test.cuda()


@pytest.mark.parametrize("name", ["downstream_cora_stub", "downstream_cora_gcn"])
def test_cuda_fed_wats_against_the_stored_reference_class_outputs(name):
    """The reference's WATS class, run stock (scipy features, CPU, same seeds) by oracle/make_golden.py, stored its
    ``wavelet_feats`` and its accuracy / confidence / ECE.  The CUDA feature builder must return those features, and
    with the stub base model the calibrator trained on them on the GPU must give the stored metrics to 4 decimals.
    The GCN base model's dropout masks come from the device's generator, so there only the features compare."""
    g = np.load(os.path.join(GOLDEN, f"{name}.npz"))
    shape, self_loops, use_gcn = str(g["shape"]), bool(g["self_loops"]), bool(g["use_gcn"])
    sh = synth.SHAPES[shape]
    rp, ci, n = synth.synth_csr(shape, self_loops=self_loops)
    adj_csr = sp.csr_matrix((np.ones(ci.numel(), np.float32), ci.numpy(), rp.numpy()), shape=(n, n))
    adj = torch.tensor(adj_csr.toarray(), dtype=torch.float32)
    feats = egnn.graph_wavelet_features(adj.cuda(), 3, 0.8)          # the call WATS.py:99 makes once swapped
    assert feats.is_cuda and feats.dtype == torch.float32 and feats.shape == g["wavelet_feats"].shape
    np.testing.assert_allclose(feats.cpu().numpy(), g["wavelet_feats"], rtol=0, atol=1e-6)
    if use_gcn:
        return
    y, logits, val, test = synth.synth_labels(sh.n, sh.n_classes, seed=42)
    x = torch.randn(sh.n, 16, generator=torch.Generator().manual_seed(7))
    torch.manual_seed(42)                       # as make_golden.py seeded the reference's constructor
    torch.cuda.manual_seed_all(42)
    np.random.seed(42)
    cal = egnn.WATS(FixedLogits(logits), x, y, adj, val, verbose=False)
    assert cal.wavelet_feats.is_cuda
    assert sorted(k for k in cal.state_dict() if k.startswith("net.")) == sorted(k for k in g.files if k.startswith("net."))
    cal.eval()
    with torch.no_grad():
        lp = cal(x, adj).cpu().numpy()
    for got, what in zip(orc.evaluate_probs(lp, y.numpy(), test.numpy()), ("acc", "conf", "ece")):
        assert round(got, 4) == round(float(g[what]), 4), f"{what}: cuda-fed {got} vs reference {float(g[what])}"


@pytest.mark.skipif(ref_shim.reference_root() is None,
                    reason="needs the reference's modules: oracle/_ref, or a checkout named by EGNN_REFERENCE_ROOT")
@pytest.mark.parametrize("shape,self_loops,use_gcn", [("cora", False, True), ("cora", True, False),
                                                      ("pubmed", True, True)])
def test_reference_wats_class_with_the_cuda_feature_builder(monkeypatch, shape, self_loops, use_gcn):
    wats_mod, model_mod, ece_mod = ref_shim.load_reference()
    assert wats_mod.WATS.__module__ == "calibration.WATS" and wats_mod is not egnn.wats
    stock = build(wats_mod, model_mod, shape, self_loops, use_gcn)
    m_stock = evaluate(ece_mod, *stock)

    calls = []

    def cuda_builder(adj_matrix, k=3, s=0.8):
        calls.append((adj_matrix.shape, k, s))
        return egnn.graph_wavelet_features(adj_matrix, k, s)

    monkeypatch.setattr(wats_mod, "graph_wavelet_features", cuda_builder)
    swapped = build(wats_mod, model_mod, shape, self_loops, use_gcn)
    m_swapped = evaluate(ece_mod, *swapped)
    assert calls == [((synth.SHAPES[shape].n,) * 2, 3, 0.8)]          # WATS.py:99 reached the CUDA builder
    f_stock, f_swapped = stock[0].wavelet_feats, swapped[0].wavelet_feats
    assert f_swapped.is_cuda and f_swapped.dtype == torch.float32 and f_swapped.shape == f_stock.shape
    assert torch.allclose(f_swapped, f_stock, rtol=0, atol=1e-6)
    assert list(stock[0].state_dict()) == list(swapped[0].state_dict())
    for a, b, what in zip(m_swapped, m_stock, ("accuracy", "confidence", "ece")):
        assert round(a, 4) == round(b, 4), f"{what}: cuda {a} vs reference {b}"
    print(f"\n[{shape}] acc/conf/ece reference {m_stock} cuda-fed {m_swapped}")
