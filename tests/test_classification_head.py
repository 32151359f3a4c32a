"""CPU tier: the classification heads (EngineBinaryClassificationFFN + BCE, EngineMulticlassClassificationFFN + cross entropy)
inside EngineMPNN, against the reference's own `MPNN.training_step` (tests/golden/fixture_mpnn_head_bce.npz,
fixture_mpnn_head_multiclass.npz; tests/make_golden_classification.py), with the kernel wrappers emulated (tests/emu.py plus the
emulations of dmpnn_bce_loss / dmpnn_ce_loss / dmpnn_class_probs(_bwd) below, written from include/dmpnn.h).  The same check
runs on the real kernels in tests/test_gpu_classification_head.py."""
import copy
import inspect

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from chemprop_b200 import engine
from oracle.ref_shim import reference_available
from tests import emu
from tests.util import golden_bmg, load_golden


# ---- emulations of the new kernels (torch, f32) ------------------------------------------------------------------
def _weights(Y, w, tw):
    m = torch.isfinite(Y)
    ww = (w.view(-1, 1) if w is not None else 1.0) * (tw.view(1, -1) if tw is not None else 1.0) * m
    return m, ww, m.sum().clamp(min=1)


def bce_loss(P, Y, w, tw, loss, dP):
    m, ww, n = _weights(Y, w, tw)
    y = torch.where(m, Y, torch.zeros_like(Y))
    L = P.clamp(min=0) - P * y + torch.log1p(torch.exp(-P.abs()))
    loss.copy_(((ww * L).sum() / n).reshape(1))
    dP.copy_(ww * (torch.sigmoid(P) - y) / n)


def ce_loss(P, Y, w, tw, loss, dP, C):
    B, T = Y.shape
    Z = P.reshape(B, T, C)
    m, ww, n = _weights(Y, w, tw)
    y = torch.where(m, Y, torch.zeros_like(Y))
    valid = (y >= 0) & (y < C) & (y == torch.floor(y))
    k = torch.where(valid, y, torch.zeros_like(y)).long()
    L = torch.logsumexp(Z, -1) - Z.gather(-1, k.unsqueeze(-1)).squeeze(-1)
    L = torch.where(valid, L, torch.full_like(L, float("nan")))
    loss.copy_((torch.where(m, ww * L, torch.zeros_like(L)).sum() / n).reshape(1))
    G = torch.softmax(Z, -1) - F.one_hot(k, C).to(Z.dtype)
    G = torch.where(valid.unsqueeze(-1), G, torch.full_like(G, float("nan")))
    G = torch.where(m.unsqueeze(-1), ww.unsqueeze(-1) * G / n, torch.zeros_like(G))
    dP.copy_(G.reshape(B, T * C))


def class_probs(P, C, Q):
    B = P.shape[0]
    Q.copy_(torch.sigmoid(P) if C == 1 else torch.softmax(P.reshape(B, -1, C), -1).reshape(B, -1))


def class_probs_bwd(Q, dQ, C, dP):
    if C == 1:
        dP.copy_(dQ * Q * (1 - Q))
        return
    B = Q.shape[0]
    q, g = Q.reshape(B, -1, C), dQ.reshape(B, -1, C)
    dP.copy_((q * (g - (g * q).sum(-1, keepdim=True))).reshape(B, -1))


def patch_engine(monkeypatch):
    emu.patch_engine(monkeypatch)
    for name in ("bce_loss", "ce_loss", "class_probs", "class_probs_bwd"):
        monkeypatch.setattr(engine, name, globals()[name])


# ---- the fixture check (shared with the GPU tier) ----------------------------------------------------------------
HEADS = {
    "bce": ("fixture_mpnn_head_bce",
            lambda N: N.EngineBinaryClassificationFFN(n_tasks=3, input_dim=40, hidden_dim=24, n_layers=2)),
    "multiclass": ("fixture_mpnn_head_multiclass",
                   lambda N: N.EngineMulticlassClassificationFFN(n_classes=4, n_tasks=2, input_dim=40, hidden_dim=24,
                                                                 n_layers=2)),
}

# torchmetrics' running accumulators of the reference criterion: not persistent in torchmetrics, buffers under the shim
METRIC_STATES = ("total_loss", "num_samples")


def reference_state(g: dict) -> dict:
    return {k[len("param."):]: torch.from_numpy(np.asarray(v)) for k, v in g.items()
            if k.startswith("param.") and not k.endswith(METRIC_STATES)}


def check_classification_head(kind: str, device: str, rtol: float = 2e-4, atol: float = 2e-6, graph: bool = False):
    """EngineMPNN.training_loss with a classification head (encoder -> aggregation -> batch norm -> FFN -> masked, sample- and
    task-weighted BCE / cross entropy) against the reference's `MPNN.training_step`: loss, every gradient, the batch-norm
    running statistics after the step, and eval-mode probabilities.  `graph`: the step runs as a captured CUDA graph."""
    import chemprop_b200.nn as N

    name, make = HEADS[kind]
    g = load_golden(name)
    model = N.EngineMPNN(N.BondMessagePassing(d_h=40, depth=3), N.MeanAggregation(), make(N), batch_norm=True)
    res = model.load_state_dict(reference_state(g), strict=True)
    assert not res.missing_keys and not res.unexpected_keys
    model = model.to(device)
    model.train()
    bmg = golden_bmg(g, device)
    Y, w = torch.from_numpy(g["Y"]).to(device), torch.from_numpy(g["w"]).to(device)
    if graph:
        from chemprop_b200.graph import CudaGraphStep

        for p in model.parameters():
            p.grad = torch.zeros_like(p)
        rm0, rv0, nb0 = model.bn.running_mean.clone(), model.bn.running_var.clone(), model.bn.num_batches_tracked.clone()

        def fn(b):
            for p in model.parameters():
                p.grad.zero_()
            loss = model.training_loss(b, Y, w)
            loss.backward()
            return loss

        step = CudaGraphStep(fn)
        step(bmg)                           # warm-up + capture + first replay
        model.bn.running_mean.copy_(rm0); model.bn.running_var.copy_(rv0); model.bn.num_batches_tracked.copy_(nb0)
        loss = step(bmg).clone()            # the step the reference took, from its initial running statistics
        assert step.captures == 1 and step.replays == 2
    else:
        loss = model.training_loss(bmg, Y, w)
        loss.backward()
    np.testing.assert_allclose(loss.detach().cpu().numpy(), g["loss"], rtol=rtol, atol=atol)
    for k, p in model.named_parameters():
        np.testing.assert_allclose(p.grad.cpu().numpy(), g["grad." + k], rtol=rtol, atol=atol, err_msg=k)
    for k in ("running_mean", "running_var", "num_batches_tracked"):
        np.testing.assert_allclose(getattr(model.bn, k).cpu().numpy(), g["after.bn." + k], rtol=1e-5, atol=1e-6, err_msg=k)
    model.eval()
    with torch.no_grad():
        preds = model(bmg)
    assert tuple(preds.shape) == g["preds_eval"].shape
    np.testing.assert_allclose(preds.cpu().numpy(), g["preds_eval"], rtol=rtol, atol=1e-5)


@pytest.mark.parametrize("kind", sorted(HEADS))
def test_engine_mpnn_classification_head_matches_reference_training_step(kind, monkeypatch):
    patch_engine(monkeypatch)
    check_classification_head(kind, "cpu")


# ---- the emulations against torch's own criteria -------------------------------------------------------------
def test_emulated_criteria_match_torch():
    torch.manual_seed(0)
    B, T, C = 9, 3, 4
    w, tw = torch.rand(B) + 0.5, torch.rand(T) + 0.5
    P = torch.randn(B, T) * 5
    Y = torch.rand(B, T)
    Y[1, 2] = Y[4, 0] = float("nan")
    m = torch.isfinite(Y)
    Pg = P.clone().requires_grad_(True)
    ref = (F.binary_cross_entropy_with_logits(Pg, Y.nan_to_num(), reduction="none") * w[:, None] * tw * m).sum() / m.sum()
    ref.backward()
    loss, dP = torch.empty(1), torch.empty_like(P)
    bce_loss(P, Y, w, tw, loss, dP)
    torch.testing.assert_close(loss[0], ref.detach())
    torch.testing.assert_close(dP, Pg.grad)

    Z = torch.randn(B, T, C) * 3
    K = torch.randint(0, C, (B, T)).float()
    K[0, 1] = float("nan")
    m = torch.isfinite(K)
    Zg = Z.clone().requires_grad_(True)
    ref = (F.cross_entropy(Zg.transpose(1, 2), K.nan_to_num().long(), reduction="none") * w[:, None] * tw * m).sum() / m.sum()
    ref.backward()
    dP = torch.empty(B, T * C)
    ce_loss(Z.reshape(B, -1), K, w, tw, loss, dP, C)
    torch.testing.assert_close(loss[0], ref.detach())
    torch.testing.assert_close(dP.reshape(B, T, C), Zg.grad)
    K[3, 2] = 4.0                                                        # out of range -> NaN, not a raise
    ce_loss(Z.reshape(B, -1), K, w, tw, loss, dP, C)
    assert torch.isnan(loss[0])
    K = torch.full((B, T), float("nan"))                                 # all masked -> 0, zero gradient
    ce_loss(Z.reshape(B, -1), K, w, tw, loss, dP, C)
    assert loss[0] == 0 and not dP.any()

    for c, X in ((1, torch.randn(B, T)), (C, torch.randn(B, T * C))):
        Xg = X.clone().requires_grad_(True)
        q = torch.sigmoid(Xg) if c == 1 else torch.softmax(Xg.reshape(B, -1, c), -1).reshape(B, -1)
        G = torch.randn_like(X)
        (q * G).sum().backward()
        Q, dX = torch.empty_like(X), torch.empty_like(X)
        class_probs(X, c, Q)
        class_probs_bwd(Q, G, c, dX)
        torch.testing.assert_close(Q, q.detach())
        torch.testing.assert_close(dX, Xg.grad)


# ---- module behaviour --------------------------------------------------------------------------------------------
def test_classification_heads_module_tree_hparams_and_shapes(monkeypatch):
    import chemprop_b200.nn as N

    patch_engine(monkeypatch)
    torch.manual_seed(0)
    b = N.EngineBinaryClassificationFFN(n_tasks=3, input_dim=16, hidden_dim=8, n_layers=2, task_weights=torch.tensor([1., 2., 3.]))
    m = N.EngineMulticlassClassificationFFN(n_classes=4, n_tasks=2, input_dim=16, hidden_dim=8, n_layers=2)
    assert (b.n_tasks, b.output_dim, m.n_tasks, m.n_classes, m.output_dim) == (3, 3, 2, 4, 8)
    assert tuple(b.criterion.task_weights.shape) == (1, 3) and tuple(m.criterion.task_weights.shape) == (1, 2)
    assert set(b.state_dict()) == {"ffn.0.0.weight", "ffn.0.0.bias", "ffn.1.2.weight", "ffn.1.2.bias", "ffn.2.2.weight",
                                  "ffn.2.2.bias", "criterion.task_weights"}
    assert m.hparams["cls"] is N.EngineMulticlassClassificationFFN and m.hparams["n_classes"] == 4
    for mod in (b, m):
        rebuilt = mod.hparams["cls"](**{k: v for k, v in mod.hparams.items() if k != "cls"})   # models/model.py:267-271
        assert type(rebuilt) is type(mod) and set(rebuilt.state_dict()) == set(mod.state_dict())
        rebuilt.load_state_dict(mod.state_dict(), strict=True)
        for k, v in mod.state_dict().items():
            assert torch.equal(rebuilt.state_dict()[k], v), k
    Z = torch.randn(5, 16)
    assert tuple(b.train_step(Z).shape) == (5, 3) and tuple(m.train_step(Z).shape) == (5, 2, 4)
    pb, pm = b(Z), m(Z)
    torch.testing.assert_close(pb, torch.sigmoid(b.train_step(Z)))
    torch.testing.assert_close(pm, torch.softmax(m.train_step(Z), -1))
    with pytest.raises(NotImplementedError):
        b.criterion(b.train_step(Z), torch.zeros(5, 3), lt_mask=torch.zeros(5, 3, dtype=torch.bool))
    with pytest.raises(NotImplementedError):
        m.criterion(m.train_step(Z), torch.zeros(5, 2), gt_mask=torch.zeros(5, 2, dtype=torch.bool))
    # an explicit mask (the reference MPNN's call: mask, NaN-free targets) equals NaN-as-mask
    Y = torch.randint(0, 4, (5, 2)).float()
    mask = torch.ones(5, 2, dtype=torch.bool)
    mask[1, 0] = False
    Yn = Y.clone()
    Yn[1, 0] = float("nan")
    torch.testing.assert_close(m.criterion(m.train_step(Z), Y, mask), m.criterion(m.train_step(Z), Yn))


def test_probabilities_are_differentiable(monkeypatch):
    import chemprop_b200.nn as N

    patch_engine(monkeypatch)
    torch.manual_seed(1)
    m = N.EngineMulticlassClassificationFFN(n_classes=3, n_tasks=2, input_dim=6, hidden_dim=5, n_layers=1)
    ref = copy.deepcopy(m)
    Z = torch.randn(4, 6)
    G = torch.randn(4, 2, 3)
    (m(Z) * G).sum().backward()
    (torch.softmax(ref.train_step(Z), -1) * G).sum().backward()
    for (k, p), (_, q) in zip(m.named_parameters(), ref.named_parameters()):
        torch.testing.assert_close(p.grad, q.grad, msg=k)


def test_cpu_tensors_raise():
    import chemprop_b200.nn as N
    from chemprop_b200 import DmpnnError

    P, Y = torch.zeros(4, 3), torch.zeros(4, 3)
    loss = torch.empty(1)
    with pytest.raises(DmpnnError):
        engine.bce_loss(P, Y, None, None, loss, torch.empty_like(P))
    with pytest.raises(DmpnnError):
        engine.ce_loss(torch.zeros(4, 6), torch.zeros(4, 3), None, None, loss, torch.empty(4, 6), 2)
    with pytest.raises(DmpnnError):
        engine.class_probs(P, 1, torch.empty_like(P))
    with pytest.raises(DmpnnError):
        engine.class_probs_bwd(P, P, 1, torch.empty_like(P))
    b = N.EngineBinaryClassificationFFN(n_tasks=3, input_dim=8, hidden_dim=4)
    m = N.EngineMulticlassClassificationFFN(n_classes=2, n_tasks=3, input_dim=8, hidden_dim=4)
    for mod in (b, m):
        with pytest.raises(DmpnnError):
            mod(torch.zeros(4, 8))
        with pytest.raises(DmpnnError):
            mod.criterion(torch.zeros(4, 3) if mod is b else torch.zeros(4, 3, 2), Y)


# ---- against the reference package (skipped where it is not reachable) --------------------------------------------
needs_reference = pytest.mark.skipif(not reference_available(), reason="reference tree not reachable")


@needs_reference
@pytest.mark.parametrize("kind", sorted(HEADS))
def test_fixture_matches_the_live_reference(kind):
    from tests import make_golden_classification as make_golden

    name = HEADS[kind][0]
    nt = torch.get_num_threads()
    torch.set_num_threads(1)                   # the summation order the generator uses
    try:
        live = make_golden.CASES[name]()
    finally:
        torch.set_num_threads(nt)
    g = load_golden(name)
    assert set(live) == set(g)
    for k in g:
        np.testing.assert_allclose(np.asarray(live[k]), np.asarray(g[k]), rtol=1e-6, atol=1e-7, err_msg=k)


@needs_reference
@pytest.mark.parametrize("kind", sorted(HEADS))
def test_reference_classification_state_dict_loads_both_ways(kind, monkeypatch):
    from oracle.ref_shim import import_reference

    import_reference()
    import chemprop.nn as ref_nn
    from chemprop.models import MPNN

    import chemprop_b200.nn as N
    from chemprop_b200.integrate import register_with_chemprop

    patch_engine(monkeypatch)
    torch.manual_seed(5)
    if kind == "bce":
        ref_pred = ref_nn.BinaryClassificationFFN(n_tasks=3, input_dim=40, hidden_dim=24, n_layers=2,
                                                  task_weights=torch.tensor([0.5, 1.0, 2.0]))
        ours_pred = N.EngineBinaryClassificationFFN(n_tasks=3, input_dim=40, hidden_dim=24, n_layers=2)
    else:
        ref_pred = ref_nn.MulticlassClassificationFFN(n_classes=4, n_tasks=2, input_dim=40, hidden_dim=24, n_layers=2,
                                                      task_weights=torch.tensor([1.5, 0.75]))
        ours_pred = N.EngineMulticlassClassificationFFN(n_classes=4, n_tasks=2, input_dim=40, hidden_dim=24, n_layers=2)
    ref = MPNN(ref_nn.BondMessagePassing(d_h=40), ref_nn.MeanAggregation(), ref_pred, batch_norm=True)
    ours = N.EngineMPNN(N.BondMessagePassing(d_h=40), N.MeanAggregation(), ours_pred, batch_norm=True)
    sd = {k: v for k, v in ref.state_dict().items() if not k.startswith("metrics.") and not k.endswith(METRIC_STATES)}
    ours.load_state_dict(sd, strict=True)                                   # reference -> engine
    for k, v in sd.items():
        assert torch.equal(ours.state_dict()[k], v), k
    assert torch.equal(ours.predictor.criterion.task_weights, ref.predictor.criterion.task_weights)
    ref2 = MPNN(ref_nn.BondMessagePassing(d_h=40), ref_nn.MeanAggregation(), copy.deepcopy(ref_pred), batch_norm=True)
    res = ref2.load_state_dict(ours.state_dict(), strict=False)             # engine -> reference
    assert not res.unexpected_keys
    assert all(k.startswith("metrics.") or k.endswith(METRIC_STATES) for k in res.missing_keys), res.missing_keys
    for k, v in ours.state_dict().items():
        assert torch.equal(ref2.state_dict()[k], v), k
    ref_args = inspect.signature(type(ref_pred).__init__).parameters                # hparams rebuild the reference class too
    assert set(ours_pred.hparams) - {"cls"} <= set(ref_args), set(ours_pred.hparams) - set(ref_args)
    assert ours_pred.n_tasks == ref_pred.n_tasks and ours_pred.output_dim == ref_pred.output_dim
    register_with_chemprop()
    from chemprop.nn.predictors import BinaryClassificationFFN, MulticlassClassificationFFN

    assert isinstance(ours_pred, BinaryClassificationFFN) == (kind == "bce")
    assert isinstance(ours_pred, MulticlassClassificationFFN) == (kind == "multiclass")    # chemprop/cli/predict.py:509, 546
