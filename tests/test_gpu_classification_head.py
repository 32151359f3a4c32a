"""GPU tier: the classification heads on the engine's kernels (csrc/head.cu: dmpnn_bce_loss, dmpnn_ce_loss, dmpnn_class_probs
and its mirror) -- the reference's own `MPNN.training_step` with BinaryClassificationFFN / MulticlassClassificationFFN
(tests/golden/fixture_mpnn_head_{bce,multiclass}.npz), eager and as one CUDA graph; the kernels against f64 torch; and the
C2-size training step with a 12-task BCE head replayed as a CUDA graph on new batches."""
import pytest
import torch
import torch.nn.functional as F

from chemprop_b200 import engine

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("kind", ["bce", "multiclass"])
@pytest.mark.parametrize("graph", [False, True])
def test_engine_mpnn_classification_head_matches_reference_training_step(kind, graph):
    from tests.test_classification_head import check_classification_head

    check_classification_head(kind, "cuda", graph=graph)


def _weights(B, T, gen):
    return (torch.rand(B, generator=gen) * 1.5 + 0.5).cuda(), (torch.rand(T, generator=gen) * 1.5 + 0.5).cuda()


def _mask_(Y, gen, frac=0.1):
    drop = torch.rand(Y.shape, generator=gen) < frac
    Y[drop.cuda()] = float("nan")
    if Y.numel() > 3:
        Y.view(-1)[1] = float("inf")                                         # any non-finite target is masked
    return Y


def _bce_inputs(B, T, seed):
    gen = torch.Generator().manual_seed(seed)
    P = torch.randn(B, T, generator=gen) * 6
    big = torch.rand(B, T, generator=gen) < 0.05
    P[big] = (torch.rand(int(big.sum()), generator=gen) * 200 - 100)         # logits up to |z| = 100
    if B * T >= 2:
        P.view(-1)[0], P.view(-1)[-1] = 100.0, -100.0
    hard = (torch.rand(B, T, generator=gen) < 0.5).float()
    soft = torch.rand(B, T, generator=gen)
    Y = torch.where(torch.rand(B, T, generator=gen) < 0.3, soft, hard)         # soft labels in [0, 1] and hard 0 / 1
    w, tw = _weights(B, T, gen)
    return P.cuda(), _mask_(Y.cuda(), gen), w, tw


def _ref_loss_and_grad(loss_fn, P, Y, w, tw):
    """f64 torch: sum(w tw m L) / sum m and its gradient w.r.t. the logits (m = isfinite(Y))."""
    m = torch.isfinite(Y)
    P64 = P.double().requires_grad_(True)
    L = loss_fn(P64, Y.double().nan_to_num(0.0, 0.0, 0.0))
    loss = (L * w.double()[:, None] * tw.double()[None, :] * m).sum() / m.sum().clamp(min=1)
    loss.backward()
    return loss.detach(), P64.grad


@pytest.mark.parametrize("B,T", [(1, 1), (14, 3), (10_000, 12), (10_000, 617)])
def test_bce_kernel_vs_f64_torch(B, T):
    P, Y, w, tw = _bce_inputs(B, T, seed=B + T)
    ref, dref = _ref_loss_and_grad(lambda z, y: F.binary_cross_entropy_with_logits(z, y, reduction="none"), P, Y, w, tw)
    loss, dP = torch.empty(1, device="cuda"), torch.empty_like(P)
    engine.bce_loss(P, Y, w, tw, loss, dP)
    torch.testing.assert_close(loss[0].double(), ref, rtol=2e-5, atol=1e-7)
    torch.testing.assert_close(dP.double(), dref, rtol=1e-5, atol=1e-6 * float(dref.abs().max().clamp(min=1e-30)))
    assert not dP[~torch.isfinite(Y)].any()


def _ce_inputs(B, T, C, seed):
    gen = torch.Generator().manual_seed(seed)
    Z = torch.randn(B, T * C, generator=gen) * 4
    big = torch.rand(B, T * C, generator=gen) < 0.02
    Z[big] = (torch.rand(int(big.sum()), generator=gen) * 100 - 50)
    K = torch.randint(0, C, (B, T), generator=gen).float()
    w, tw = _weights(B, T, gen)
    return Z.cuda(), _mask_(K.cuda(), gen), w, tw


@pytest.mark.parametrize("B", [1, 513, 10_000])
@pytest.mark.parametrize("C,T", [(2, 1), (4, 2), (10, 12)])
def test_ce_kernel_vs_f64_torch(B, C, T):
    Z, K, w, tw = _ce_inputs(B, T, C, seed=B * 7 + C * 3 + T)
    m = torch.isfinite(K)
    ref, dref = _ref_loss_and_grad(
        lambda z, y: F.cross_entropy(z.reshape(B, T, C).transpose(1, 2), y.long(), reduction="none"), Z, K, w, tw)
    loss, dP = torch.empty(1, device="cuda"), torch.empty_like(Z)
    engine.ce_loss(Z, K, w, tw, loss, dP, C)
    torch.testing.assert_close(loss[0].double(), ref, rtol=2e-5, atol=1e-7)
    torch.testing.assert_close(dP.double(), dref, rtol=1e-5, atol=1e-6 * float(dref.abs().max().clamp(min=1e-30)))
    assert not dP.reshape(B, T, C)[~m].any()


@pytest.mark.parametrize("B,T,C", [(1, 1, 1), (513, 12, 1), (10_000, 617, 1), (1, 2, 4), (513, 12, 3), (10_000, 12, 10)])
def test_class_probs_kernels_vs_f64_torch(B, T, C):
    gen = torch.Generator().manual_seed(B + T + C)
    Z = (torch.randn(B, T * C, generator=gen) * 8).cuda()
    Z.view(-1)[0] = 100.0
    Z.view(-1)[-1] = -100.0
    G = torch.randn(B, T * C, generator=gen).cuda()
    Z64 = Z.double().requires_grad_(True)
    q64 = torch.sigmoid(Z64) if C == 1 else torch.softmax(Z64.reshape(B, T, C), -1).reshape(B, -1)
    (q64 * G.double()).sum().backward()
    Q, dZ = torch.empty_like(Z), torch.empty_like(Z)
    engine.class_probs(Z, C, Q)
    engine.class_probs_bwd(Q, G, C, dZ)
    torch.testing.assert_close(Q.double(), q64.detach(), rtol=1e-5, atol=1e-7)
    torch.testing.assert_close(dZ.double(), Z64.grad, rtol=1e-4, atol=1e-5)


def test_all_targets_masked_gives_zero_loss_and_gradient():
    P, Y, w, tw = _bce_inputs(257, 5, seed=1)
    Y.fill_(float("nan"))
    loss, dP = torch.full((1,), 7.0, device="cuda"), torch.full_like(P, 7.0)
    engine.bce_loss(P, Y, w, tw, loss, dP)
    assert float(loss) == 0.0 and not dP.any()
    Z, K, w, tw = _ce_inputs(257, 5, 3, seed=2)
    K.fill_(float("nan"))
    loss, dP = torch.full((1,), 7.0, device="cuda"), torch.full_like(Z, 7.0)
    engine.ce_loss(Z, K, w, tw, loss, dP, 3)
    assert float(loss) == 0.0 and not dP.any()


@pytest.mark.parametrize("bad", [4.0, -1.0, 1.5])
def test_out_of_range_class_gives_nan_loss(bad):
    Z, K, w, tw = _ce_inputs(513, 2, 4, seed=3)
    K[100, 1] = bad
    loss, dP = torch.empty(1, device="cuda"), torch.empty_like(Z)
    engine.ce_loss(Z, K, w, tw, loss, dP, 4)
    assert torch.isnan(loss).all()
    K[100, 1] = 3.0
    engine.ce_loss(Z, K, w, tw, loss, dP, 4)
    assert torch.isfinite(loss).all() and torch.isfinite(dP).all()


@pytest.mark.parametrize("kind", ["bce", "ce"])
def test_two_launches_are_bit_identical(kind):
    if kind == "bce":
        P, Y, w, tw = _bce_inputs(10_000, 617, seed=4)
        run = lambda loss, dP: engine.bce_loss(P, Y, w, tw, loss, dP)
    else:
        P, Y, w, tw = _ce_inputs(10_000, 12, 10, seed=5)
        run = lambda loss, dP: engine.ce_loss(P, Y, w, tw, loss, dP, 10)
    outs = []
    for _ in range(2):
        loss, dP = torch.empty(1, device="cuda"), torch.empty_like(P)
        run(loss, dP)
        outs.append((loss, dP))
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])


def test_c2_bf16_step_with_bce_head_replays_new_batches_as_one_cuda_graph():
    """10 k molecules (C2), bf16 BondMessagePassing, mean aggregation, batch norm, a 2-layer FFN with a 12-task BCE head: the
    graph replays a NEW batch of the same signature (new features and targets) and equals an eager step on it."""
    from chemprop_b200.data import BatchMolGraph, make_molecules
    from chemprop_b200.graph import CudaGraphStep
    from chemprop_b200.nn import BondMessagePassing, EngineBinaryClassificationFFN, EngineMPNN

    torch.manual_seed(0)
    n = 10_000
    mgs = make_molecules(n, seed=3, mean_atoms=25.0)
    head = EngineBinaryClassificationFFN(n_tasks=12, input_dim=300, hidden_dim=300, n_layers=2,
                                         task_weights=torch.linspace(0.5, 2.0, 12))
    model = EngineMPNN(BondMessagePassing(precision="bf16"), predictor=head, batch_norm=True).cuda().train()
    for p in model.parameters():
        p.grad = torch.zeros_like(p)
    gen = torch.Generator().manual_seed(1)

    def targets():
        Y = (torch.rand(n, 12, generator=gen) < 0.3).float()
        Y[torch.rand(n, 12, generator=gen) < 0.2] = float("nan")               # Tox21-style missing labels
        return Y.cuda()

    Y, w = targets(), (torch.rand(n, generator=gen) + 0.5).cuda()

    def fn(b):
        for p in model.parameters():
            p.grad.zero_()
        loss = model.training_loss(b, Y, w)
        loss.backward()
        return loss

    step = CudaGraphStep(fn)
    a = BatchMolGraph(mgs)
    a.to("cuda")
    step(a)
    b = BatchMolGraph(mgs)
    b.V = b.V * 0.5 + 0.1                                                      # new features, same topology
    b.to("cuda")
    Y.copy_(targets())
    bn_state = {k: v.clone() for k, v in model.bn.state_dict().items()}
    loss_g = step(b).clone()
    grads_g = {k: p.grad.clone() for k, p in model.named_parameters()}
    assert step.captures == 1 and step.replays == 2
    model.bn.load_state_dict(bn_state)
    loss_e = fn(b)
    assert torch.isfinite(loss_e)
    torch.testing.assert_close(loss_g, loss_e, rtol=1e-5, atol=1e-6)
    for k, p in model.named_parameters():
        torch.testing.assert_close(grads_g[k], p.grad, rtol=1e-4, atol=1e-6, msg=k)
    model.eval()
    with torch.no_grad():
        probs = model(b)
    assert tuple(probs.shape) == (n, 12) and bool(((probs >= 0) & (probs <= 1)).all())
