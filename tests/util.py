"""Shared helpers for the test-suite (golden loading, module construction)."""
from __future__ import annotations

import glob
import json
import os

import numpy as np
import torch

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def golden_names(prefix: str = "", mab: bool = False) -> list[str]:
    """Golden cases of Bond / AtomMessagePassing (default) or of the mol-atom-bond variants (`mab=True`)."""
    names = sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(GOLDEN_DIR, "*.npz")))
    return [n for n in names if n != "collate_fixture" and not n.startswith("fixture_") and n.startswith(prefix)
            and n.startswith("mab_") == mab]


def load_golden(name: str) -> dict:
    z = np.load(os.path.join(GOLDEN_DIR, f"{name}.npz"), allow_pickle=False)
    d = {k: z[k] for k in z.files}
    if "config" in d:
        d["config"] = json.loads(str(d["config"]))
    return d


def params_of(g: dict, dtype=torch.float32, device="cpu") -> dict:
    out = {}
    for k, v in g.items():
        if k.startswith("param."):
            out[k[len("param."):]] = torch.from_numpy(v).to(device=device, dtype=dtype)
    return out


def oracle_forward(g: dict, dtype=torch.float32, requires_grad: bool = False):
    """Run oracle/restatement.py on a golden case's inputs; returns (H_v, params dict)."""
    from oracle import restatement as R

    cfg = g["config"]
    P = params_of(g, dtype)
    if requires_grad:
        for p in P.values():
            p.requires_grad_(True)
    V = torch.from_numpy(g["V"]).to(dtype)
    E = torch.from_numpy(g["E"]).to(dtype)
    if cfg.get("graph_transform"):
        V = (V - torch.from_numpy(g["gt_V_mean"]).to(dtype)) / torch.from_numpy(g["gt_V_scale"]).to(dtype)
        E = (E - torch.from_numpy(g["gt_E_mean"]).to(dtype)) / torch.from_numpy(g["gt_E_scale"]).to(dtype)
    ei = torch.from_numpy(g["edge_index"])
    rev = torch.from_numpy(g["rev_edge_index"])
    V_d = torch.from_numpy(g["V_d"]).to(dtype) if "V_d" in g else None
    H = R.message_passing_forward(
        cfg["kind"], V, E, ei, rev, P["W_i.weight"], P.get("W_i.bias"), P["W_h.weight"], P.get("W_h.bias"),
        P["W_o.weight"], P.get("W_o.bias"), cfg["depth"], activation_name(cfg),
        cfg.get("undirected", False), V_d, P.get("W_d.weight"), P.get("W_d.bias"), prelu_weight=P.get("tau.weight"))
    return H, P


def activation_name(cfg: dict) -> str:
    return cfg["activation_module"].lower() if cfg.get("activation_module") else cfg.get("activation", "relu")


def activation_arg(cfg: dict):
    """What the golden case handed to the module constructor: a name, or a module instance."""
    return getattr(torch.nn, cfg["activation_module"])() if cfg.get("activation_module") else cfg.get("activation", "relu")


COMPOSED_GOLDENS = ("bond_d3_prelu", "atom_d3_prelu_bias", "bond_d3_selu", "bond_d3_softplus", "atom_d3_undirected",
                    "atom_d4_undir_elu", "bond_d3_undir_prelu", "atom_d3_noedges_prelu")


def build_engine_module(g: dict, device="cuda", precision="fp32", fused=True):
    """chemprop_b200 module holding the golden case's weights."""
    from chemprop_b200.nn import AtomMessagePassing, BondMessagePassing, GraphTransform, ScaleTransform

    cfg = g["config"]
    gt = None
    if cfg.get("graph_transform"):
        gt = GraphTransform(ScaleTransform(g["gt_V_mean"][0], g["gt_V_scale"][0]),
                            ScaleTransform(g["gt_E_mean"][0], g["gt_E_scale"][0]))
    cls = BondMessagePassing if cfg["kind"] == "bond" else AtomMessagePassing
    mp = cls(d_v=cfg.get("d_v", 72), d_e=cfg.get("d_e", 14), d_h=cfg["d_h"], bias=cfg.get("bias", False),
             depth=cfg["depth"], activation=activation_arg(cfg), undirected=cfg.get("undirected", False),
             dropout=cfg.get("dropout", 0.0), d_vd=cfg.get("d_vd"), graph_transform=gt, precision=precision)
    mp.fused = fused
    mp.load_state_dict({k: v for k, v in params_of(g).items()}, strict=False)
    mp = mp.to(device)
    if gt is not None or cfg.get("eval"):
        mp.eval()
    return mp


def golden_bmg(g: dict, device="cuda"):
    from chemprop_b200.data import BatchMolGraph

    bmg = BatchMolGraph.from_tensors(
        torch.from_numpy(g["V"]), torch.from_numpy(g["E"]), torch.from_numpy(g["edge_index"]),
        torch.from_numpy(g["rev_edge_index"]), torch.from_numpy(g["batch"]), int(g["n_mols"]))
    bmg.to(device)
    return bmg


class RecordingDropout(torch.nn.Dropout):
    """nn.Dropout that remembers the (scaled) masks it applied, in call order."""

    def __init__(self, p):
        super().__init__(p)
        self.masks = []

    def forward(self, x):
        m = torch.nn.functional.dropout(torch.ones_like(x), self.p, self.training)
        self.masks.append(m)
        return x * m


def dropout_mask_for_mask(kind: str, undirected: bool, act: str, device: str, n_mols: int = 12, d_h: int = 32):
    """Training-mode dropout on the composed tier vs the oracle fed with the very masks the run drew (edge-level masks
    mapped from the engine's dst-sorted row order back to the caller's edge order through `perm`).

    An f32 pre-activation within rounding of an activation's kink (ReLU / PReLU at 0) can land on the other side of it
    than its f64 counterpart, and one such element shifts whole gradient rows by its upstream gradient.  So the oracle
    takes the engine's side of the kink at exactly those elements (its pre-activations, recorded in the same order,
    mapped like the masks) -- and every one of them must agree with the oracle's pre-activation to the forward bound."""
    from chemprop_b200.data import BatchMolGraph, make_molecules
    from chemprop_b200.engine import get_layout
    from chemprop_b200.nn import AtomMessagePassing, BondMessagePassing, MeanAggregation
    from oracle import restatement as R

    torch.manual_seed(3)
    bmg = BatchMolGraph(make_molecules(n_mols, seed=4, mean_atoms=10, std_atoms=4, shuffle_edges=True, min_atoms=1))
    ref = BatchMolGraph(make_molecules(n_mols, seed=4, mean_atoms=10, std_atoms=4, shuffle_edges=True, min_atoms=1))
    cls = BondMessagePassing if kind == "bond" else AtomMessagePassing
    depth, d_vd = 3, 4
    mp = cls(d_h=d_h, depth=depth, bias=True, dropout=0.4, activation=act, undirected=undirected, d_vd=d_vd)
    mp.dropout = RecordingDropout(0.4)
    mp.train()
    assert mp.uses_composed_tier()
    V_d = torch.randn(bmg.V.shape[0], d_vd)
    P = {k: v.detach().double().requires_grad_(True) for k, v in mp.state_dict().items()}
    pre = []                                      # the engine's activation inputs: H_0, every depth step, the read-out
    mp.tau.register_forward_pre_hook(lambda mod, args: pre.append(args[0].detach().double().cpu()))
    mp = mp.to(device)
    bmg.to(device)
    H = mp(bmg, V_d.to(device))
    a = MeanAggregation()(H, bmg.batch)
    a.square().sum().backward()
    masks = [m.cpu() for m in mp.dropout.masks]
    assert len(masks) == (depth - 1) + 2 and 0.2 < float((masks[0] == 0).float().mean()) < 0.6
    perm = get_layout(bmg).perm.long().cpu()
    ref_masks = []
    for m in masks[: depth - 1]:                  # edge-level masks were drawn in the internal (dst-sorted) row order
        mm = torch.empty_like(m)
        mm[perm] = m
        ref_masks.append(mm.double())
    ref_masks += [m.double() for m in masks[depth - 1:]]
    assert len(pre) == depth + 1
    for i in range(depth):                        # H_0 and the depth steps are edge-level, in the internal row order
        z = torch.empty_like(pre[i])
        z[perm] = pre[i]
        pre[i] = z
    base_tau = R.activation(act, P.get("tau.weight"))
    kinks = []                                    # per activation call: elements where the oracle follows the engine's side

    def tau(x):
        z = pre[len(kinks)]
        other_side = (x.detach() > 0) != (z > 0)
        kinks.append((int(other_side.sum()), float((x.detach() - z)[other_side].abs().max()) if other_side.any() else 0.0))
        return base_tau(x + torch.where(other_side, z - x.detach(), torch.zeros_like(z)))   # value shift only: d/dx = 1

    H_ref = R.message_passing_forward(kind, ref.V.double(), ref.E.double(), ref.edge_index, ref.rev_edge_index,
                                      P["W_i.weight"], P["W_i.bias"], P["W_h.weight"], P["W_h.bias"], P["W_o.weight"],
                                      P["W_o.bias"], depth, tau, undirected, V_d.double(), P["W_d.weight"], P["W_d.bias"],
                                      dropout_masks=ref_masks)
    R.aggregate(H_ref, ref.batch, "mean").square().sum().backward()
    assert len(kinks) == depth + 1 and max(d for _, d in kinks) <= 1e-5, kinks      # sides differ only within rounding
    assert (H.detach().double().cpu() - H_ref.detach()).abs().max().item() <= 1e-5
    bad = {}
    for k, p in mp.named_parameters():
        g = P[k].grad
        assert p.grad is not None, k
        d = (p.grad.double().cpu() - g).abs()
        tol = 1e-4 * max(1.0, g.abs().max().item())
        if d.max().item() > tol:       # every offending parameter: max error, bound, how many entries and which rows
            bad[k] = (d.max().item(), tol, int((d > tol).sum()), sorted({int(i) for i in (d > tol).nonzero()[:, 0][:8]}))
    assert not bad, (bad, kinks)
    return kinks


def mab_oracle_forward(g: dict, dtype=torch.float32, requires_grad: bool = False):
    """oracle/restatement.mab_forward on a MAB golden case's inputs; returns (H_v | None, H_e | None, params)."""
    from oracle import restatement as R

    cfg = g["config"]
    P = params_of(g, dtype)
    if requires_grad:
        for p in P.values():
            p.requires_grad_(True)
    t = lambda k: torch.from_numpy(g[k]).to(dtype) if k in g else None  # noqa: E731
    H_v, H_e = R.mab_forward(
        cfg["kind"][4:], t("V"), t("E"), torch.from_numpy(g["edge_index"]), torch.from_numpy(g["rev_edge_index"]),
        P["W_i.weight"], P.get("W_i.bias"), P["W_h.weight"], P.get("W_h.bias"), P.get("W_vo.weight"), P.get("W_vo.bias"),
        P.get("W_eo.weight"), P.get("W_eo.bias"), cfg["depth"], activation_name(cfg), cfg.get("undirected", False),
        t("V_d"), P.get("W_vd.weight"), P.get("W_vd.bias"), t("E_d"), P.get("W_ed.weight"), P.get("W_ed.bias"),
        prelu_weight=P.get("tau.weight"), return_vertex=cfg.get("vertex", True), return_edge=cfg.get("edge", True))
    return H_v, H_e, P


def build_mab_module(g: dict, device="cuda"):
    from chemprop_b200.nn import MABAtomMessagePassing, MABBondMessagePassing

    cfg = g["config"]
    cls = MABBondMessagePassing if cfg["kind"] == "mab_bond" else MABAtomMessagePassing
    mp = cls(d_v=cfg.get("d_v", 72), d_e=cfg.get("d_e", 14), d_h=cfg["d_h"], bias=cfg.get("bias", False),
             depth=cfg["depth"], activation=activation_arg(cfg), undirected=cfg.get("undirected", False),
             d_vd=cfg.get("d_vd"), d_ed=cfg.get("d_ed"), return_vertex_embeddings=cfg.get("vertex", True),
             return_edge_embeddings=cfg.get("edge", True))
    mp.load_state_dict(params_of(g), strict=True)      # the reference's state-dict keys, all of them
    return mp.to(device)


def run_mab_case(g: dict, device: str):
    """Module forward + the golden's loss (sum(mean_agg(H_v) * G) + sum(H_e * G_e)) + backward; returns (mp, H_v, H_e)."""
    from chemprop_b200.nn import MeanAggregation

    mp = build_mab_module(g, device)
    bmg = golden_bmg(g, device)
    d = lambda k: torch.from_numpy(g[k]).to(device) if k in g else None  # noqa: E731
    H_v, H_e = mp(bmg, d("V_d"), d("E_d"))
    loss = 0.0
    if H_v is not None:
        loss = loss + (MeanAggregation()(H_v, bmg.batch) * d("G")).sum()
    if H_e is not None:
        loss = loss + (H_e * d("G_e")).sum()
    loss.backward()
    return mp, H_v, H_e


def check_mab_case(g: dict, mp, H_v, H_e, atol: float, grad_rtol: float = 1e-4):
    cfg = g["config"]
    assert (H_v is None) == (not cfg.get("vertex", True)) and (H_e is None) == (not cfg.get("edge", True))
    if H_v is not None:
        np.testing.assert_allclose(H_v.detach().cpu().numpy(), g["H_v"], rtol=1e-5, atol=atol)
    if H_e is not None:
        assert tuple(H_e.shape) == g["H_e"].shape
        np.testing.assert_allclose(H_e.detach().cpu().numpy(), g["H_e"], rtol=1e-5, atol=atol)   # caller's edge order
    grads = {k: p.grad for k, p in mp.named_parameters()}
    n = 0
    for k, v in g.items():
        if k.startswith("grad."):
            got = grads[k[len("grad."):]]
            assert got is not None, k
            np.testing.assert_allclose(got.cpu().numpy(), v, rtol=grad_rtol, atol=10 * atol, err_msg=k)
            n += 1
    assert n >= 3


def check_attentive(device: str, atol: float = 2e-6):
    """AttentiveAggregation against the reference's fixture (tests/golden/fixture_attentive.npz): output and the gradients
    w.r.t. the atom states and the logit layer."""
    from chemprop_b200.nn import AttentiveAggregation

    g = load_golden("fixture_attentive")
    agg = AttentiveAggregation(output_size=g["H"].shape[1])
    agg.load_state_dict({"W.weight": torch.from_numpy(g["param.W.weight"]), "W.bias": torch.from_numpy(g["param.W.bias"])})
    agg = agg.to(device)
    H = torch.from_numpy(g["H"]).to(device).requires_grad_(True)
    out = agg(H, torch.from_numpy(g["batch"]).to(device))
    np.testing.assert_allclose(out.detach().cpu().numpy(), g["out"], rtol=1e-5, atol=atol)
    (out * torch.from_numpy(g["G"]).to(device)).sum().backward()
    np.testing.assert_allclose(H.grad.cpu().numpy(), g["grad.H"], rtol=1e-4, atol=atol)
    np.testing.assert_allclose(agg.W.weight.grad.cpu().numpy(), g["grad.W.weight"], rtol=1e-4, atol=atol)
    np.testing.assert_allclose(agg.W.bias.grad.cpu().numpy(), g["grad.W.bias"], rtol=1e-4, atol=atol)
    assert agg.hparams == {"dim": 0, "cls": AttentiveAggregation, "output_size": g["H"].shape[1]}


def fused_dropout_vs_oracle(device: str, depth: int = 3, bias: bool = True, d_h: int = 64, n_mols: int = 60, p: float = 0.3):
    """Training-mode dropout on the fused bf16 / ReLU path (engine.dropout_fused_ok) vs the oracle fed with the very keep
    masks the run drew (mapped from the engine's row order to the caller's edge order): hidden states within the bf16
    bound, gradients within a bound that a wrong 1 / (1 - p) factor anywhere in the mirror would break."""
    from chemprop_b200.data import BatchMolGraph, make_molecules
    from chemprop_b200.engine import get_layout
    from chemprop_b200.nn import BondMessagePassing, MeanAggregation
    from oracle import restatement as R

    torch.manual_seed(11)
    mgs = make_molecules(n_mols, seed=6, mean_atoms=12, std_atoms=4, shuffle_edges=True)
    bmg, ref = BatchMolGraph(mgs), BatchMolGraph(mgs)
    mp = BondMessagePassing(d_h=d_h, depth=depth, bias=bias, dropout=p, precision="bf16")
    P = {k: v.detach().double().requires_grad_(True) for k, v in mp.state_dict().items()}
    masks = []

    def mask_fn(like):
        m = torch.empty_like(like).bernoulli_(1.0 - p)
        masks.append(m)
        return m

    mp._mask_fn = mask_fn
    mp = mp.to(device).train()
    bmg.to(device)
    lay = get_layout(bmg)
    assert not mp.uses_composed_tier(lay) and mp.uses_composed_tier()          # monolithic for THIS batch
    H = mp(bmg)
    MeanAggregation()(H, bmg.batch).float().square().sum().backward()
    assert len(masks) == depth and all(m.dtype == torch.bfloat16 for m in masks)          # depth - 1 edge sites + read-out
    nE, nV, perm = ref.E.shape[0], ref.V.shape[0], lay.perm.long().cpu()
    keep = 1.0 - p
    ref_masks = []
    for m in masks[:-1]:
        mm = torch.empty((nE, d_h), dtype=torch.float64)
        mm[perm] = m[:nE, :d_h].double().cpu() / keep
        ref_masks.append(mm)
    ref_masks.append(masks[-1][:nV, :d_h].double().cpu() / keep)
    H_ref = R.message_passing_forward("bond", ref.V.double(), ref.E.double(), ref.edge_index, ref.rev_edge_index,
                                      P["W_i.weight"], P.get("W_i.bias"), P["W_h.weight"], P.get("W_h.bias"), P["W_o.weight"],
                                      P["W_o.bias"], depth, "relu", False, dropout_masks=ref_masks)
    R.aggregate(H_ref, ref.batch, "mean").square().sum().backward()
    frac0 = float((H_ref == 0).double().mean())
    assert frac0 > p * 0.8                                                      # dropout really happened
    tol = 1e-2 * max(1.0, H_ref.detach().abs().max().item())
    assert (H.detach().double().cpu() - H_ref.detach()).abs().max().item() <= tol
    for k, prm in mp.named_parameters():
        g = P[k].grad if P[k].grad is not None else torch.zeros_like(P[k])
        got = prm.grad.double().cpu()
        fro = float((got - g).norm() / max(1e-9, g.norm()))
        assert fro <= 0.12, (k, fro)              # a missing / doubled 1/(1-p) = 1.43 would show as >= 0.3


def check_constrainer(device: str, atol: float = 2e-6):
    """ConstrainerFFN against the reference's fixture (tests/golden/fixture_constrainer.npz): adjusted predictions, the
    constraint itself, and the gradients w.r.t. fingerprints, predictions and the MLP."""
    from chemprop_b200.nn import ConstrainerFFN

    g = load_golden("fixture_constrainer")
    mod = ConstrainerFFN(n_constraints=2, fp_dim=20, hidden_dim=16, n_layers=2, activation="tanh")
    mod.load_state_dict({k[len("param."):]: torch.from_numpy(v) for k, v in g.items() if k.startswith("param.")})   # strict
    mod = mod.to(device)
    fp = torch.from_numpy(g["fp"]).to(device).requires_grad_(True)
    preds = torch.from_numpy(g["preds"]).to(device).requires_grad_(True)
    batch, cons = torch.from_numpy(g["batch"]).to(device), torch.from_numpy(g["constraints"]).to(device)
    out = mod(fp, preds, batch, cons)
    np.testing.assert_allclose(out.detach().cpu().numpy(), g["out"], rtol=1e-5, atol=atol)
    sums = torch.zeros(cons.shape, device=device).index_add_(0, batch, out.detach())
    assert (sums[:, [0, 2]] - cons[:, [0, 2]]).abs().max().item() <= 1e-4           # the constrained columns sum to the constraint
    (out * torch.from_numpy(g["G"]).to(device)).sum().backward()
    np.testing.assert_allclose(fp.grad.cpu().numpy(), g["grad.fp"], rtol=1e-4, atol=atol)
    np.testing.assert_allclose(preds.grad.cpu().numpy(), g["grad.preds"], rtol=1e-4, atol=atol)
    for k, p in mod.named_parameters():
        np.testing.assert_allclose(p.grad.cpu().numpy(), g["grad." + k], rtol=1e-4, atol=atol, err_msg=k)
    assert mod.hparams["cls"] is ConstrainerFFN and mod.hparams["n_constraints"] == 2


def check_constrainer_empty_trailing(device: str, atol: float = 2e-6):
    """ffn.py:123 sizes by `constraints.shape[0]`: a batch whose LAST molecules own no row (bond constrainer on 'C' or
    '[Na+]': no bonds) must work, and an all-unconstrained column set is the identity.  Against oracle.restatement.constrain
    (the reference's op sequence)."""
    from chemprop_b200.nn import ConstrainerFFN
    from oracle import restatement as R

    torch.manual_seed(4)
    mod = ConstrainerFFN(n_constraints=2, fp_dim=12, hidden_dim=8, n_layers=1, activation="relu")
    ref_k = lambda fp: mod.to("cpu").ffn(fp)
    batch = torch.tensor([0, 0, 0, 2, 2, 3, 3, 3, 3])          # 6 molecules: 1, 4 and 5 own no row
    fp, preds = torch.randn(9, 12), torch.randn(9, 2)
    cons = torch.randn(6, 2)
    want = R.constrain(ref_k(fp), preds, batch, cons).detach()
    mod = mod.to(device)
    out = mod(fp.to(device), preds.to(device), batch.to(device), cons.to(device))
    np.testing.assert_allclose(out.detach().cpu().numpy(), want.numpy(), rtol=1e-5, atol=atol)
    none = torch.full((6, 2), float("nan"))
    out2 = mod(fp.to(device), preds.to(device), batch.to(device), none.to(device))
    assert torch.equal(out2.cpu(), preds)
    import pytest as _pt
    from chemprop_b200 import DmpnnError
    with _pt.raises(DmpnnError):
        mod(fp.to(device), preds.to(device), batch.to(device), cons[:3].to(device))       # index 3 >= 3 rows


def check_mpnn_head(device: str, rtol: float = 2e-4, atol: float = 2e-6, graph: bool = False):
    """EngineMPNN.training_loss (encoder -> aggregation -> batch norm -> FFN -> masked / weighted MSE, every step on libdmpnn)
    against the reference's own `MPNN.training_step` (tests/golden/fixture_mpnn_head.npz: loss, every gradient, the batch-norm
    running statistics after the step, eval-mode predictions).  `graph`: the step runs as a captured CUDA graph."""
    import chemprop_b200.nn as N

    g = load_golden("fixture_mpnn_head")
    model = N.EngineMPNN(N.BondMessagePassing(d_h=40, depth=3), N.MeanAggregation(),
                         N.EngineRegressionFFN(n_tasks=2, input_dim=40, hidden_dim=24, n_layers=2), batch_norm=True)
    state = {k[len("param."):]: torch.from_numpy(np.asarray(v)) for k, v in g.items() if k.startswith("param.")}
    missing = model.load_state_dict({k: v for k, v in state.items() if not k.endswith(("total_loss", "num_samples"))}, strict=True)
    assert not missing.missing_keys and not missing.unexpected_keys
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
        loss = step(bmg)                    # warm-up (2 eager steps) + capture + first replay: 4 updates of the running statistics
        # one more replay from the fixture's initial running statistics: this is the step the reference took
        model.bn.running_mean.copy_(rm0); model.bn.running_var.copy_(rv0); model.bn.num_batches_tracked.copy_(nb0)
        loss = step(bmg).clone()
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
        np.testing.assert_allclose(model(bmg).cpu().numpy(), g["preds_eval"], rtol=rtol, atol=1e-5)


def full_size_checks(kind: str, n_mols: int, device: str, gen_kw: dict | None = None, module_kw: dict | None = None,
                     tile_tags: set | None = None, grad_tol: float = 6e-2, oracle: bool = True) -> dict:
    """The benchmarked tier (bf16, fused depth step) on ONE batch of a BASELINE configuration's size, held to
      (1) the oracle (f32 CPU restatement) -- hidden states, aggregates and every weight gradient -- at the bounds of the
          medium-size parity tests;
    and to the size-independent properties of the path:
      (2) reproducibility: the same batch twice gives bit-identical outputs and gradients (no float atomics anywhere);
      (3) linearity of the hand-written mirror in the upstream gradient: doubling it doubles every weight gradient EXACTLY
          (a power of two commutes with every rounding on the way);
      (4) a checksum of checksums: the column sums of the per-molecule sums equal the column sums of the atom states;
      (5) molecule-order invariance: the loader's tile-packing order and the sampler's order give the same per-molecule
          aggregates (molecules never interact: chemprop/data/collate.py:48-56).
    Used on the GPU (tests/test_gpu_zzz_full_size.py) and, at a small size through the emulated kernel wrappers, on the CPU
    (tests/test_host_logic.py) so that the checks themselves are exercised without hardware.  Returns the measured figures."""
    from chemprop_b200 import engine
    from chemprop_b200.data import BatchMolGraph, make_cgr_graphs, make_molecules, tile_packing_order_of
    from chemprop_b200.nn import AtomMessagePassing, BondMessagePassing, MeanAggregation, SumAggregation
    from oracle import restatement as R

    torch.manual_seed(0)
    gen_kw = dict(gen_kw or {})
    cgr = gen_kw.pop("cgr", False)
    pool = gen_kw.pop("pool", n_mols)         # bench.py draws its resident batch as the first n_mols molecules of a larger pool
    mgs = (make_cgr_graphs if cgr else make_molecules)(pool, **gen_kw)[:n_mols]
    order = tile_packing_order_of(mgs)
    packed = [mgs[i] for i in order]
    d_v, d_e = mgs[0].V.shape[1], mgs[0].E.shape[1]
    cls = BondMessagePassing if kind == "bond" else AtomMessagePassing
    kw = dict(d_v=d_v, d_e=d_e, d_h=300, depth=3, precision="bf16")
    kw.update(module_kw or {})
    mp = cls(**kw)
    host = BatchMolGraph(packed)
    P = {k: v.detach().clone().requires_grad_(True) for k, v in mp.state_dict().items()}
    if oracle:
        nt = torch.get_num_threads()
        torch.set_num_threads(min(nt, 16))    # torch's CPU scatter / index kernels regress beyond a few dozen threads (bench.py)
        try:
            H_ref = R.message_passing_forward(kind, host.V, host.E, host.edge_index, host.rev_edge_index, P["W_i.weight"],
                                              P.get("W_i.bias"), P["W_h.weight"], P.get("W_h.bias"), P["W_o.weight"],
                                              P["W_o.bias"], kw["depth"])
            a_ref = R.aggregate(H_ref, host.batch, "mean")
            G = a_ref.detach().clone() / n_mols   # upstream gradient of 0.5 * mean-over-molecules |agg|^2, held fixed (see (3))
            (a_ref * G).sum().backward()
        finally:
            torch.set_num_threads(nt)
        H_ref, a_ref = H_ref.detach(), a_ref.detach()
    else:                                     # properties only (sizes the CPU oracle needs minutes for)
        G = torch.randn(n_mols, kw["d_h"]) / n_mols

    mp = mp.to(device)
    Gd = G.to(device)

    def run(batch_mgs, scale=1.0):
        bmg = BatchMolGraph(batch_mgs)
        bmg.to(device)
        mp.zero_grad(set_to_none=True)
        engine.STEP_EVENTS = [] if str(device) != "cpu" else None          # CUDA events: which depth-step kernels ran
        try:
            H = mp(bmg)
            tags = {t for t, _, _ in (engine.STEP_EVENTS or [])}
        finally:
            engine.STEP_EVENTS = None
        a = MeanAggregation()(H, bmg.batch)
        s = SumAggregation()(H, bmg.batch)
        return bmg, H, a, s, tags

    bmg, H, a, s, tags = run(packed)
    if tile_tags is not None and str(device) != "cpu":
        assert tags == tile_tags, tags                                      # the fused kernel ran every depth step
    (a * Gd).sum().backward()
    grads = {k: p.grad.detach().clone() for k, p in mp.named_parameters()}
    out = {"tiles": bmg._meta_host[0], "rows": int(bmg.E.shape[0]), "atoms": int(bmg.V.shape[0])}

    # (1) the oracle
    scale = 1.0
    if oracle:
        scale = max(1.0, H_ref.abs().max().item())
        out["err_H"] = (H.detach().float().cpu() - H_ref).abs().max().item()
        out["err_agg"] = (a.detach().float().cpu() - a_ref).abs().max().item()
        assert out["err_H"] <= 1e-2 * scale and out["err_agg"] <= 1e-2 * scale, out
        out["err_grad"] = {}
        for k, g in grads.items():
            ref = P[k].grad
            out["err_grad"][k] = ((g.float().cpu() - ref).abs().max() / ref.abs().max().clamp_min(1e-12)).item()
            assert out["err_grad"][k] <= grad_tol, (k, out["err_grad"][k])   # bf16 storage flips ReLU derivatives near zero:
                                                                              # noise that averages out with the batch size
    else:
        scale = max(1.0, H.detach().float().abs().max().item())

    # (2) reproducibility, bit for bit
    _, H2, a2, s2, _ = run(packed)
    (a2 * Gd).sum().backward()
    assert torch.equal(H2, H) and torch.equal(a2, a) and torch.equal(s2, s)
    for k, p in mp.named_parameters():
        assert torch.equal(p.grad, grads[k]), ("not reproducible", k)

    # (3) linearity of the mirror: upstream gradient x 2 -> every weight gradient x 2, exactly
    _, H3, a3, _, _ = run(packed)
    (a3 * (2.0 * Gd)).sum().backward()
    for k, p in mp.named_parameters():
        assert torch.equal(p.grad, 2.0 * grads[k]), ("mirror not linear in the upstream gradient", k)

    # (4) checksum of checksums (f32 sums in different orders: relative to the sum of magnitudes)
    Hf = H.detach().float()
    lhs, rhs = s.detach().float().sum(0).cpu(), Hf.sum(0).cpu()
    mag = Hf.abs().sum(0).cpu().clamp_min(1e-6)
    out["checksum_rel"] = ((lhs - rhs).abs() / mag).max().item()
    assert out["checksum_rel"] <= 1e-4, out["checksum_rel"]

    # (5) molecule order: molecule order[j] sits at position j of the packed batch
    _, _, a_plain, _, _ = run(mgs)
    idx = torch.as_tensor(np.asarray(order), dtype=torch.long, device=a_plain.device)
    out["order_diff"] = (a_plain.detach().float()[idx] - a.detach().float()).abs().max().item()
    assert out["order_diff"] <= 1e-2 * scale, out["order_diff"]
    return out
