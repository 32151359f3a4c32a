"""TEST INFRASTRUCTURE ONLY.  Generates tests/golden/*.npz by running the UNMODIFIED reference
(chemprop v2.3.1 at /root/reference, imported through oracle/ref_shim.py) on small seeded cases.
Run here (the reference cannot travel to the GPU box); the outputs are committed.

    python -m oracle.make_golden

Each .npz holds the inputs (V, E, edge_index, rev_edge_index, batch, n_mols, optional V_d), the
module's state_dict, its config, and the reference results: H_v = mp(bmg[, V_d]), the
Mean/Sum/Norm aggregations of H_v, and the weight gradients of loss = sum(mean_agg(H_v) * G).
"""
from __future__ import annotations

import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle.ref_shim import REFERENCE_ROOT, import_reference  # noqa: E402

GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")

# name -> config.  graph: how the batch is made (see make_batch)
CASES = {
    "bond_d3_relu":        dict(kind="bond", depth=3, d_h=64, graph="mols6"),
    "bond_d1":             dict(kind="bond", depth=1, d_h=48, graph="mols6"),
    "bond_d2_bias":        dict(kind="bond", depth=2, d_h=64, bias=True, graph="mols6"),
    "bond_d6":             dict(kind="bond", depth=6, d_h=40, graph="mols6"),
    "bond_d3_undirected":  dict(kind="bond", depth=3, d_h=64, undirected=True, graph="mols6"),
    "bond_d3_leakyrelu":   dict(kind="bond", depth=3, d_h=64, activation="leakyrelu", graph="mols6"),
    "bond_d3_tanh":        dict(kind="bond", depth=3, d_h=64, activation="tanh", bias=True, graph="mols6"),
    "bond_d3_elu":         dict(kind="bond", depth=3, d_h=64, activation="elu", graph="mols6"),
    "bond_d3_shuffled":    dict(kind="bond", depth=3, d_h=64, graph="mols6_shuffled"),
    "bond_d3_chain":       dict(kind="bond", depth=3, d_h=300, graph="chain5"),
    "bond_d3_noedges":     dict(kind="bond", depth=3, d_h=32, graph="single_atoms4"),
    "bond_d3_mixed":       dict(kind="bond", depth=3, d_h=64, graph="mixed"),
    "bond_d3_vd":          dict(kind="bond", depth=3, d_h=64, d_vd=5, graph="mols6"),
    "bond_d3_h300":        dict(kind="bond", depth=3, d_h=300, graph="mols6"),
    "bond_d3_big_mol":     dict(kind="bond", depth=3, d_h=32, graph="bigmol"),
    "bond_d3_trained":     dict(kind="bond", depth=3, d_h=300, graph="mols6", checkpoint="example_model_v2_regression_mol.pt"),
    "bond_d3_graphtf":     dict(kind="bond", depth=3, d_h=32, graph="mols6", graph_transform=True),
    "atom_d3_relu":        dict(kind="atom", depth=3, d_h=64, graph="mols6"),
    "atom_d1":             dict(kind="atom", depth=1, d_h=48, graph="mols6"),
    "atom_d3_bias_tanh":   dict(kind="atom", depth=3, d_h=64, bias=True, activation="tanh", graph="mols6"),
    "atom_d3_shuffled":    dict(kind="atom", depth=3, d_h=64, graph="mols6_shuffled"),
    "atom_d3_chain":       dict(kind="atom", depth=3, d_h=64, graph="chain5"),
    "atom_d3_noedges":     dict(kind="atom", depth=3, d_h=32, graph="single_atoms4"),
    "atom_d3_cgr":         dict(kind="atom", depth=3, d_h=64, d_v=106, d_e=28, graph="cgr3"),
    "atom_d4_mixed":       dict(kind="atom", depth=4, d_h=64, graph="mixed"),
    # composed-tier configurations (chemprop_b200/composed.py): activations the kernels do not fuse, AtomMP undirected
    "bond_d3_prelu":       dict(kind="bond", depth=3, d_h=64, activation="prelu", graph="mols6"),
    "atom_d3_prelu_bias":  dict(kind="atom", depth=3, d_h=64, activation="prelu", bias=True, graph="mols6"),
    "bond_d3_selu":        dict(kind="bond", depth=3, d_h=64, activation="selu", graph="mols6"),
    "bond_d3_softplus":    dict(kind="bond", depth=3, d_h=48, activation_module="Softplus", bias=True, graph="mols6_shuffled"),
    "atom_d3_undirected":  dict(kind="atom", depth=3, d_h=64, undirected=True, graph="mols6"),
    "atom_d4_undir_elu":   dict(kind="atom", depth=4, d_h=40, undirected=True, activation="elu", bias=True, graph="mixed"),
    "bond_d3_undir_prelu": dict(kind="bond", depth=3, d_h=64, undirected=True, activation="prelu", graph="mols6_shuffled"),
    "atom_d3_noedges_prelu": dict(kind="atom", depth=3, d_h=32, activation="prelu", graph="single_atoms4"),
    "bond_d3_dropout_eval": dict(kind="bond", depth=3, d_h=64, dropout=0.3, eval=True, graph="mols6"),
    # mol-atom-bond variants (chemprop/nn/message_passing/mol_atom_bond.py): vertex AND per-edge embeddings
    "mab_bond_d3":         dict(kind="mab_bond", depth=3, d_h=64, graph="mols6"),
    "mab_atom_d3_desc":    dict(kind="mab_atom", depth=3, d_h=48, bias=True, d_vd=4, d_ed=3, activation="tanh", graph="mols6_shuffled"),
    "mab_bond_edges_only": dict(kind="mab_bond", depth=3, d_h=40, undirected=True, activation="prelu", vertex=False, graph="mixed"),
    "mab_atom_d2_vertex_only": dict(kind="mab_atom", depth=2, d_h=32, edge=False, graph="mols6"),
    "mab_bond_noedges":    dict(kind="mab_bond", depth=3, d_h=32, graph="single_atoms4"),
    # BASELINE config 1: the reference's own CPU case -- tests/data/regression.csv (SMILES topology through
    # oracle/smiles_topology.py), BondMessagePassing h = 300 depth 3, batch = 50; and all 500 molecules at h = 64
    "config1_regression_b50": dict(kind="bond", depth=3, d_h=300, graph="regression_csv:0:50"),
    "config1_regression_all500": dict(kind="bond", depth=3, d_h=64, graph="regression_csv:0:500"),
}


def make_batch(spec: str, d_v: int, d_e: int, seed: int):
    from chemprop_b200.data.synthetic import make_chain_graph, make_molecule, make_molecules

    rng = np.random.default_rng(seed)
    if spec.startswith("regression_csv:"):
        import csv

        from oracle.smiles_topology import to_molgraph

        _, lo, hi = spec.split(":")
        with open(os.path.join(REFERENCE_ROOT, "tests", "data", "regression.csv")) as f:
            rows = list(csv.DictReader(f))
        return [to_molgraph(r["smiles"], d_v, d_e) for r in rows[int(lo):int(hi)]]
    if spec == "mols6":
        return make_molecules(6, seed=seed, mean_atoms=12, std_atoms=5, d_v=d_v, d_e=d_e)
    if spec == "mols6_shuffled":
        return make_molecules(6, seed=seed, mean_atoms=12, std_atoms=5, d_v=d_v, d_e=d_e, shuffle_edges=True)
    if spec == "chain5":
        return [make_chain_graph(5, d_v, d_e)]
    if spec == "single_atoms4":
        return [make_molecule(rng, 1, d_v, d_e) for _ in range(4)]
    if spec == "mixed":
        sizes = [1, 7, 1, 2, 15, 1, 1, 30, 3]
        return [make_molecule(rng, n, d_v, d_e) for n in sizes]
    if spec == "bigmol":  # one molecule with > 128 directed edges (oversized tile) between small ones
        return [make_molecule(rng, 5, d_v, d_e), make_molecule(rng, 90, d_v, d_e), make_molecule(rng, 8, d_v, d_e)]
    if spec == "cgr3":
        return make_molecules(3, seed=seed, mean_atoms=40, std_atoms=8, min_atoms=20, max_atoms=70, d_v=d_v, d_e=d_e,
                              ring_frac=0.03)
    raise KeyError(spec)


def load_checkpoint_state(path: str) -> dict:
    """Tensors of a reference checkpoint (needs the imported reference for unpickling hparams)."""
    import pickle
    import types

    class _Anything(dict):  # stands in for classes of packages that are not installed (lightning.fabric ...)
        def __init__(self, *a, **k):
            pass

        def __setstate__(self, state):
            pass

        def __call__(self, *a, **k):
            return self

    class _Unpickler(pickle.Unpickler):
        def find_class(self, module, name):
            try:
                return super().find_class(module, name)
            except Exception:
                return type(name, (_Anything,), {})

    pm = types.ModuleType("permissive_pickle")
    pm.__dict__.update(pickle.__dict__)
    pm.Unpickler = _Unpickler
    d = torch.load(path, map_location="cpu", weights_only=False, pickle_module=pm)
    return {k[len("message_passing."):]: v for k, v in d["state_dict"].items() if k.startswith("message_passing.")}


def run_case(name: str, cfg: dict, seed: int) -> dict:
    import_reference()
    from chemprop.data import BatchMolGraph
    from chemprop.data.molgraph import MolGraph
    from chemprop.nn import (AtomMessagePassing, BondMessagePassing, MeanAggregation, NormAggregation,
                             SumAggregation)
    from chemprop.nn.transforms import GraphTransform, ScaleTransform

    d_v, d_e, d_h = cfg.get("d_v", 72), cfg.get("d_e", 14), cfg["d_h"]
    mgs = make_batch(cfg["graph"], d_v, d_e, seed)
    ref_mgs = [MolGraph(m.V, m.E, m.edge_index, m.rev_edge_index) for m in mgs]
    bmg = BatchMolGraph(ref_mgs)
    torch.manual_seed(seed)
    gt = None
    rng = np.random.default_rng(seed + 1)
    if cfg.get("graph_transform"):
        gt = GraphTransform(ScaleTransform(rng.normal(0, 0.2, d_v), rng.uniform(0.5, 2.0, d_v)),
                            ScaleTransform(rng.normal(0, 0.2, d_e), rng.uniform(0.5, 2.0, d_e)))
    cls = BondMessagePassing if cfg["kind"] == "bond" else AtomMessagePassing
    activation = getattr(torch.nn, cfg["activation_module"])() if cfg.get("activation_module") else cfg.get("activation", "relu")
    mp = cls(d_v=d_v, d_e=d_e, d_h=d_h, bias=cfg.get("bias", False), depth=cfg["depth"],
             activation=activation, undirected=cfg.get("undirected", False), dropout=cfg.get("dropout", 0.0),
             d_vd=cfg.get("d_vd"), graph_transform=gt)
    if cfg.get("checkpoint"):
        sd = load_checkpoint_state(os.path.join(REFERENCE_ROOT, "tests", "data", cfg["checkpoint"]))
        mp.load_state_dict(sd)
    if gt is not None or cfg.get("eval"):
        mp.eval()  # transforms act in eval mode only (transforms.py:66-67); dropout is the identity
    V_d = None
    if cfg.get("d_vd"):
        V_d = torch.from_numpy(rng.normal(size=(bmg.V.shape[0], cfg["d_vd"])).astype(np.float32))
    before = [t.clone() for t in (bmg.V, bmg.E, bmg.edge_index, bmg.rev_edge_index, bmg.batch)]
    H_v = mp(bmg, V_d)
    for a, b in zip(before, (bmg.V, bmg.E, bmg.edge_index, bmg.rev_edge_index, bmg.batch)):
        assert torch.equal(a, b), "reference mutated its input"
    aggs = {}
    for nm, agg in (("mean", MeanAggregation()), ("sum", SumAggregation()), ("norm", NormAggregation())):
        aggs[nm] = agg(H_v, bmg.batch)
    G = torch.from_numpy(rng.normal(size=tuple(aggs["mean"].shape)).astype(np.float32))
    loss = (aggs["mean"] * G).sum()
    loss.backward()
    out = dict(
        V=bmg.V.numpy(), E=bmg.E.numpy(), edge_index=bmg.edge_index.numpy(),
        rev_edge_index=bmg.rev_edge_index.numpy(), batch=bmg.batch.numpy(), n_mols=np.int64(len(bmg)),
        H_v=H_v.detach().numpy(), agg_mean=aggs["mean"].detach().numpy(), agg_sum=aggs["sum"].detach().numpy(),
        agg_norm=aggs["norm"].detach().numpy(), G=G.numpy(), loss=np.float64(loss.item()),
        config=np.array(json.dumps(cfg)),
    )
    if V_d is not None:
        out["V_d"] = V_d.numpy()
    if gt is not None:
        out["gt_V_mean"], out["gt_V_scale"] = gt.V_transform.mean.numpy(), gt.V_transform.scale.numpy()
        out["gt_E_mean"], out["gt_E_scale"] = gt.E_transform.mean.numpy(), gt.E_transform.scale.numpy()
    for k, v in mp.state_dict().items():
        if k.startswith(("W_i", "W_h", "W_o", "W_d", "tau.")):
            out["param." + k] = v.detach().numpy()
    for k, p in mp.named_parameters():
        if p.grad is not None:
            out["grad." + k] = p.grad.numpy()
    return out


def run_mab_case(name: str, cfg: dict, seed: int) -> dict:
    """MAB variants: outputs (H_v, H_e); loss = sum(mean_agg(H_v) * G) + sum(H_e * G_e)."""
    import_reference()
    from chemprop.data import BatchMolGraph
    from chemprop.data.molgraph import MolGraph
    from chemprop.nn import MeanAggregation
    from chemprop.nn.message_passing import MABAtomMessagePassing, MABBondMessagePassing

    d_v, d_e, d_h = cfg.get("d_v", 72), cfg.get("d_e", 14), cfg["d_h"]
    mgs = make_batch(cfg["graph"], d_v, d_e, seed)
    bmg = BatchMolGraph([MolGraph(m.V, m.E, m.edge_index, m.rev_edge_index) for m in mgs])
    torch.manual_seed(seed)
    rng = np.random.default_rng(seed + 1)
    cls = MABBondMessagePassing if cfg["kind"] == "mab_bond" else MABAtomMessagePassing
    mp = cls(d_v=d_v, d_e=d_e, d_h=d_h, bias=cfg.get("bias", False), depth=cfg["depth"],
             activation=cfg.get("activation", "relu"), undirected=cfg.get("undirected", False), d_vd=cfg.get("d_vd"),
             d_ed=cfg.get("d_ed"), return_vertex_embeddings=cfg.get("vertex", True),
             return_edge_embeddings=cfg.get("edge", True))
    V_d = torch.from_numpy(rng.normal(size=(bmg.V.shape[0], cfg["d_vd"])).astype(np.float32)) if cfg.get("d_vd") else None
    E_d = torch.from_numpy(rng.normal(size=(bmg.E.shape[0], cfg["d_ed"])).astype(np.float32)) if cfg.get("d_ed") else None
    H_v, H_e = mp(bmg, V_d, E_d)
    out = dict(V=bmg.V.numpy(), E=bmg.E.numpy(), edge_index=bmg.edge_index.numpy(),
               rev_edge_index=bmg.rev_edge_index.numpy(), batch=bmg.batch.numpy(), n_mols=np.int64(len(bmg)),
               config=np.array(json.dumps(cfg)))
    loss = torch.zeros(())
    if H_v is not None:
        agg = MeanAggregation()(H_v, bmg.batch)
        G = torch.from_numpy(rng.normal(size=tuple(agg.shape)).astype(np.float32))
        loss = loss + (agg * G).sum()
        out.update(H_v=H_v.detach().numpy(), agg_mean=agg.detach().numpy(), G=G.numpy())
    if H_e is not None:
        G_e = torch.from_numpy(rng.normal(size=tuple(H_e.shape)).astype(np.float32))
        loss = loss + (H_e * G_e).sum()
        out.update(H_e=H_e.detach().numpy(), G_e=G_e.numpy())
    loss.backward()
    out["loss"] = np.float64(loss.item())
    if V_d is not None:
        out["V_d"] = V_d.numpy()
    if E_d is not None:
        out["E_d"] = E_d.numpy()
    for k, v in mp.state_dict().items():
        out["param." + k] = v.detach().numpy()
    for k, p in mp.named_parameters():
        if p.grad is not None:
            out["grad." + k] = p.grad.numpy()
    return out


def collate_case() -> dict:
    """The reference's collate fixture (tests/unit/data/test_dataloader.py:10-84) through the real collate."""
    import_reference()
    from chemprop.data import BatchMolGraph
    from chemprop.data.molgraph import MolGraph

    mg1 = MolGraph(V=np.array([[1.0], [2.0], [3.0]]), E=np.array([[0.5], [1.5], [0.5], [1.5]]),
                   edge_index=np.array([[0, 1, 0, 2], [1, 0, 2, 0]]), rev_edge_index=np.array([1, 0, 3, 2]))
    mg2 = MolGraph(V=np.array([[4.0], [5.0]]), E=np.array([[2.5], [2.5]]), edge_index=np.array([[0, 1], [1, 0]]),
                   rev_edge_index=np.array([1, 0]))
    bmg = BatchMolGraph([mg1, mg2])
    out = dict(V=bmg.V.numpy(), E=bmg.E.numpy(), edge_index=bmg.edge_index.numpy(),
               rev_edge_index=bmg.rev_edge_index.numpy(), batch=bmg.batch.numpy(), n_mols=np.int64(2))
    for i, mg in enumerate((mg1, mg2)):
        out[f"mg{i}.V"], out[f"mg{i}.E"] = mg.V, mg.E
        out[f"mg{i}.edge_index"], out[f"mg{i}.rev_edge_index"] = mg.edge_index, mg.rev_edge_index
    return out


def attentive_case() -> dict:
    """AttentiveAggregation (chemprop/nn/agg.py:116-133) of the real reference on seeded atom states."""
    import_reference()
    from chemprop.nn.agg import AttentiveAggregation

    rng = np.random.default_rng(77)
    sizes = [5, 1, 12, 7, 30, 2]
    batch = torch.from_numpy(np.repeat(np.arange(len(sizes)), sizes))
    H = torch.from_numpy(rng.normal(0, 0.5, size=(sum(sizes), 24)).astype(np.float32)).requires_grad_(True)
    torch.manual_seed(77)
    agg = AttentiveAggregation(output_size=24)
    out = agg(H, batch)
    G = torch.from_numpy(rng.normal(size=tuple(out.shape)).astype(np.float32))
    (out * G).sum().backward()
    return {"H": H.detach().numpy(), "batch": batch.numpy(), "out": out.detach().numpy(), "G": G.numpy(),
            "param.W.weight": agg.W.weight.detach().numpy(), "param.W.bias": agg.W.bias.detach().numpy(),
            "grad.H": H.grad.numpy(), "grad.W.weight": agg.W.weight.grad.numpy(), "grad.W.bias": agg.W.bias.grad.numpy()}


def constrainer_case() -> dict:
    """ConstrainerFFN (chemprop/nn/ffn.py:70-145) of the real reference: 2 constrained columns of 3, 2-layer tanh MLP."""
    import_reference()
    from chemprop.nn.ffn import ConstrainerFFN

    rng = np.random.default_rng(88)
    sizes = [3, 1, 9, 4, 22]
    batch = torch.from_numpy(np.repeat(np.arange(len(sizes)), sizes))
    n = sum(sizes)
    torch.manual_seed(88)
    mod = ConstrainerFFN(n_constraints=2, fp_dim=20, hidden_dim=16, n_layers=2, activation="tanh")
    fp = torch.from_numpy(rng.normal(0, 0.7, size=(n, 20)).astype(np.float32)).requires_grad_(True)
    preds = torch.from_numpy(rng.normal(size=(n, 3)).astype(np.float32)).requires_grad_(True)
    cons = rng.normal(size=(len(sizes), 3)).astype(np.float32)
    cons[:, 1] = np.nan                                              # column 1 is unconstrained (ffn.py:136)
    constraints = torch.from_numpy(cons)
    out = mod(fp, preds, batch, constraints)
    G = torch.from_numpy(rng.normal(size=tuple(out.shape)).astype(np.float32))
    (out * G).sum().backward()
    d = {"fp": fp.detach().numpy(), "preds": preds.detach().numpy(), "batch": batch.numpy(), "constraints": cons,
         "out": out.detach().numpy(), "G": G.numpy(), "grad.fp": fp.grad.numpy(), "grad.preds": preds.grad.numpy()}
    for k, v in mod.state_dict().items():
        d["param." + k] = v.detach().numpy()
    for k, p in mod.named_parameters():
        d["grad." + k] = p.grad.numpy()
    return d


def mpnn_head_case() -> dict:
    """The reference's own training step (chemprop/models/model.py:134-147): `MPNN(BondMessagePassing, MeanAggregation,
    RegressionFFN(n_tasks = 2, 2 layers), batch_norm = True).training_step(batch)` on a seeded batch with a NaN target and
    per-molecule weights: loss, predictions, every gradient, and the batch-norm running statistics after the step."""
    import_reference()
    import chemprop.nn as ref_nn
    from chemprop.data import BatchMolGraph as RefBMG
    from chemprop.data.molgraph import MolGraph as RefMG
    from chemprop.models import MPNN

    from chemprop_b200.data.synthetic import make_molecules

    rng = np.random.default_rng(97)
    torch.manual_seed(97)
    mgs = make_molecules(14, seed=97, mean_atoms=9, std_atoms=3, min_atoms=1)
    bmg = RefBMG([RefMG(*m) for m in mgs])
    mp = ref_nn.BondMessagePassing(d_h=40, depth=3)
    model = MPNN(mp, ref_nn.MeanAggregation(), ref_nn.RegressionFFN(n_tasks=2, input_dim=40, hidden_dim=24, n_layers=2),
                 batch_norm=True)
    model.log = lambda *a, **k: None                     # Lightning's logger is not part of the path
    with torch.no_grad():                                # non-trivial affine / running statistics
        model.bn.weight.uniform_(0.5, 1.5)
        model.bn.bias.normal_(0, 0.2)
        model.bn.running_mean.normal_(0, 0.1)
        model.bn.running_var.uniform_(0.5, 2.0)
    state0 = {k: v.detach().clone().numpy() for k, v in model.state_dict().items()}
    Y = rng.normal(size=(14, 2)).astype(np.float32)
    Y[3, 1] = np.nan
    Y[9, 0] = np.nan
    w = rng.uniform(0.5, 2.0, size=(14,)).astype(np.float32)
    model.train()
    batch = (bmg, None, None, torch.from_numpy(Y), torch.from_numpy(w), None, None)
    loss = model.training_step(batch, 0)
    loss.backward()
    with torch.no_grad():
        model.eval()
        preds_eval = model(bmg)
    d = {"V": bmg.V.numpy(), "E": bmg.E.numpy(), "edge_index": bmg.edge_index.numpy(),
         "rev_edge_index": bmg.rev_edge_index.numpy(), "batch": bmg.batch.numpy(), "n_mols": np.int64(14), "Y": Y, "w": w,
         "loss": loss.detach().numpy(), "preds_eval": preds_eval.numpy()}
    for k, v in state0.items():
        if not k.startswith("metrics."):
            d["param." + k] = v
    for k, v in model.state_dict().items():
        if k.startswith("bn.running") or k == "bn.num_batches_tracked":
            d["after." + k] = v.detach().numpy()
    for k, p in model.named_parameters():
        if p.grad is not None:
            d["grad." + k] = p.grad.numpy()
    return d


# (kind, depth, bias, undirected, activation): the reference's own modules on the synthetic generator's molecules
LIVE_CASES = [("bond", 3, False, False, "relu"), ("bond", 4, True, True, "elu"), ("atom", 3, True, False, "leakyrelu"),
              ("atom", 2, False, False, "tanh"), ("bond", 1, False, False, "relu")]


def live_case_name(kind: str, depth: int, bias: bool, undirected: bool, act: str) -> str:
    return f"fixture_live_{kind}_d{depth}_{act}" + ("_bias" if bias else "") + ("_undirected" if undirected else "")


def live_case_weights(shapes: dict, seed: int = 7) -> dict:
    """Weights of a live case, by name (the module's state-dict keys, sorted): uniform in +-1/sqrt(fan_in), seeded, so that
    the fixture needs no stored weights."""
    rng = np.random.default_rng(seed)
    out = {}
    for k in sorted(shapes):
        fan_in = shapes[k.replace(".bias", ".weight")][-1]
        out[k] = rng.uniform(-1.0, 1.0, size=shapes[k]).astype(np.float32) / np.float32(np.sqrt(fan_in))
    return out


def live_sample(n: int, k: int, seed: int) -> np.ndarray:
    """Sorted indices of a fixed sample of k out of n (all n when n <= k)."""
    return np.arange(n) if n <= k else np.sort(np.random.default_rng(seed).choice(n, size=k, replace=False))


def live_case(kind: str, depth: int, bias: bool, undirected: bool, act: str) -> dict:
    """40 molecules of chemprop_b200.data.make_molecules(40, seed=11, shuffle_edges=True), collated by the reference's
    BatchMolGraph (SHA-256 of each array); its {Bond,Atom}MessagePassing(d_h=96) holding live_case_weights(): H = mp(bmg),
    its mean aggregation, and the weight gradients of loss = sum(mean_agg(H)^2) -- a fixed sample of the entries of each
    (no entry for a weight without a gradient)."""
    import hashlib

    import_reference()
    from chemprop.data import BatchMolGraph
    from chemprop.data.molgraph import MolGraph
    from chemprop.nn import AtomMessagePassing, BondMessagePassing, MeanAggregation

    from chemprop_b200.data.synthetic import make_molecules

    bmg = BatchMolGraph([MolGraph(*m) for m in make_molecules(40, seed=11, shuffle_edges=True)])
    mp = (BondMessagePassing if kind == "bond" else AtomMessagePassing)(d_h=96, depth=depth, bias=bias,
                                                                          undirected=undirected, activation=act)
    W = live_case_weights({k: tuple(v.shape) for k, v in mp.state_dict().items()})
    mp.load_state_dict({k: torch.from_numpy(v) for k, v in W.items()})
    d = {"sha256." + k: hashlib.sha256(np.ascontiguousarray(getattr(bmg, k).numpy()).tobytes()).hexdigest()
         for k in ("V", "E", "edge_index", "rev_edge_index", "batch")}
    d["keys"] = " ".join(sorted(W))
    H = mp(bmg)
    a = MeanAggregation()(H, bmg.batch)
    a.square().sum().backward()
    d["rows.H_v"] = live_sample(H.shape[0], 24, 1)
    d["H_v"] = H.detach().numpy()[d["rows.H_v"]]
    d["agg_mean"] = a.detach().numpy()[live_sample(a.shape[0], 16, 2)]
    for k, p in mp.named_parameters():
        if p.grad is not None:
            d["idx.grad." + k] = live_sample(p.grad.numel(), 512, 3)
            d["grad." + k] = p.grad.numpy().reshape(-1)[d["idx.grad." + k]]
    return d


def seeded_sampler_case() -> dict:
    """The reference's SeededSampler(203, seed=99): the sample order of two consecutive epochs."""
    import_reference()
    from chemprop.data.samplers import SeededSampler

    s = SeededSampler(203, 99)
    return {"order": np.stack([np.fromiter(iter(s), dtype=np.int64) for _ in range(2)]), "n": 203, "seed": 99}


def main():
    """`python -m oracle.make_golden [name ...]`: all cases, or only the named ones (a case's seed is its position in
    CASES, so adding cases at the end never changes the committed ones)."""
    os.makedirs(GOLDEN_DIR, exist_ok=True)
    torch.set_num_threads(1)  # deterministic summation order
    only = set(sys.argv[1:])
    for case in LIVE_CASES:
        name = live_case_name(*case)
        if name in only or not only:
            np.savez_compressed(os.path.join(GOLDEN_DIR, f"{name}.npz"), **live_case(*case))
            print(name)
            only.discard(name)
    if "fixture_seeded_sampler" in only or not only:
        np.savez_compressed(os.path.join(GOLDEN_DIR, "fixture_seeded_sampler.npz"), **seeded_sampler_case())
        print("fixture_seeded_sampler")
        only.discard("fixture_seeded_sampler")
    if not only and len(sys.argv) > 1:
        return
    if "fixture_attentive" in only or not only:
        np.savez_compressed(os.path.join(GOLDEN_DIR, "fixture_attentive.npz"), **attentive_case())
        print("fixture_attentive")
        only.discard("fixture_attentive")
        if not only and len(sys.argv) > 1:
            return
    if "fixture_mpnn_head" in only or not only:
        np.savez_compressed(os.path.join(GOLDEN_DIR, "fixture_mpnn_head.npz"), **mpnn_head_case())
        print("fixture_mpnn_head")
        only.discard("fixture_mpnn_head")
        if not only and len(sys.argv) > 1:
            return
    if "fixture_constrainer" in only or not only:
        np.savez_compressed(os.path.join(GOLDEN_DIR, "fixture_constrainer.npz"), **constrainer_case())
        print("fixture_constrainer")
        only.discard("fixture_constrainer")
        if not only and len(sys.argv) > 1:
            return
    assert only <= set(CASES), only - set(CASES)
    for i, (name, cfg) in enumerate(CASES.items()):
        if only and name not in only:
            continue
        out = (run_mab_case if cfg["kind"].startswith("mab_") else run_case)(name, cfg, seed=100 + i)
        np.savez_compressed(os.path.join(GOLDEN_DIR, f"{name}.npz"), **out)
        ref = out["H_v"] if "H_v" in out else out["H_e"]
        print(f"{name:24s} V={out['V'].shape[0]:4d} E={out['E'].shape[0]:4d} B={int(out['n_mols'])} "
              f"|H|={np.abs(ref).mean():.4f} loss={float(out['loss']):+.5f}")
    if not only:
        np.savez_compressed(os.path.join(GOLDEN_DIR, "collate_fixture.npz"), **collate_case())
        print("collate_fixture")


if __name__ == "__main__":
    main()
