"""CPU tier: pins oracle/restatement.py against the reference through the committed golden vectors and fixtures
(produced by the unmodified reference, oracle/make_golden.py)."""
import numpy as np
import pytest
import torch

from oracle import layout_np, restatement as R
from oracle.make_golden import LIVE_CASES, live_case_name, live_case_weights, live_sample
from tests.util import golden_names, load_golden, mab_oracle_forward, oracle_forward

TOL = dict(rtol=1e-5, atol=1e-6)  # same torch ops on the same machine: differences are summation-order only


@pytest.mark.parametrize("name", golden_names())
def test_restatement_matches_golden(name):
    torch.set_num_threads(1)
    g = load_golden(name)
    H, P = oracle_forward(g, torch.float32, requires_grad=True)
    np.testing.assert_allclose(H.detach().numpy(), g["H_v"], **TOL)
    batch = torch.from_numpy(g["batch"])
    for mode in ("mean", "sum", "norm"):
        out = R.aggregate(H, batch, mode)
        np.testing.assert_allclose(out.detach().numpy(), g[f"agg_{mode}"], **TOL)
    loss = (R.aggregate(H, batch, "mean") * torch.from_numpy(g["G"])).sum()
    assert abs(loss.item() - float(g["loss"])) <= 1e-5 * max(1.0, abs(float(g["loss"])))
    loss.backward()
    for k, v in g.items():
        if k.startswith("grad."):
            got = P[k[len("grad."):]].grad
            assert got is not None, k
            np.testing.assert_allclose(got.numpy(), v, rtol=1e-4, atol=2e-6, err_msg=k)


@pytest.mark.parametrize("name", golden_names(mab=True))
def test_mab_restatement_matches_golden(name):
    """mol_atom_bond.py variants: vertex and per-edge embeddings and every weight gradient."""
    torch.set_num_threads(1)
    g = load_golden(name)
    H_v, H_e, P = mab_oracle_forward(g, torch.float32, requires_grad=True)
    loss = torch.zeros(())
    if "H_v" in g:
        np.testing.assert_allclose(H_v.detach().numpy(), g["H_v"], **TOL)
        loss = loss + (R.aggregate(H_v, torch.from_numpy(g["batch"]), "mean") * torch.from_numpy(g["G"])).sum()
    else:
        assert H_v is None
    if "H_e" in g:
        np.testing.assert_allclose(H_e.detach().numpy(), g["H_e"], **TOL)
        loss = loss + (H_e * torch.from_numpy(g["G_e"])).sum()
    else:
        assert H_e is None
    assert abs(loss.item() - float(g["loss"])) <= 1e-5 * max(1.0, abs(float(g["loss"])))
    loss.backward()
    for k, v in g.items():
        if k.startswith("grad."):
            np.testing.assert_allclose(P[k[len("grad."):]].grad.numpy(), v, rtol=1e-4, atol=2e-6, err_msg=k)


def test_attentive_restatement_matches_reference_fixture():
    g = load_golden("fixture_attentive")
    H = torch.from_numpy(g["H"]).requires_grad_(True)
    W, b = (torch.from_numpy(g[k]).requires_grad_(True) for k in ("param.W.weight", "param.W.bias"))
    out = R.attentive_aggregate(H, torch.from_numpy(g["batch"]), W, b)
    np.testing.assert_allclose(out.detach().numpy(), g["out"], **TOL)
    (out * torch.from_numpy(g["G"])).sum().backward()
    for t, k in ((H, "grad.H"), (W, "grad.W.weight"), (b, "grad.W.bias")):
        np.testing.assert_allclose(t.grad.numpy(), g[k], rtol=1e-4, atol=2e-6, err_msg=k)


def test_smiles_topology_parser_of_config1():
    """oracle/smiles_topology.py (BASELINE config 1 graphs): atoms / bonds of hand-checked SMILES, featuriser edge order."""
    from oracle.smiles_topology import parse, to_molgraph

    atoms, bonds = parse("Cc1occc1C(=O)Nc2ccccc2")                      # 2-methyl-3-furanilide: 15 heavy atoms, 2 rings
    assert len(atoms) == 15 and len(bonds) == 16 and (6, 7, 1) in bonds and (1, 5, 3) in bonds and (9, 14, 3) in bonds
    atoms, bonds = parse("c1ccc2[nH]ccc2c1")                            # indole
    assert len(atoms) == 9 and len(bonds) == 10 and atoms[4] == ("N", True, 1)
    atoms, bonds = parse("ClC(Br)(F)C#N")
    assert [a[0] for a in atoms] == ["Cl", "C", "Br", "F", "C", "N"] and (4, 5, 2) in bonds and len(bonds) == 5
    assert len(parse("CC.O")[1]) == 1 and len(parse("C1CC1")[1]) == 3 and len(parse("F/C=C/F")[1]) == 3
    for bad in ("C1CC", "C(C", "C*C"):
        with pytest.raises(ValueError):
            parse(bad)
    mg = to_molgraph("CC(=O)O")
    assert mg.V.shape == (4, 72) and mg.E.shape == (6, 14) and mg.edge_index.tolist() == [[0, 1, 1, 2, 1, 3], [1, 0, 2, 1, 3, 1]]
    assert mg.rev_edge_index.tolist() == [1, 0, 3, 2, 5, 4] and np.array_equal(mg.E[0], mg.E[1]) and mg.E[2, 1] == 1
    g = load_golden("config1_regression_b50")                           # the committed graphs of config 1: 50 molecules
    assert int(g["n_mols"]) == 50 and g["config"]["d_h"] == 300 and g["V"].shape[1] == 72 and g["E"].shape[1] == 14
    assert np.array_equal(g["rev_edge_index"], np.arange(g["E"].shape[0]) ^ 1)


def test_constrain_restatement_matches_reference_fixture():
    g = load_golden("fixture_constrainer")
    t = lambda k: torch.from_numpy(g[k])  # noqa: E731
    h = torch.tanh(torch.nn.functional.linear(t("fp"), t("param.ffn.0.0.weight"), t("param.ffn.0.0.bias")))
    h = torch.tanh(torch.nn.functional.linear(h, t("param.ffn.1.2.weight"), t("param.ffn.1.2.bias")))
    k = torch.nn.functional.linear(h, t("param.ffn.2.2.weight"), t("param.ffn.2.2.bias"))
    out = R.constrain(k, t("preds"), t("batch"), t("constraints"))
    np.testing.assert_allclose(out.numpy(), g["out"], **TOL)


def test_restatement_fp64_close_to_fp32_golden():
    g = load_golden("bond_d3_h300")
    H, _ = oracle_forward(g, torch.float64)
    assert np.abs(H.numpy() - g["H_v"]).max() < 2e-6


def test_collate_restatement_matches_reference_fixture():
    """tests/unit/data/test_dataloader.py:10-84 fixture, collated by the real reference."""
    from chemprop_b200.data import MolGraph

    g = load_golden("collate_fixture")
    mgs = [MolGraph(g[f"mg{i}.V"], g[f"mg{i}.E"], g[f"mg{i}.edge_index"], g[f"mg{i}.rev_edge_index"]) for i in range(2)]
    V, E, ei, rev, batch = R.collate(mgs)
    for a, k in ((V, "V"), (E, "E"), (ei, "edge_index"), (rev, "rev_edge_index"), (batch, "batch")):
        assert a.dtype == g[k].dtype and np.array_equal(a, g[k]), k
    for a, k in zip(R.collate_torch(mgs), ("V", "E", "edge_index", "rev_edge_index", "batch")):
        assert np.array_equal(a.numpy(), g[k]) and a.dtype in (torch.float32, torch.int64), k


def test_layout_restatement_properties():
    g = load_golden("bond_d3_mixed")
    L = layout_np.build_layout(g["edge_index"], g["rev_edge_index"], g["batch"], int(g["n_mols"]))
    E = g["edge_index"].shape[1]
    dst = g["edge_index"][1]
    assert np.array_equal(np.sort(L["perm"]), np.arange(E))
    assert np.all(np.diff(dst[L["perm"]]) >= 0)                       # sorted by destination
    for v in range(len(g["batch"])):                                  # stable inside a bucket
        seg = L["perm"][L["rowptr"][v]:L["rowptr"][v + 1]]
        assert np.all(np.diff(seg) > 0) and np.all(dst[seg] == v)
    assert np.array_equal(L["rev_row"][L["rev_row"]], np.arange(E))   # still an involution
    assert L["flags"] == 7
    rows = np.diff(L["mol_row_ptr"][L["tile_mol_ptr"]])
    assert rows.max() <= 128 and L["tile_mol_ptr"][-1] == int(g["n_mols"])
    Lb = layout_np.build_layout(*(load_golden("bond_d3_big_mol")[k] for k in ("edge_index", "rev_edge_index", "batch")), 3)
    assert Lb["max_tile_rows"] > 128 and Lb["n_tiles"] == 3


@pytest.mark.parametrize("kind,depth,bias,undirected,act", LIVE_CASES)
def test_restatement_matches_live_reference(kind, depth, bias, undirected, act):
    """The reference's own modules and collate on the synthetic generator's molecules (oracle/make_golden.py live_case):
    the restated collate is bit-identical, and the restatement's hidden states, mean aggregation and weight gradients
    match the reference's on the same weights."""
    import hashlib

    from chemprop_b200.data.synthetic import make_molecules
    from chemprop_b200.nn import AtomMessagePassing, BondMessagePassing

    g = load_golden(live_case_name(kind, depth, bias, undirected, act))
    torch.set_num_threads(1)
    mgs = make_molecules(40, seed=11, shuffle_edges=True)
    arrays = dict(zip(("V", "E", "edge_index", "rev_edge_index", "batch"), R.collate(mgs)))
    for k, v in arrays.items():
        assert hashlib.sha256(np.ascontiguousarray(v).tobytes()).hexdigest() == str(g["sha256." + k]), k
    cls = BondMessagePassing if kind == "bond" else AtomMessagePassing
    shapes = {k: tuple(v.shape) for k, v in cls(d_h=96, depth=depth, bias=bias, undirected=undirected,
                                                  activation=act).state_dict().items()}
    assert " ".join(sorted(shapes)) == str(g["keys"])                  # the engine module's state dict is the reference's
    P = {k: torch.from_numpy(v).requires_grad_(True) for k, v in live_case_weights(shapes).items()}
    V, E, ei, rev, batch = (torch.from_numpy(arrays[k]) for k in ("V", "E", "edge_index", "rev_edge_index", "batch"))
    H = R.message_passing_forward(kind, V, E, ei, rev, P["W_i.weight"], P.get("W_i.bias"), P["W_h.weight"],
                                  P.get("W_h.bias"), P["W_o.weight"], P.get("W_o.bias"), depth, act, undirected)
    np.testing.assert_allclose(H.detach().numpy()[g["rows.H_v"]], g["H_v"], **TOL)
    a = R.aggregate(H, batch, "mean")
    np.testing.assert_allclose(a.detach().numpy()[live_sample(a.shape[0], 16, 2)], g["agg_mean"], **TOL)
    a.square().sum().backward()
    for k, p in P.items():
        if "grad." + k not in g:
            assert p.grad is None, k
            continue
        got = p.grad.numpy().reshape(-1)[g["idx.grad." + k]]
        np.testing.assert_allclose(got, g["grad." + k], rtol=1e-4, atol=1e-6, err_msg=k)
