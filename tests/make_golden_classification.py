"""TEST INFRASTRUCTURE ONLY.  Generates the classification-head fixtures, tests/golden/fixture_mpnn_head_bce.npz and
fixture_mpnn_head_multiclass.npz, by running the UNMODIFIED reference chemprop (`REFERENCE_ROOT`, imported through
oracle/ref_shim.py): its `MPNN.training_step` with `BinaryClassificationFFN` + `BCELoss` and `MulticlassClassificationFFN` +
`CrossEntropyLoss`.  The fixtures hold the keys of oracle/make_golden.py's `fixture_mpnn_head` (inputs, initial state dict,
loss, every gradient, batch-norm statistics after the step, eval predictions).  Run where the reference is reachable; the
outputs are committed.

    python -m tests.make_golden_classification [fixture_mpnn_head_bce] [fixture_mpnn_head_multiclass]
"""
from __future__ import annotations

import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
from oracle.ref_shim import import_reference  # noqa: E402

GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")


def _mpnn_classification_head_case(make_predictor, make_targets, seed: int) -> dict:
    """`MPNN(BondMessagePassing(d_h = 40), MeanAggregation, <predictor>, batch_norm = True).training_step(batch)` of the
    reference on 14 seeded molecules with NaN targets and per-molecule weights; the keys of `mpnn_head_case`."""
    import_reference()
    import chemprop.nn as ref_nn
    from chemprop.data import BatchMolGraph as RefBMG
    from chemprop.data.molgraph import MolGraph as RefMG
    from chemprop.models import MPNN

    from chemprop_b200.data.synthetic import make_molecules

    rng = np.random.default_rng(seed)
    torch.manual_seed(seed)
    mgs = make_molecules(14, seed=seed, mean_atoms=9, std_atoms=3, min_atoms=1)
    bmg = RefBMG([RefMG(*m) for m in mgs])
    mp = ref_nn.BondMessagePassing(d_h=40, depth=3)
    model = MPNN(mp, ref_nn.MeanAggregation(), make_predictor(ref_nn), batch_norm=True)
    model.log = lambda *a, **k: None
    with torch.no_grad():
        model.bn.weight.uniform_(0.5, 1.5)
        model.bn.bias.normal_(0, 0.2)
        model.bn.running_mean.normal_(0, 0.1)
        model.bn.running_var.uniform_(0.5, 2.0)
    state0 = {k: v.detach().clone().numpy() for k, v in model.state_dict().items()}
    Y = make_targets(rng)
    w = rng.uniform(0.5, 2.0, size=(14,)).astype(np.float32)
    model.train()
    loss = model.training_step((bmg, None, None, torch.from_numpy(Y), torch.from_numpy(w), None, None), 0)
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


def mpnn_head_bce_case() -> dict:
    """BinaryClassificationFFN(n_tasks = 3, 2 layers, task weights (0.5, 1, 2)) + BCELoss: 0 / 1 labels, one soft label
    (0.3) and three NaN (masked) targets."""
    def targets(rng):
        Y = (rng.uniform(size=(14, 3)) < 0.4).astype(np.float32)
        Y[2, 1] = 0.3
        Y[3, 0] = Y[9, 2] = Y[11, 1] = np.nan
        return Y

    return _mpnn_classification_head_case(
        lambda ref_nn: ref_nn.BinaryClassificationFFN(n_tasks=3, input_dim=40, hidden_dim=24, n_layers=2,
                                                      task_weights=torch.tensor([0.5, 1.0, 2.0])), targets, seed=98)


def mpnn_head_multiclass_case() -> dict:
    """MulticlassClassificationFFN(n_classes = 4, n_tasks = 2, 2 layers, task weights (1.5, 0.75)) + CrossEntropyLoss:
    class ids with two NaN (masked) targets."""
    def targets(rng):
        Y = rng.integers(0, 4, size=(14, 2)).astype(np.float32)
        Y[5, 0] = Y[12, 1] = np.nan
        return Y

    return _mpnn_classification_head_case(
        lambda ref_nn: ref_nn.MulticlassClassificationFFN(n_classes=4, n_tasks=2, input_dim=40, hidden_dim=24, n_layers=2,
                                                          task_weights=torch.tensor([1.5, 0.75])), targets, seed=99)


CASES = {"fixture_mpnn_head_bce": mpnn_head_bce_case, "fixture_mpnn_head_multiclass": mpnn_head_multiclass_case}


def main():
    """All cases, or only the named ones; one thread, for a fixed summation order."""
    torch.set_num_threads(1)
    only = set(sys.argv[1:])
    assert only <= set(CASES), only - set(CASES)
    for name, case in CASES.items():
        if not only or name in only:
            np.savez_compressed(os.path.join(GOLDEN_DIR, f"{name}.npz"), **case())
            print(name)


if __name__ == "__main__":
    main()
