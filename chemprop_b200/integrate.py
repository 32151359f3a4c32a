"""Glue for running the engine's modules inside an installed chemprop (optional; nothing here is imported by the
engine itself, and chemprop need not be installed).

The engine's modules already satisfy chemprop's module protocols (`MessagePassing` / `Aggregation`:
chemprop/nn/message_passing/proto.py:9-34, chemprop/nn/agg.py:19-59): `MPNN(message_passing=<engine module>,
agg=<engine module>, predictor=...)` works as is, checkpoints rebuild them through `hparams["cls"]`
(chemprop/models/model.py:267-271) and reference state dicts load unchanged.  What is left is nominal typing:
chemprop's CLI asks `isinstance(mp, BondMessagePassing)` (chemprop/cli/predict.py:256).  `register_with_chemprop()`
registers the engine classes as virtual subclasses of their chemprop counterparts (the reference classes have an
ABC metaclass through their `HasHParams` protocol base), so those checks hold without inheriting any reference code.
"""
from __future__ import annotations


def register_with_chemprop() -> dict:
    """Returns {engine class: chemprop class} for the pairs that were registered.  Raises ImportError when chemprop is
    not importable."""
    import chemprop.nn as ref_nn
    from chemprop.nn.message_passing import mol_atom_bond as ref_mab

    from . import nn as ours

    pairs = {
        ours.BondMessagePassing: ref_nn.BondMessagePassing,
        ours.AtomMessagePassing: ref_nn.AtomMessagePassing,
        ours.MABBondMessagePassing: ref_mab.MABBondMessagePassing,
        ours.MABAtomMessagePassing: ref_mab.MABAtomMessagePassing,
        ours.MeanAggregation: ref_nn.MeanAggregation,
        ours.SumAggregation: ref_nn.SumAggregation,
        ours.NormAggregation: ref_nn.NormAggregation,
        ours.AttentiveAggregation: ref_nn.AttentiveAggregation,
        ours.Aggregation: ref_nn.Aggregation,
        # chemprop/cli/predict.py:509, 546 branch on isinstance(model.predictor, MulticlassClassificationFFN)
        ours.EngineBinaryClassificationFFN: ref_nn.BinaryClassificationFFN,
        ours.EngineMulticlassClassificationFFN: ref_nn.MulticlassClassificationFFN,
    }
    try:
        from chemprop.nn.ffn import ConstrainerFFN as ref_constrainer

        pairs[ours.ConstrainerFFN] = ref_constrainer
    except Exception:  # noqa: BLE001 -- older chemprop without the mol-atom-bond models
        pass
    done = {}
    for mine, theirs in pairs.items():
        reg = getattr(theirs, "register", None)
        if reg is None:
            continue
        reg(mine)
        done[mine] = theirs
    return done
