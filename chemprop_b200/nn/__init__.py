from .agg import (Aggregation, AggregationRegistry, AttentiveAggregation, MeanAggregation, NormAggregation,
                  SumAggregation)
from .constrainer import ConstrainerFFN
from .head import (EngineBatchNorm1d, EngineBinaryClassificationFFN, EngineLinear, EngineMPNN,
                   EngineMulticlassClassificationFFN, EngineRegressionFFN)
from .message_passing import AtomMessagePassing, BondMessagePassing
from .mol_atom_bond import MABAtomMessagePassing, MABBondMessagePassing
from .transforms import GraphTransform, ScaleTransform

__all__ = ["Aggregation", "AggregationRegistry", "AttentiveAggregation", "MeanAggregation", "NormAggregation", "SumAggregation",
           "AtomMessagePassing", "BondMessagePassing", "ConstrainerFFN", "MABAtomMessagePassing", "MABBondMessagePassing",
           "GraphTransform", "ScaleTransform", "EngineMPNN", "EngineRegressionFFN", "EngineBatchNorm1d", "EngineLinear",
           "EngineBinaryClassificationFFN", "EngineMulticlassClassificationFFN"]
