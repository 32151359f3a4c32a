"""Molecule-level head of the training step on the engine's kernels (SURVEY.md section 8f-2): what chemprop's `MPNN` does
after the encoder -- `H = agg(H_v, batch)`, `H = bn(H)`, `preds = predictor(H)`, `loss = criterion(preds, targets, mask, w)`
(chemprop/models/model.py:126-161, nn/ffn.py:38-61, nn/predictors.py:101-170, nn/metrics.py:78-123, 139-141) -- for the
regression and classification cases: Mean / Sum / Norm aggregation, optional BatchNorm1d, the MLP of `RegressionFFN` /
`BinaryClassificationFFN` / `MulticlassClassificationFFN`, masked + weighted MSE / BCE / cross entropy.

Every arithmetic step is a libdmpnn launch (aggregation: dmpnn_segment_sum; batch norm: dmpnn_bn_train_fwd / dmpnn_bn_bwd;
the MLP's GEMMs: dmpnn_linear_fwd / dmpnn_linear_wgrad with the activation in the epilogue; the criterion and its gradient:
dmpnn_mse_loss / dmpnn_bce_loss / dmpnn_ce_loss; the classifiers' probabilities: dmpnn_class_probs), none synchronises with
the host, so the encoder + head + backward (+ a capturable optimizer) replay as ONE CUDA graph
(`chemprop_b200.graph.CudaGraphStep`).

Module tree and state-dict keys are the reference's: `bn.{weight,bias,running_mean,running_var,num_batches_tracked}`,
`predictor.ffn.<i>.<j>.{weight,bias}`, `predictor.criterion.task_weights` -- a reference `MPNN` state dict loads with
`strict=True` into `EngineMPNN` (tests/test_dropin_reference_model.py) and vice versa."""
from __future__ import annotations

from typing import Sequence

import torch
from torch import Tensor, nn

from .. import _lib
from .. import engine as K
from .agg import Aggregation, MeanAggregation
from .constrainer import build_mlp
from .message_passing import DEFAULT_HIDDEN_DIM, engine_activation, is_fused_activation


class BatchNormTrainFunction(torch.autograd.Function):
    """nn.BatchNorm1d in training mode on a b x d f32 matrix: dmpnn_bn_train_fwd / dmpnn_bn_bwd."""

    @staticmethod
    def forward(ctx, X, gamma, beta, running_mean, running_var, eps, momentum):
        K._require_cuda(X)
        Xc = X.float().contiguous()
        d = Xc.shape[1]
        Y, Xhat = torch.empty_like(Xc), torch.empty_like(Xc)
        mean, invstd = torch.empty(d, device=X.device), torch.empty(d, device=X.device)
        g = None if gamma is None else gamma.detach().float().contiguous()
        b = None if beta is None else beta.detach().float().contiguous()
        K.bn_train_fwd(Xc, g, b, running_mean, running_var, eps, momentum, Y, Xhat, mean, invstd)
        ctx.save_for_backward(Xhat, invstd, g)
        ctx.has = (gamma is not None, beta is not None)
        return Y

    @staticmethod
    def backward(ctx, dY):
        Xhat, invstd, g = ctx.saved_tensors
        dYc = dY.float().contiguous()
        d = dYc.shape[1]
        dX = torch.empty_like(dYc)
        dg = torch.empty(d, device=dYc.device) if ctx.has[0] else None
        db = torch.empty(d, device=dYc.device) if ctx.has[1] else None
        K.bn_bwd(dYc, Xhat, g, invstd, dX, dg, db)
        return dX, dg, db, None, None, None, None


class MSELossFunction(torch.autograd.Function):
    """chemprop's MSE criterion: sum(w_b * tw_t * mask * (p - y)^2) / sum(mask), mask = isfinite(targets); loss and
    dLoss/dPreds in one launch (dmpnn_mse_loss)."""

    @staticmethod
    def forward(ctx, preds, targets, weights, task_weights):
        K._require_cuda(preds, targets)
        P, Y = preds.float().contiguous(), targets.float().contiguous()
        w = None if weights is None else weights.float().reshape(-1).contiguous()
        tw = None if task_weights is None else task_weights.float().reshape(-1).contiguous()
        loss = torch.empty(1, device=P.device)
        dP = torch.empty_like(P)
        K.mse_loss(P, Y, w, tw, loss, dP)
        ctx.save_for_backward(dP)
        ctx.pdtype = preds.dtype
        return loss.reshape(())

    @staticmethod
    def backward(ctx, g):
        (dP,) = ctx.saved_tensors
        return (dP * g).to(ctx.pdtype), None, None, None


class BCELossFunction(torch.autograd.Function):
    """chemprop's BCELoss on logits: sum(w_b * tw_t * mask * bce(z, y)) / sum(mask), mask = isfinite(targets); loss and
    dLoss/dLogits in one launch (dmpnn_bce_loss)."""

    @staticmethod
    def forward(ctx, preds, targets, weights, task_weights):
        K._require_cuda(preds, targets)
        P, Y = preds.float().contiguous(), targets.float().contiguous()
        w = None if weights is None else weights.float().reshape(-1).contiguous()
        tw = None if task_weights is None else task_weights.float().reshape(-1).contiguous()
        loss = torch.empty(1, device=P.device)
        dP = torch.empty_like(P)
        K.bce_loss(P, Y, w, tw, loss, dP)
        ctx.save_for_backward(dP)
        ctx.pdtype = preds.dtype
        return loss.reshape(())

    @staticmethod
    def backward(ctx, g):
        (dP,) = ctx.saved_tensors
        return (dP * g).to(ctx.pdtype), None, None, None


class CrossEntropyLossFunction(torch.autograd.Function):
    """chemprop's CrossEntropyLoss on `b x t x C` logits and `b x t` class ids: sum(w_b * tw_t * mask * ce) / sum(mask);
    loss and dLoss/dLogits in one launch (dmpnn_ce_loss).  An out-of-range class id gives a NaN loss (no host sync)."""

    @staticmethod
    def forward(ctx, preds, targets, weights, task_weights):
        K._require_cuda(preds, targets)
        if preds.dim() != 3 or tuple(preds.shape[:2]) != tuple(targets.shape):
            raise ValueError(f"expected preds b x t x C and targets b x t, got {tuple(preds.shape)} and {tuple(targets.shape)}")
        C = preds.shape[2]
        P, Y = preds.float().reshape(preds.shape[0], -1).contiguous(), targets.float().contiguous()
        w = None if weights is None else weights.float().reshape(-1).contiguous()
        tw = None if task_weights is None else task_weights.float().reshape(-1).contiguous()
        loss = torch.empty(1, device=P.device)
        dP = torch.empty_like(P)
        K.ce_loss(P, Y, w, tw, loss, dP, C)
        ctx.save_for_backward(dP)
        ctx.meta = (preds.dtype, preds.shape)
        return loss.reshape(())

    @staticmethod
    def backward(ctx, g):
        (dP,) = ctx.saved_tensors
        dtype, shape = ctx.meta
        return (dP.reshape(shape) * g).to(dtype), None, None, None


class ClassProbsFunction(torch.autograd.Function):
    """Eval output of the classification heads on `b x (t C)` logits: sigmoid (C == 1) or the softmax of each group of C
    columns (dmpnn_class_probs); mirror from the saved probabilities (dmpnn_class_probs_bwd)."""

    @staticmethod
    def forward(ctx, logits, C):
        K._require_cuda(logits)
        P = logits.float().contiguous()
        Q = torch.empty_like(P)
        K.class_probs(P, C, Q)
        ctx.save_for_backward(Q)
        ctx.meta = (logits.dtype, C)
        return Q

    @staticmethod
    def backward(ctx, dQ):
        (Q,) = ctx.saved_tensors
        dtype, C = ctx.meta
        dP = torch.empty_like(Q)
        K.class_probs_bwd(Q, dQ.float().contiguous(), C, dP)
        return dP.to(dtype), None


class LinearActFunction(torch.autograd.Function):
    """Y = act(X . W^T + b) with the activation in the GEMM epilogue (dmpnn_linear_fwd); mirror: dZ = dY * act'(Y)
    (dmpnn_act_bwd), dW / db (dmpnn_linear_wgrad), dX = dZ . W (dmpnn_linear_fwd)."""

    @staticmethod
    def forward(ctx, X, W, b, act, act_param):
        K._require_cuda(X, W)
        Xc, Wc = X.float().contiguous(), W.detach().float().contiguous()
        bc = None if b is None else b.detach().float().contiguous()
        R, Kd = Xc.shape
        N = Wc.shape[0]
        Y = torch.empty((R, N), dtype=torch.float32, device=X.device)
        if R > 0:
            K.linear_fwd(Xc, Kd, Wc, Y, N, bias=bc, act=act, act_param=act_param, R=R, pad_to=N)
        ctx.save_for_backward(Xc, Wc, Y)
        ctx.cfg = (act, act_param, b is not None, W.dtype, None if b is None else b.dtype)
        return Y

    @staticmethod
    def backward(ctx, dY):
        Xc, Wc, Y = ctx.saved_tensors
        act, ap, has_b, wdt, bdt = ctx.cfg
        R, Kd = Xc.shape
        N = Wc.shape[0]
        dYc = dY.float().contiguous()
        dZ = dYc
        if act != _lib.ACT_NONE and R > 0:
            dZ = torch.empty_like(dYc)
            K.act_bwd(dYc, Y, R, N, act=act, act_param=ap, dZ=dZ)
        dW = torch.zeros_like(Wc)
        db = torch.zeros(N, dtype=torch.float32, device=Wc.device) if has_b else None
        dX = torch.zeros_like(Xc) if ctx.needs_input_grad[0] else None
        if R > 0:
            K.linear_wgrad(dZ, Xc, Kd, dW, N, dbias=db, R=R)
            if dX is not None:
                K.linear_fwd(dZ, N, Wc.t().contiguous(), dX, Kd, R=R, pad_to=Kd)
        return dX, dW.to(wdt), (None if db is None else db.to(bdt)), None, None


class EngineLinear(nn.Linear):
    """nn.Linear (same parameters / state-dict keys) executed by dmpnn_linear_fwd / dmpnn_linear_wgrad (f32)."""

    def forward(self, x: Tensor, act: int = _lib.ACT_NONE, act_param: float = 0.0) -> Tensor:
        return LinearActFunction.apply(x, self.weight, self.bias, act, act_param)


class _Criterion(nn.Module):
    """chemprop's `ChempropMetric` call signature and `task_weights` buffer (1 x t); masked, weighted MSE."""
    _function = MSELossFunction

    def __init__(self, task_weights):
        super().__init__()
        self.register_buffer("task_weights", torch.as_tensor(task_weights, dtype=torch.float).view(1, -1))

    def forward(self, preds, targets, mask=None, weights=None, lt_mask=None, gt_mask=None):
        if lt_mask is not None or gt_mask is not None:
            raise NotImplementedError("bounded MSE is not part of the engine's head; use the reference criterion")
        t = targets if mask is None else torch.where(mask, targets, torch.full_like(targets, float("nan")))
        return self._function.apply(preds, t, weights, self.task_weights)


class _BCECriterion(_Criterion):
    """chemprop's `BCELoss` (nn/metrics.py:292-295): binary cross entropy on logits, soft labels accepted."""
    _function = BCELossFunction


class _CrossEntropyCriterion(_Criterion):
    """chemprop's `CrossEntropyLoss` (nn/metrics.py:298-303): preds `b x t x C` logits, targets `b x t` class ids."""
    _function = CrossEntropyLossFunction


class _EngineFFN(nn.Module):
    """The MLP of chemprop's `_FFNPredictorBase` (chemprop/nn/predictors.py:101-157) with the reference's module tree
    (`ffn.<i>.<j>`, `criterion.task_weights`); GEMMs on the engine."""
    n_targets = 1
    _criterion = _Criterion

    def __init__(self, output_dim: int, n_tasks: int, input_dim: int, hidden_dim: int | Sequence[int], n_layers: int,
                 dropout: float, activation, task_weights):
        super().__init__()
        ffn = build_mlp(input_dim, output_dim, hidden_dim, n_layers, dropout, activation)
        for block in ffn:                         # same tree, engine-backed Linear layers
            for i, m in enumerate(block):
                if isinstance(m, nn.Linear):
                    e = EngineLinear(m.in_features, m.out_features, m.bias is not None)
                    e.load_state_dict(m.state_dict())
                    block[i] = e
        self.ffn = ffn
        self.criterion = self._criterion(torch.ones(n_tasks) if task_weights is None else task_weights)
        self.output_transform = nn.Identity()

    @property
    def input_dim(self) -> int:
        return self.ffn[0][-1].in_features

    @property
    def output_dim(self) -> int:
        return self.ffn[-1][-1].out_features

    @property
    def n_tasks(self) -> int:
        return self.output_dim

    def _mlp(self, Z: Tensor) -> Tensor:
        """`self.ffn(Z)` (nn/ffn.py:38-61: Linear, then [act, dropout, Linear] per further layer) with every activation the
        engine fuses folded into the epilogue of the GEMM before it."""
        blocks = [list(b) for b in self.ffn]
        X = Z
        for k, block in enumerate(blocks):
            lin = block[-1]
            if k + 1 == len(blocks):
                X = lin(X)
                break
            tau, drop = blocks[k + 1][0], blocks[k + 1][1]
            if is_fused_activation(tau):
                X = lin(X, *engine_activation(tau))          # act(W x + b) in the GEMM epilogue
            else:
                X = tau(lin(X))
            X = drop(X)                                      # identity when p = 0 or in eval mode
        return X


class EngineRegressionFFN(_EngineFFN):
    """`RegressionFFN` (chemprop/nn/predictors.py:156-164) with the reference's module tree; GEMMs on the engine."""

    def __init__(self, n_tasks: int = 1, input_dim: int = DEFAULT_HIDDEN_DIM, hidden_dim: int | Sequence[int] = 300,
                 n_layers: int = 1, dropout: float = 0.0, activation="relu", task_weights=None):
        super().__init__(n_tasks, n_tasks, input_dim, hidden_dim, n_layers, dropout, activation, task_weights)
        self.hparams = dict(n_tasks=n_tasks, input_dim=input_dim, hidden_dim=hidden_dim, n_layers=n_layers, dropout=dropout,
                            activation=activation, cls=self.__class__)

    def forward(self, Z: Tensor) -> Tensor:
        return self.output_transform(self._mlp(Z))

    train_step = forward


class EngineBinaryClassificationFFN(_EngineFFN):
    """`BinaryClassificationFFN` (chemprop/nn/predictors.py:235-247): `train_step` gives the `b x t` logits the BCE criterion
    takes, `forward` their sigmoid (dmpnn_class_probs).  `threshold` is kept in `hparams` only, as in the reference, where
    the BCE criterion ignores it."""
    _criterion = _BCECriterion

    def __init__(self, n_tasks: int = 1, input_dim: int = DEFAULT_HIDDEN_DIM, hidden_dim: int | Sequence[int] = 300,
                 n_layers: int = 1, dropout: float = 0.0, activation="relu", task_weights=None, threshold: float | None = None):
        super().__init__(n_tasks, n_tasks, input_dim, hidden_dim, n_layers, dropout, activation, task_weights)
        self.hparams = dict(n_tasks=n_tasks, input_dim=input_dim, hidden_dim=hidden_dim, n_layers=n_layers, dropout=dropout,
                            activation=activation, task_weights=task_weights, threshold=threshold, cls=self.__class__)

    def forward(self, Z: Tensor) -> Tensor:
        return ClassProbsFunction.apply(self._mlp(Z), 1)

    def train_step(self, Z: Tensor) -> Tensor:
        return self._mlp(Z)


class EngineMulticlassClassificationFFN(_EngineFFN):
    """`MulticlassClassificationFFN` (chemprop/nn/predictors.py:271-314): `n_tasks * n_classes` outputs; `train_step` gives
    the `b x t x C` logits the cross-entropy criterion takes, `forward` the softmax over the classes (dmpnn_class_probs)."""
    _criterion = _CrossEntropyCriterion

    def __init__(self, n_classes: int, n_tasks: int = 1, input_dim: int = DEFAULT_HIDDEN_DIM,
                 hidden_dim: int | Sequence[int] = 300, n_layers: int = 1, dropout: float = 0.0, activation="relu",
                 task_weights=None, threshold: float | None = None):
        super().__init__(n_tasks * n_classes, n_tasks, input_dim, hidden_dim, n_layers, dropout, activation, task_weights)
        self.n_classes = n_classes
        self.hparams = dict(n_classes=n_classes, n_tasks=n_tasks, input_dim=input_dim, hidden_dim=hidden_dim,
                            n_layers=n_layers, dropout=dropout, activation=activation, task_weights=task_weights,
                            threshold=threshold, cls=self.__class__)

    @property
    def n_tasks(self) -> int:
        return self.output_dim // (self.n_targets * self.n_classes)

    def forward(self, Z: Tensor) -> Tensor:
        return ClassProbsFunction.apply(self._mlp(Z), self.n_classes).reshape(Z.shape[0], -1, self.n_classes)

    def train_step(self, Z: Tensor) -> Tensor:
        return self._mlp(Z).reshape(Z.shape[0], -1, self.n_classes)


class EngineBatchNorm1d(nn.BatchNorm1d):
    """nn.BatchNorm1d (same parameters / buffers); training mode runs dmpnn_bn_train_fwd / dmpnn_bn_bwd."""

    def forward(self, x: Tensor) -> Tensor:
        # torch's own path where the kernel has no equivalent: eval mode, CPU tensors, no running statistics, and
        # momentum=None (cumulative average: the factor 1 / num_batches_tracked is host state, a sync per step)
        if not self.training or not x.is_cuda or self.running_mean is None or self.momentum is None:
            return super().forward(x)
        if x.dim() != 2:
            raise ValueError(f"expected a 2D input (molecules x features), got {x.dim()}D")
        if x.shape[0] <= 1:                       # as torch: the batch variance of one row is undefined (the reference's
            raise ValueError(f"Expected more than 1 value per channel when training, got input size {tuple(x.shape)}")  # loader drops such a batch, dataloader.py:77-86)
        if self.num_batches_tracked is not None:
            self.num_batches_tracked.add_(1)
        return BatchNormTrainFunction.apply(x, self.weight, self.bias, self.running_mean, self.running_var, self.eps,
                                            self.momentum)


class EngineMPNN(nn.Module):
    """`chemprop.models.MPNN` reduced to the path (models/model.py:66-161): message passing -> aggregation -> batch norm ->
    predictor -> criterion, all on the engine.  `training_loss(bmg, targets, weights=None)` is `MPNN.training_step` without
    Lightning's logging; `forward(bmg)` gives the predictions."""

    def __init__(self, message_passing: nn.Module, agg: Aggregation | None = None, predictor: nn.Module | None = None,
                 batch_norm: bool = False):
        super().__init__()
        self.message_passing = message_passing
        self.agg = agg if agg is not None else MeanAggregation()
        self.bn = EngineBatchNorm1d(message_passing.output_dim) if batch_norm else nn.Identity()
        self.predictor = predictor if predictor is not None else EngineRegressionFFN(input_dim=message_passing.output_dim)

    def fingerprint(self, bmg, V_d: Tensor | None = None, X_d: Tensor | None = None) -> Tensor:
        H = self.bn(self.agg(self.message_passing(bmg, V_d), bmg.batch))
        return H if X_d is None else torch.cat((H, X_d), dim=1)

    def forward(self, bmg, V_d: Tensor | None = None, X_d: Tensor | None = None) -> Tensor:
        return self.predictor(self.fingerprint(bmg, V_d, X_d))

    def training_loss(self, bmg, targets: Tensor, weights: Tensor | None = None, V_d=None, X_d=None) -> Tensor:
        preds = self.predictor.train_step(self.fingerprint(bmg, V_d, X_d))
        return self.predictor.criterion(preds, targets, None, weights)      # NaN targets are the mask (model.py:140-141)
