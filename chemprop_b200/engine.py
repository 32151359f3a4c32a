"""Host side of the engine: device layout, thin wrappers over the C ABI (raw pointers in, nothing
allocated inside the library) and the autograd functions the nn modules call.

PyTorch here is plumbing only: it owns device memory (caching allocator), streams and the
autograd graph; every arithmetic step on the path is a kernel of libdmpnn_sm100.so.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass

import torch
from torch import Tensor

from . import _lib
from ._lib import (ACT_ELU, ACT_LEAKYRELU, ACT_NONE, ACT_RELU, ACT_TANH, BF16, F32, SCALE_DIV_CONST,
                   SCALE_INV_COUNT, SCALE_NONE, DmpnnError)

# backward of the bf16 tier: True = the last mirror step sums the dZ^t into dH_0 in its epilogue (one W_i GEMM);
# False = the terms stay apart and the W_i gradient accumulates one GEMM per term (measured faster at depth 3)
SUM_IN_EPILOGUE = False

# True: a BatchMolGraph that carries host-computed layout meta words (our collate: dmpnn_batch_meta_host) is trusted
# and the step never synchronises on the device copy; False: always read the device-computed words (one sync per batch)
HOST_META = os.environ.get("DMPNN_HOST_META", "1") != "0"      # DMPNN_HOST_META=0: A/B switch for measurements

HIDDEN_ALIGN = 64  # hidden row stride padded to 64 elements: bf16 rows start on 128-byte lines (one TMA request per box row)

# Optional device-side timing of the depth step (bench.py's roofline): when a list, every depth step
# appends (tag, start_event, end_event) recorded on the launching stream.
STEP_EVENTS: list | None = None


class _StepTimer:
    def __init__(self, tag: str):
        self.tag = tag

    def __enter__(self):
        if STEP_EVENTS is not None:
            self.e0 = torch.cuda.Event(enable_timing=True)
            self.e1 = torch.cuda.Event(enable_timing=True)
            self.e0.record(torch.cuda.current_stream())
        return self

    def __exit__(self, *exc):
        if STEP_EVENTS is not None:
            self.e1.record(torch.cuda.current_stream())
            STEP_EVENTS.append((self.tag, self.e0, self.e1))
        return False


_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)
_raw_device = getattr(torch._C, "_cuda_getDevice", None)


def _stream() -> int:
    """cudaStream_t of torch's current stream on the current device.  Called once per kernel launch (~60 per training step):
    the raw accessors cost ~0.3 us, `torch.cuda.current_stream().cuda_stream` ~15 us (0.45 ms of host time per step)."""
    if _raw_stream is not None and _raw_device is not None:
        return _raw_stream(_raw_device())
    return torch.cuda.current_stream().cuda_stream


def _dt(t: Tensor) -> int:
    if t.dtype == torch.float32:
        return F32
    if t.dtype == torch.bfloat16:
        return BF16
    raise DmpnnError(f"unsupported dtype {t.dtype}")


def _ptr(t: Tensor | None) -> int | None:
    return None if t is None else t.data_ptr()


def _ld(t: Tensor) -> int:
    assert t.dim() == 2 and (t.stride(1) == 1 or t.shape[1] <= 1), "rows must be contiguous"
    return max(int(t.stride(0)), int(t.shape[1]))


def _require_cuda(*ts: Tensor):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise DmpnnError(
                "chemprop_b200 runs on CUDA (sm_100a) only; got a CPU tensor. There is no CPU fallback: "
                "move the BatchMolGraph and the module to the GPU."
            )


def pad_hidden(h: int) -> int:
    return (h + HIDDEN_ALIGN - 1) // HIDDEN_ALIGN * HIDDEN_ALIGN


# ----------------------------------------------------------------------------------------------
# layout
# ----------------------------------------------------------------------------------------------
@dataclass
class Layout:
    V: int
    E: int
    B: int
    perm: Tensor
    inv_perm: Tensor
    rowptr: Tensor
    src_row: Tensor
    dst_row: Tensor
    rev_row: Tensor
    mol_atom_ptr: Tensor
    mol_row_ptr: Tensor
    tile_mol_ptr: Tensor
    tile_row_ptr: Tensor
    tile_atom_ptr: Tensor
    meta: Tensor
    _meta_host: list | None = None
    _work: tuple | None = None
    _atom_work: tuple | None = None

    def _host(self):
        if self._meta_host is None:
            self._meta_host = self.meta.tolist()  # one small D2H sync per batch
        return self._meta_host

    @property
    def n_tiles(self) -> int:
        return self._host()[_lib.META_N_TILES]

    @property
    def flags(self) -> int:
        return self._host()[_lib.META_FLAGS]

    @property
    def max_indeg(self) -> int:
        return self._host()[_lib.META_MAX_INDEG]

    @property
    def max_tile_rows(self) -> int:
        return self._host()[_lib.META_MAX_TILE_ROWS]

    @property
    def max_tile_atoms(self) -> int:
        return self._host()[_lib.META_MAX_TILE_ATOMS]

    def validate(self):
        check_flags(self.flags)

    def step_tables(self):
        """(tile_row_ptr, tile_atom_ptr, n_tiles, work_flag, n_work_dev, dst_row) for the fused depth step.  Batches whose
        molecules all fit a 128-row tile pass the layout's tile tables as they are; a batch with larger molecules (condensed
        reaction graphs) gets the work table of dmpnn_work_table_build: oversized tiles cut into 128-row windows, built once
        per batch on the device (no host read-back: the kernel reads the window count from device memory)."""
        if self.max_tile_rows <= 128:
            return self.tile_row_ptr, self.tile_atom_ptr, self.n_tiles, None, None, None
        if self._work is None:
            lib = _lib.load()
            dev = self.rowptr.device
            cap = self.n_tiles + self.E // 128 + 2
            wr = torch.empty(cap + 1, dtype=torch.int32, device=dev)
            wa = torch.empty(cap + 1, dtype=torch.int32, device=dev)
            wf = torch.zeros(cap + 1, dtype=torch.int8, device=dev)
            nw = torch.zeros(1, dtype=torch.int32, device=dev)
            _lib.check(lib.dmpnn_work_table_build(self.tile_row_ptr.data_ptr(), self.tile_atom_ptr.data_ptr(), self.n_tiles,
                                                  wr.data_ptr(), wa.data_ptr(), wf.data_ptr(), nw.data_ptr(), _stream()),
                       "dmpnn_work_table_build")
            self._work = (wr, wa, wf, nw)
        wr, wa, wf, nw = self._work
        return wr, wa, self.n_tiles, wf, nw, self.dst_row


def check_flags(f: int):
    if not f & _lib.FLAG_INDEX_IN_RANGE:
        raise DmpnnError("BatchMolGraph indices out of range (edge_index / rev_edge_index / batch)")
    if not f & _lib.FLAG_BATCH_SORTED:
        raise DmpnnError("BatchMolGraph.batch must be non-decreasing and edges must stay inside a molecule")
    if not f & _lib.FLAG_REV_INVOLUTION:
        raise DmpnnError(
            "rev_edge_index is not a proper reverse-edge map (rev[rev[e]]==e with swapped endpoints); "
            "the engine requires it (every featuriser-made graph satisfies it)"
        )


def build_layout(edge_index: Tensor, rev_edge_index: Tensor, batch: Tensor, n_mols: int,
                 meta_host: list | None = None) -> Layout:
    """dmpnn_layout_build on the current stream.  Inputs are the reference's int64 index tensors.
    `meta_host`: the meta words already computed on the host for this very batch (dmpnn_batch_meta_host, by our
    collate): the layout then never reads `meta` back from the device -- no sync in the training step."""
    _require_cuda(edge_index, rev_edge_index, batch)
    lib = _lib.load()
    dev = edge_index.device
    edge_index = edge_index.contiguous()
    rev_edge_index = rev_edge_index.contiguous()
    batch = batch.contiguous()
    if edge_index.dtype != torch.int64 or rev_edge_index.dtype != torch.int64 or batch.dtype != torch.int64:
        raise DmpnnError("edge_index / rev_edge_index / batch must be int64 (as in the reference BatchMolGraph)")
    E = int(edge_index.shape[1])
    V = int(batch.shape[0])
    B = int(n_mols)
    i32 = dict(dtype=torch.int32, device=dev)
    perm = torch.empty(max(E, 1), **i32)
    inv_perm = torch.empty(max(E, 1), **i32)
    rowptr = torch.empty(V + 1, **i32)
    src_row = torch.empty(max(E, 1), **i32)
    dst_row = torch.empty(max(E, 1), **i32)
    rev_row = torch.empty(max(E, 1), **i32)
    # the zero-initialised outputs are views of ONE buffer (one memset instead of six fill launches per step)
    sizes = (B + 1, B + 1, B + 2, B + 2, B + 2, _lib.META_WORDS)
    zbuf = torch.zeros(sum(sizes), **i32)
    mol_atom_ptr, mol_row_ptr, tile_mol_ptr, tile_row_ptr, tile_atom_ptr, meta = torch.split(zbuf, sizes)
    nbytes = C.c_size_t(0)
    _lib.check(lib.dmpnn_layout_workspace_bytes(V, E, B, C.byref(nbytes)), "dmpnn_layout_workspace_bytes")
    ws = torch.empty(max(nbytes.value, 256), dtype=torch.uint8, device=dev)
    rc = lib.dmpnn_layout_build(
        edge_index.data_ptr(), rev_edge_index.data_ptr(), batch.data_ptr(), V, E, B,
        perm.data_ptr(), inv_perm.data_ptr(), rowptr.data_ptr(), src_row.data_ptr(), dst_row.data_ptr(),
        rev_row.data_ptr(), mol_atom_ptr.data_ptr(), mol_row_ptr.data_ptr(), tile_mol_ptr.data_ptr(),
        tile_row_ptr.data_ptr(), tile_atom_ptr.data_ptr(), meta.data_ptr(), ws.data_ptr(), _stream(),
    )
    _lib.check(rc, "dmpnn_layout_build")
    return Layout(V, E, B, perm[:E], inv_perm[:E], rowptr, src_row[:E], dst_row[:E], rev_row[:E], mol_atom_ptr,
                  mol_row_ptr, tile_mol_ptr, tile_row_ptr, tile_atom_ptr, meta,
                  None if meta_host is None else list(meta_host))


def get_layout(bmg) -> Layout:
    """Layout of a BatchMolGraph (ours or the reference's), cached on the object when it allows it."""
    lay = getattr(bmg, "_layout", None)
    if lay is not None and lay.rowptr.device == bmg.edge_index.device:
        return lay
    meta_host = getattr(bmg, "_meta_host", None) if HOST_META else None
    if meta_host is not None:
        check_flags(meta_host[_lib.META_FLAGS])      # an invalid batch is refused before anything is launched
        lay = build_layout(bmg.edge_index, bmg.rev_edge_index, bmg.batch, len(bmg), meta_host)
    else:
        lay = build_layout(bmg.edge_index, bmg.rev_edge_index, bmg.batch, len(bmg))
    lay.validate()
    try:
        bmg._layout = lay
    except AttributeError:  # reference BatchMolGraph is a slots dataclass: rebuild per call
        pass
    # let Aggregation.forward(H, bmg.batch) find the molecule offsets without a device sync
    try:
        bt = bmg.batch
        bt._dmpnn_seg, bt._dmpnn_seg_v = (lay.mol_atom_ptr, bt.to(torch.int32), lay.B), bt._version
    except Exception:
        pass
    return lay


def segments_of(batch: Tensor, n_seg: int | None = None):
    """(ptr int32 [B+1], seg_of_row int32 [V], B) for a sorted int64 `batch` (agg.py:74-75).  `n_seg`: the segment count
    is given by the caller (nn/ffn.py:123 sizes by the constraints' rows): trailing segments without rows come out empty
    (`ptr[s] == ptr[s+1]`), an index >= n_seg is an error."""
    seg = getattr(batch, "_dmpnn_seg", None)          # attached by get_layout / an earlier call; void after an in-place change
    if (seg is not None and getattr(batch, "_dmpnn_seg_v", None) == batch._version and seg[0].device == batch.device
            and (n_seg is None or seg[2] == n_seg)):
        return seg
    _require_cuda(batch)
    lib = _lib.load()
    n = int(batch.shape[0])
    if n_seg is None:
        B = int(batch.max().item()) + 1 if n > 0 else 0   # same device sync as the reference (agg.py:75)
    else:
        B = int(n_seg)
    ptr = torch.zeros(B + 1, dtype=torch.int32, device=batch.device)
    status = torch.zeros(1, dtype=torch.int32, device=batch.device)
    bc = batch.contiguous()
    _lib.check(lib.dmpnn_sorted_index_to_ptr(bc.data_ptr(), n, B, ptr.data_ptr(), status.data_ptr(), _stream()),
               "dmpnn_sorted_index_to_ptr")
    st = int(status.item())
    if st & 1:       # V_RANGE of csrc/layout.cu
        raise DmpnnError(f"`batch` holds a molecule index outside [0, {B})")
    if st != 0:
        raise DmpnnError("Aggregation: `batch` must be non-decreasing (atoms of a molecule contiguous)")
    seg = (ptr, bc.to(torch.int32), B)
    if n_seg is None:
        try:
            batch._dmpnn_seg, batch._dmpnn_seg_v = seg, batch._version
        except Exception:
            pass
    return seg


# ----------------------------------------------------------------------------------------------
# op wrappers (tensors in, launches on the current stream)
# ----------------------------------------------------------------------------------------------
def linear_fwd(X1: Tensor, K1: int, W: Tensor, out: Tensor, N: int, *, idx1: Tensor | None = None,
               X2: Tensor | None = None, K2: int = 0, idx2: Tensor | None = None, bias: Tensor | None = None,
               res: Tensor | None = None, act: int = ACT_NONE, act_param: float = 0.0, R: int | None = None,
               pad_to: int | None = None):
    lib = _lib.load()
    R = out.shape[0] if R is None else R
    assert W.dtype == torch.float32 and (W.stride(1) == 1 or W.shape[1] == 1) and W.shape[0] == N and W.shape[1] == K1 + K2
    rc = lib.dmpnn_linear_fwd(
        X1.data_ptr(), _dt(X1), _ld(X1), _ptr(idx1), K1,
        _ptr(X2), _dt(X2) if X2 is not None else F32, _ld(X2) if X2 is not None else 0, _ptr(idx2), K2,
        W.data_ptr(), W.stride(0), _ptr(bias),
        _ptr(res), _dt(res) if res is not None else F32, _ld(res) if res is not None else 0,
        act, float(act_param), out.data_ptr(), _dt(out), _ld(out), pad_to if pad_to is not None else min(_ld(out), out.shape[1]),
        R, N, _stream(),
    )
    _lib.check(rc, "dmpnn_linear_fwd")


def linear_wgrad(dY: Tensor, X1: Tensor, K1: int, dW: Tensor, N: int, *, idx1: Tensor | None = None,
                 X2: Tensor | None = None, K2: int = 0, idx2: Tensor | None = None, dbias: Tensor | None = None,
                 accumulate: bool = False, R: int | None = None):
    lib = _lib.load()
    R = dY.shape[0] if R is None else R
    assert dW.dtype == torch.float32 and dW.stride(1) == 1
    nbytes = C.c_size_t(0)
    _lib.check(lib.dmpnn_linear_wgrad_workspace_bytes(R, N, K1 + K2, C.byref(nbytes)), "wgrad_workspace_bytes")
    ws = torch.empty(nbytes.value, dtype=torch.uint8, device=dY.device)
    rc = lib.dmpnn_linear_wgrad(
        dY.data_ptr(), _dt(dY), _ld(dY), X1.data_ptr(), _dt(X1), _ld(X1), _ptr(idx1), K1,
        _ptr(X2), _dt(X2) if X2 is not None else F32, _ld(X2) if X2 is not None else 0, _ptr(idx2), K2,
        dW.data_ptr(), dW.stride(0), _ptr(dbias), 1 if accumulate else 0, R, N, ws.data_ptr(), _stream(),
    )
    _lib.check(rc, "dmpnn_linear_wgrad")


def segment_sum(X: Tensor, ptr: Tensor, n_seg: int, Ccols: int, out: Tensor, *, idx: Tensor | None = None,
                act: int = ACT_NONE, act_param: float = 0.0, scale_mode: int = SCALE_NONE, scale: float = 1.0,
                pad_to: int | None = None):
    lib = _lib.load()
    rc = lib.dmpnn_segment_sum(
        X.data_ptr(), _dt(X), _ld(X), _ptr(idx), ptr.data_ptr(), n_seg, Ccols, act, float(act_param),
        scale_mode, float(scale), out.data_ptr(), _dt(out), _ld(out),
        pad_to if pad_to is not None else min(_ld(out), out.shape[1]), _stream(),
    )
    _lib.check(rc, "dmpnn_segment_sum")


def segment_bcast(G: Tensor, seg_of_row: Tensor, ptr: Tensor | None, R: int, Ccols: int, out: Tensor, *,
                  scale_mode: int = SCALE_NONE, scale: float = 1.0, n_seg: int = 0):
    """n_seg > 0: rows of segment s are [ptr[s], ptr[s+1]) -- walk segments instead of looking every row up."""
    lib = _lib.load()
    rc = lib.dmpnn_segment_bcast(G.data_ptr(), _dt(G), _ld(G), seg_of_row.data_ptr(), _ptr(ptr),
                                 n_seg if ptr is not None else 0, R, Ccols,
                                 scale_mode, float(scale), out.data_ptr(), _dt(out), _ld(out), _stream())
    _lib.check(rc, "dmpnn_segment_bcast")


def bond_message(X: Tensor, lay: Layout, Ccols: int, out: Tensor, *, act: int = ACT_NONE, act_param: float = 0.0,
                 permute_on_read: bool = False):
    lib = _lib.load()
    if lay.E == 0:
        return
    rc = lib.dmpnn_bond_message(X.data_ptr(), _dt(X), _ld(X), lay.rowptr.data_ptr(), lay.rev_row.data_ptr(),
                                lay.V, Ccols, act, float(act_param), 1 if permute_on_read else 0,
                                out.data_ptr(), _dt(out), _ld(out), _stream())
    _lib.check(rc, "dmpnn_bond_message")


def rev_average(X: Tensor, lay: Layout, Ccols: int, out: Tensor, *, act: int = ACT_NONE, act_param: float = 0.0):
    lib = _lib.load()
    if lay.E == 0:
        return
    rc = lib.dmpnn_rev_average(X.data_ptr(), _dt(X), _ld(X), lay.rev_row.data_ptr(), lay.E, Ccols, act,
                               float(act_param), out.data_ptr(), _dt(out), _ld(out), _stream())
    _lib.check(rc, "dmpnn_rev_average")


def act_bwd(G: Tensor, Yact: Tensor, R: int, Ccols: int, *, act: int, act_param: float = 0.0,
            gidx: Tensor | None = None, from_preact: bool = False, dZ: Tensor | None = None,
            acc: Tensor | None = None):
    lib = _lib.load()
    if R == 0:
        return
    rc = lib.dmpnn_act_bwd(
        G.data_ptr(), _dt(G), _ld(G), _ptr(gidx), Yact.data_ptr(), _dt(Yact), _ld(Yact),
        1 if from_preact else 0, act, float(act_param),
        _ptr(dZ), _dt(dZ) if dZ is not None else F32, _ld(dZ) if dZ is not None else 0,
        _ptr(acc), _dt(acc) if acc is not None else F32, _ld(acc) if acc is not None else 0,
        R, Ccols, _stream(),
    )
    _lib.check(rc, "dmpnn_act_bwd")


# ----------------------------------------------------------------------------------------------
# message passing: forward / backward drivers
# ----------------------------------------------------------------------------------------------
@dataclass
class MPConfig:
    depth: int
    act: int
    act_param: float
    undirected: bool
    hidden_dtype: torch.dtype  # torch.float32 (<=1e-5 tier) or torch.bfloat16 (<=1e-2 tier)
    fused: bool = True         # use the tcgen05 fused depth-step kernel when applicable
    dropout_p: float = 0.0     # > 0: training-mode dropout on the fused bf16 / ReLU path (dropout_fused_ok)
    mask_fn: object = None     # keep-mask source `f(like) -> {0,1} tensor like `like``; None = torch's bernoulli_


def _hidden(rows: int, hp: int, dtype, dev) -> Tensor:
    return torch.zeros((max(rows, 1), hp), dtype=dtype, device=dev)


UNDIRECTED_FUSED = os.environ.get("DMPNN_UNDIRECTED_FUSED", "1") != "0"   # DMPNN_UNDIRECTED_FUSED=0: A/B switch (message + GEMM launches)


def _fused_step_ok(cfg: MPConfig, lay: Layout, h: int) -> bool:
    """The fused tcgen05 depth step applies: bf16 tier, h <= 304.  Molecules of any size: those with more than 128 directed
    edges run as 128-row windows of the same kernel (Layout.step_tables).  `undirected=True` (base.py:202-203) runs on it too:
    the reverse-edge average is a prologue pass that produces the step's input (bond_forward)."""
    ok = (cfg.fused and cfg.hidden_dtype == torch.bfloat16 and h <= 304 and lay.E > 0 and (not cfg.undirected or (UNDIRECTED_FUSED and h % 4 == 0))
          and _fused_available())
    if not ok and cfg.fused and cfg.hidden_dtype == torch.bfloat16 and lay.E > 0:
        _warn_once("unfused", "chemprop_b200: this batch leaves the fused depth-step kernel (" +
                   (f"d_h = {h} > 304" if h > 304 else "undirected=True with d_h % 4 != 0" if cfg.undirected else
                    "kernel unavailable") + "): the depth loop runs as separate message + GEMM launches")
    return ok


_WARNED: set = set()


def _warn_once(key: str, msg: str):
    if key not in _WARNED:
        _WARNED.add(key)
        import warnings

        warnings.warn(msg, RuntimeWarning, stacklevel=3)


_FUSED_STATE: dict = {}


def _fused_available() -> bool:
    if "ok" not in _FUSED_STATE:
        lib = _lib.load()
        n = C.c_size_t(0)
        _FUSED_STATE["ok"] = lib.dmpnn_pack_weight_bf16_bytes(304, 304, C.byref(n)) == 0
    return _FUSED_STATE["ok"]


def pack_weight_bf16(W: Tensor) -> Tensor:
    lib = _lib.load()
    N, K = W.shape
    n = C.c_size_t(0)
    _lib.check(lib.dmpnn_pack_weight_bf16_bytes(N, K, C.byref(n)), "dmpnn_pack_weight_bf16_bytes")
    out = torch.empty(n.value, dtype=torch.uint8, device=W.device)
    Wc = W.detach().contiguous().float()
    _lib.check(lib.dmpnn_pack_weight_bf16(Wc.data_ptr(), Wc.stride(0), N, K, out.data_ptr(), _stream()),
               "dmpnn_pack_weight_bf16")
    return out


def pack_weight_tc(W: Tensor, transpose: bool = False) -> Tensor:
    """Pack an nn.Linear weight (N x K; or, with transpose, a K x N matrix used as B[n][k] = W[k][n]) for
    dmpnn_linear_tc_bf16."""
    lib = _lib.load()
    Wc = W.detach().float()
    if Wc.stride(1) != 1:
        Wc = Wc.contiguous()
    N, K = (Wc.shape[1], Wc.shape[0]) if transpose else (Wc.shape[0], Wc.shape[1])
    n = C.c_size_t(0)
    _lib.check(lib.dmpnn_pack_weight_tc_bytes(N, K, C.byref(n)), "dmpnn_pack_weight_tc_bytes")
    out = torch.empty(n.value, dtype=torch.uint8, device=W.device)
    _lib.check(lib.dmpnn_pack_weight_tc(Wc.data_ptr(), Wc.stride(0), N, K, 1 if transpose else 0, out.data_ptr(),
                                        _stream()), "dmpnn_pack_weight_tc")
    return out


def linear_tc(A: Tensor, K: int, Wpk: Tensor, N: int, out: Tensor, *, bias: Tensor | None = None,
              res: Tensor | None = None, act: int = ACT_NONE, act_param: float = 0.0, R: int | None = None):
    """out = act(A[:, :K] . W^T + bias + res) on the tensor cores (bf16 operands, f32 accumulate)."""
    lib = _lib.load()
    R = out.shape[0] if R is None else R
    assert A.dtype == torch.bfloat16 and out.dtype == torch.bfloat16 and (res is None or res.dtype == torch.bfloat16)
    rc = lib.dmpnn_linear_tc_bf16(A.data_ptr(), _ld(A), R, K, Wpk.data_ptr(), N, _ptr(bias), _ptr(res),
                                  _ld(res) if res is not None else 0, act, float(act_param),
                                  out.data_ptr(), _ld(out), _stream())
    _lib.check(rc, "dmpnn_linear_tc_bf16")


def wgrad_tc(dY: Tensor, X: Tensor, R: int, N: int, K: int, dW: Tensor, *, accumulate: bool = False):
    """dW[n, :K] (+)= sum_r dY[r, n] X[r, :K] on the tensor cores (bf16 operands)."""
    lib = _lib.load()
    assert dY.dtype == torch.bfloat16 and X.dtype == torch.bfloat16 and dW.dtype == torch.float32
    n = C.c_size_t(0)
    _lib.check(lib.dmpnn_wgrad_tc_workspace_bytes(N, K, C.byref(n)), "dmpnn_wgrad_tc_workspace_bytes")
    ws = torch.empty(n.value, dtype=torch.uint8, device=dW.device)
    rc = lib.dmpnn_wgrad_tc_bf16(dY.data_ptr(), _ld(dY), X.data_ptr(), _ld(X), R, N, K, dW.data_ptr(), dW.stride(0),
                                 1 if accumulate else 0, ws.data_ptr(), _stream())
    _lib.check(rc, "dmpnn_wgrad_tc_bf16")


def wgrad_tc_multi(dYs: list, X: Tensor, R: int, N: int, K: int, dW: Tensor, *, accumulate: bool = False):
    """dW[n, :K] (+)= sum_t sum_r dY_t[r, n] X[r, :K]: up to three terms per launch share the X stream; longer lists are
    issued in groups, accumulating."""
    lib = _lib.load()
    nxb = ((K + 15) // 16 * 16 + 63) // 64             # X boxes of a stage (csrc/wgrad_tc.cu: 2 * terms + nxb <= 9)
    per = max(1, min(3, (9 - nxb) // 2))
    n = C.c_size_t(0)
    _lib.check(lib.dmpnn_wgrad_tc_workspace_bytes(N, K, C.byref(n)), "dmpnn_wgrad_tc_workspace_bytes")
    ws = torch.empty(n.value, dtype=torch.uint8, device=dW.device)
    for i in range(0, len(dYs), per):
        grp = dYs[i:i + per]
        assert all(t.dtype == torch.bfloat16 and _ld(t) == _ld(grp[0]) for t in grp) and X.dtype == torch.bfloat16
        arr = (C.c_void_p * len(grp))(*[t.data_ptr() for t in grp])
        rc = lib.dmpnn_wgrad_tc_multi_bf16(C.cast(arr, C.c_void_p), len(grp), _ld(grp[0]), X.data_ptr(), _ld(X), R, N, K,
                                           dW.data_ptr(), dW.stride(0), 1 if (accumulate or i > 0) else 0, ws.data_ptr(), _stream())
        _lib.check(rc, "dmpnn_wgrad_tc_multi_bf16")


# ---- fp32-accurate tensor-core GEMMs (3xTF32, csrc/gemm_x3.cu) -------------------------------------------------
X3_ENABLED = os.environ.get("DMPNN_X3", "1") != "0"          # DMPNN_X3=0: A/B switch (fp32 tier on the SIMT f32 GEMMs)


def _x3_ok(cfg: "MPConfig", *dims: int) -> bool:
    """fp32 tier on the tensor cores: f32 hidden states, fused kernels enabled, every GEMM dimension a multiple of 4
    (16-byte operand rows)."""
    return (X3_ENABLED and cfg.fused and cfg.hidden_dtype == torch.float32 and all(d % 4 == 0 and 0 < d <= 4096 for d in dims)
            and _fused_available())


def pack_weight_x3(W: Tensor, transpose: bool = False) -> Tensor:
    """nn.Linear weight (N x K; with transpose: a K x N matrix used as B[n][k] = W[k][n]) split into tf32 hi / lo parts and
    laid out for dmpnn_linear_x3."""
    lib = _lib.load()
    Wc = W.detach()
    if Wc.dtype != torch.float32 or Wc.stride(1) != 1:
        Wc = Wc.float().contiguous()
    N, K = (Wc.shape[1], Wc.shape[0]) if transpose else (Wc.shape[0], Wc.shape[1])
    n = C.c_size_t(0)
    _lib.check(lib.dmpnn_pack_weight_x3_bytes(N, K, C.byref(n)), "dmpnn_pack_weight_x3_bytes")
    out = torch.empty(n.value, dtype=torch.uint8, device=W.device)
    _lib.check(lib.dmpnn_pack_weight_x3(Wc.data_ptr(), Wc.stride(0), N, K, 1 if transpose else 0, out.data_ptr(), _stream()),
               "dmpnn_pack_weight_x3")
    return out


def linear_x3(A: Tensor, K: int, Wpk: Tensor, N: int, out: Tensor, *, idx: Tensor | None = None, bias: Tensor | None = None,
              res: Tensor | None = None, act: int = ACT_NONE, act_param: float = 0.0, R: int | None = None,
              pad_to: int | None = None):
    """out[:, :N] = act(A[idx][:, :K] . W^T + bias + res) with f32 accuracy on the tensor cores; columns [N, pad_to) zeroed."""
    lib = _lib.load()
    R = out.shape[0] if R is None else R
    assert A.dtype == torch.float32 and out.dtype == torch.float32 and (res is None or res.dtype == torch.float32)
    pad_to = min(_ld(out), out.shape[1]) if pad_to is None else pad_to
    rc = lib.dmpnn_linear_x3(A.data_ptr(), _ld(A), _ptr(idx), R, K, Wpk.data_ptr(), N, _ptr(bias), _ptr(res),
                             _ld(res) if res is not None else 0, act, float(act_param), out.data_ptr(), _ld(out),
                             max(N, min(pad_to, (N + 15) // 16 * 16)), _stream())
    _lib.check(rc, "dmpnn_linear_x3")


def wgrad_x3(dY: Tensor, X: Tensor, R: int, N: int, K: int, dW: Tensor, *, accumulate: bool = False):
    """dW[n, :K] (+)= sum_r dY[r, n] X[r, :K] with f32 accuracy on the tensor cores."""
    lib = _lib.load()
    assert dY.dtype == torch.float32 and X.dtype == torch.float32 and dW.dtype == torch.float32
    n = C.c_size_t(0)
    _lib.check(lib.dmpnn_wgrad_x3_workspace_bytes(N, K, C.byref(n)), "dmpnn_wgrad_x3_workspace_bytes")
    ws = torch.empty(n.value, dtype=torch.uint8, device=dW.device)
    rc = lib.dmpnn_wgrad_x3(dY.data_ptr(), _ld(dY), X.data_ptr(), _ld(X), R, N, K, dW.data_ptr(), dW.stride(0),
                            1 if accumulate else 0, ws.data_ptr(), _stream())
    _lib.check(rc, "dmpnn_wgrad_x3")


# ---- molecule-level head (csrc/head.cu) ------------------------------------------------------------------------
def bn_train_fwd(X: Tensor, gamma, beta, running_mean, running_var, eps: float, momentum: float, Y: Tensor, Xhat: Tensor,
                 mean: Tensor, invstd: Tensor):
    lib = _lib.load()
    B, d = X.shape
    rc = lib.dmpnn_bn_train_fwd(X.data_ptr(), X.stride(0), B, d, _ptr(gamma), _ptr(beta), float(eps), float(momentum),
                                _ptr(running_mean), _ptr(running_var), Y.data_ptr(), Y.stride(0), Xhat.data_ptr(),
                                Xhat.stride(0), mean.data_ptr(), invstd.data_ptr(), _stream())
    _lib.check(rc, "dmpnn_bn_train_fwd")


def bn_bwd(dY: Tensor, Xhat: Tensor, gamma, invstd: Tensor, dX: Tensor, dgamma, dbeta):
    lib = _lib.load()
    B, d = dY.shape
    rc = lib.dmpnn_bn_bwd(dY.data_ptr(), dY.stride(0), Xhat.data_ptr(), Xhat.stride(0), B, d, _ptr(gamma), invstd.data_ptr(),
                          dX.data_ptr(), dX.stride(0), _ptr(dgamma), _ptr(dbeta), _stream())
    _lib.check(rc, "dmpnn_bn_bwd")


def mse_loss(P: Tensor, Y: Tensor, w, tw, loss: Tensor, dP: Tensor):
    lib = _lib.load()
    B, T = P.shape
    rc = lib.dmpnn_mse_loss(P.data_ptr(), P.stride(0) if B else T, Y.data_ptr(), Y.stride(0) if B else T, _ptr(w), _ptr(tw), B, T,
                            loss.data_ptr(), dP.data_ptr(), dP.stride(0) if B else T, _stream())
    _lib.check(rc, "dmpnn_mse_loss")


def bce_loss(P: Tensor, Y: Tensor, w, tw, loss: Tensor, dP: Tensor):
    """BCE with logits, P / Y / dP: B x T (dmpnn_bce_loss)."""
    _require_cuda(P, Y, w, tw, loss, dP)
    lib = _lib.load()
    B, T = P.shape
    rc = lib.dmpnn_bce_loss(P.data_ptr(), P.stride(0) if B else T, Y.data_ptr(), Y.stride(0) if B else T, _ptr(w), _ptr(tw), B, T,
                            loss.data_ptr(), dP.data_ptr(), dP.stride(0) if B else T, _stream())
    _lib.check(rc, "dmpnn_bce_loss")


def ce_loss(P: Tensor, Y: Tensor, w, tw, loss: Tensor, dP: Tensor, C: int):
    """Cross entropy over groups of C logits, P / dP: B x (T C), Y: B x T class ids (dmpnn_ce_loss)."""
    _require_cuda(P, Y, w, tw, loss, dP)
    lib = _lib.load()
    B, T = Y.shape
    TC = T * C
    rc = lib.dmpnn_ce_loss(P.data_ptr(), P.stride(0) if B else TC, Y.data_ptr(), Y.stride(0) if B else T, _ptr(w), _ptr(tw), B, T,
                           C, loss.data_ptr(), dP.data_ptr(), dP.stride(0) if B else TC, _stream())
    _lib.check(rc, "dmpnn_ce_loss")


def class_probs(P: Tensor, C: int, Q: Tensor):
    """Q = sigmoid(P) (C == 1) or the softmax of each group of C columns, P / Q: B x (T C) (dmpnn_class_probs)."""
    _require_cuda(P, Q)
    lib = _lib.load()
    B, TC = P.shape
    rc = lib.dmpnn_class_probs(P.data_ptr(), P.stride(0) if B else TC, B, TC // C, C, Q.data_ptr(), Q.stride(0) if B else TC,
                               _stream())
    _lib.check(rc, "dmpnn_class_probs")


def class_probs_bwd(Q: Tensor, dQ: Tensor, C: int, dP: Tensor):
    """dP from the saved probabilities Q and the upstream dQ (dmpnn_class_probs_bwd)."""
    _require_cuda(Q, dQ, dP)
    lib = _lib.load()
    B, TC = Q.shape
    rc = lib.dmpnn_class_probs_bwd(Q.data_ptr(), Q.stride(0) if B else TC, dQ.data_ptr(), dQ.stride(0) if B else TC, B, TC // C, C,
                                   dP.data_ptr(), dP.stride(0) if B else TC, _stream())
    _lib.check(rc, "dmpnn_class_probs_bwd")


def column_sum(Y: Tensor, R: int, N: int, out: Tensor, *, accumulate: bool = False):
    lib = _lib.load()
    n = C.c_size_t(0)
    _lib.check(lib.dmpnn_linear_wgrad_workspace_bytes(R, N, 1, C.byref(n)), "wgrad_workspace_bytes")
    ws = torch.empty(n.value, dtype=torch.uint8, device=out.device)
    rc = lib.dmpnn_column_sum(Y.data_ptr(), _dt(Y), _ld(Y), R, N, out.data_ptr(), 1 if accumulate else 0,
                              ws.data_ptr(), _stream())
    _lib.check(rc, "dmpnn_column_sum")


def bond_message_bwd_masked(dM: Tensor, Yact: Tensor, lay: Layout, Ccols: int, out: Tensor, *, act: int,
                            act_param: float = 0.0):
    lib = _lib.load()
    if lay.E == 0:
        return
    rc = lib.dmpnn_bond_message_bwd_masked(dM.data_ptr(), _dt(dM), _ld(dM), lay.rowptr.data_ptr(),
                                           lay.rev_row.data_ptr(), lay.V, Ccols, Yact.data_ptr(), _ld(Yact), act,
                                           float(act_param), out.data_ptr(), _ld(out), _stream())
    _lib.check(rc, "dmpnn_bond_message_bwd_masked")


def sum_act_bwd(Zs: list, G: Tensor | None, Ypre: Tensor | None, out: Tensor, R: int, Ccols: int, *, act: int,
                act_param: float = 0.0):
    """out = sum(Zs) + G * tau'(Ypre) in one pass (<= 8 addends per call; longer lists are folded)."""
    lib = _lib.load()
    if R == 0:
        return
    Zs = list(Zs)
    while len(Zs) > 8:   # fold the first eight into one buffer
        tmp = torch.empty_like(Zs[0])
        sum_act_bwd(Zs[:8], None, None, tmp, R, Ccols, act=act, act_param=act_param)
        Zs = [tmp] + Zs[8:]
    ref = Zs[0] if Zs else G
    arr = (C.c_void_p * 8)(*[z.data_ptr() for z in Zs] + [None] * (8 - len(Zs)))
    rc = lib.dmpnn_sum_act_bwd(C.cast(arr, C.c_void_p), len(Zs), _ld(ref), _ptr(G), _ld(G) if G is not None else 0,
                               _ptr(Ypre), _ld(Ypre) if Ypre is not None else 0, _dt(ref), act, float(act_param),
                               out.data_ptr(), _dt(out), _ld(out), R, Ccols, _stream())
    _lib.check(rc, "dmpnn_sum_act_bwd")


def concat_bf16(X1: Tensor, K1: int, out: Tensor, R: int, *, idx1: Tensor | None = None, X2: Tensor | None = None,
                K2: int = 0, idx2: Tensor | None = None, width: int | None = None):
    lib = _lib.load()
    width = out.shape[1] if width is None else width
    rc = lib.dmpnn_concat_bf16(X1.data_ptr(), _dt(X1), _ld(X1), _ptr(idx1), K1,
                               _ptr(X2), _dt(X2) if X2 is not None else F32, _ld(X2) if X2 is not None else 0,
                               _ptr(idx2), K2, out.data_ptr(), _ld(out), width, R, _stream())
    _lib.check(rc, "dmpnn_concat_bf16")


def dropout_keep_bits(rows: int, h: int, cfg: "MPConfig", like: Tensor) -> Tensor:
    """uint16 [rows, pad16(h) / 16] keep bits for one dropout site of the fused path (dmpnn_dropout_bits: Philox4x32-10 keyed
    by the device generator's seed and current offset, so `torch.manual_seed` governs the masks as in the reference; the
    offset is then advanced).  `cfg.mask_fn` (test hook) supplies a {0, 1} tensor instead, which is packed into the same words."""
    nj = (h + 15) // 16
    dev = like.device
    if cfg.mask_fn is not None:
        M = cfg.mask_fn(like)[:rows, : nj * 16].to(torch.int32).reshape(rows, nj, 16)
        w = (M << torch.arange(16, device=dev, dtype=torch.int32)).sum(-1)
        return w.to(torch.uint16).contiguous()
    if torch.cuda.is_current_stream_capturing():
        raise DmpnnError("training-mode dropout inside a captured CUDA graph is not supported (the Philox offset is host state)")
    lib = _lib.load()
    gen = torch.cuda.default_generators[dev.index if dev.index is not None else torch.cuda.current_device()]
    seed, off = int(gen.initial_seed()) & (2 ** 64 - 1), int(gen.get_offset())
    gen.set_offset(off + 4)
    bits = torch.empty((max(rows, 1), nj), dtype=torch.uint16, device=dev)
    _lib.check(lib.dmpnn_dropout_bits(bits.data_ptr(), rows, nj, float(cfg.dropout_p), seed, off, _stream()), "dmpnn_dropout_bits")
    return bits


def concat_f32(X1: Tensor, K1: int, out: Tensor, R: int, *, idx1: Tensor | None = None, X2: Tensor | None = None,
               K2: int = 0, idx2: Tensor | None = None, width: int | None = None):
    lib = _lib.load()
    width = out.shape[1] if width is None else width
    assert out.dtype == torch.float32
    rc = lib.dmpnn_concat_f32(X1.data_ptr(), _dt(X1), _ld(X1), _ptr(idx1), K1,
                              _ptr(X2), _dt(X2) if X2 is not None else F32, _ld(X2) if X2 is not None else 0,
                              _ptr(idx2), K2, out.data_ptr(), _ld(out), width, R, _stream())
    _lib.check(rc, "dmpnn_concat_f32")


def bond_step_fused(H_prev: Tensor, H0: Tensor, H_next: Tensor, h: int, Wpk: Tensor, bias: Tensor | None,
                    lay: Layout, act: int, act_param: float, first_step: bool, M_out: Tensor | None = None,
                    drop_bits: Tensor | None = None, drop_scale: float = 1.0):
    """One fused depth step; M_out (first step only) also receives the message M^1 the step consumed; `drop_bits`
    (dropout_keep_bits) applies training-mode dropout with scale `drop_scale` in the epilogue."""
    lib = _lib.load()
    trp, tap, nt, wf, nw, dr = lay.step_tables()
    rc = lib.dmpnn_bond_step_fused_bf16(
        H_prev.data_ptr(), H0.data_ptr(), H_next.data_ptr(), _ld(H0), H0.shape[0], h, Wpk.data_ptr(), _ptr(bias),
        lay.rowptr.data_ptr(), lay.rev_row.data_ptr(), trp.data_ptr(), tap.data_ptr(),
        nt, act, float(act_param), 1 if first_step else 0, _ptr(M_out), _ptr(wf), _ptr(nw), _ptr(dr), _ptr(drop_bits),
        float(drop_scale), _stream(),
    )
    _lib.check(rc, "dmpnn_bond_step_fused_bf16")


def h_is_mult4(Wh: Tensor) -> bool:
    return Wh.shape[0] % 4 == 0


def _tc_ok(cfg: MPConfig, h: int, *Ks: int) -> bool:
    """Tensor-core linear kernels apply: bf16 tier, fused kernels enabled, sizes inside the kernel limits."""
    ok = (cfg.fused and cfg.hidden_dtype == torch.bfloat16 and h <= 304 and all(k <= 448 for k in Ks)
          and _fused_available())
    if not ok and cfg.fused and cfg.hidden_dtype == torch.bfloat16 and _fused_available():
        _warn_once("tc_limits", f"chemprop_b200: precision='bf16' with d_h = {h}, GEMM inner dimensions {tuple(Ks)}: outside the "
                   "tensor-core kernels' limits (d_h <= 304, d_v + d_e and d_v + d_h <= 448); the linear layers run on the f32 "
                   "FMA pipes with bf16 storage (the fp32 tier's 3xTF32 tensor-core GEMMs take d_h up to 4096)")
    return ok


def _empty_hidden(rows: int, hp: int, dtype, dev) -> Tensor:
    """Uninitialised hidden buffer: only for producers that write every column below pad16(h)."""
    return torch.empty((max(rows, 1), hp), dtype=dtype, device=dev)


def scale_mask_(X: Tensor, M: Tensor, scale: float):
    """X <- X * M * scale in place over the whole (contiguous) buffer -- dmpnn_scale_mask."""
    lib = _lib.load()
    assert X.is_contiguous() and M.is_contiguous() and X.shape == M.shape and X.dtype == M.dtype
    rc = lib.dmpnn_scale_mask(X.data_ptr(), M.data_ptr(), X.data_ptr(), _dt(X), X.numel(), float(scale), _stream())
    _lib.check(rc, "dmpnn_scale_mask")


def _dropout_(X: Tensor, cfg: MPConfig):
    """nn.Dropout(p) in training mode on a hidden buffer (base.py:139, :182): keep mask from torch's RNG stream (so
    torch.manual_seed governs it, as in the reference), applied with the exact f32 scale 1 / (1 - p)."""
    keep = 1.0 - cfg.dropout_p
    M = cfg.mask_fn(X) if cfg.mask_fn is not None else torch.empty_like(X).bernoulli_(keep)
    scale_mask_(X, M, 1.0 / keep)


def dropout_fused_ok(cfg: MPConfig, lay: Layout, h: int, d_v: int, d_e: int) -> bool:
    """Training-mode dropout can stay on the fused bf16 path: ReLU (tau' of the post-dropout state is the keep mask times
    tau' of the pre-dropout one, so no mask is stored and the scale 1 / (1 - p) folds into the packed weights of the
    mirror), directed bonds, every GEMM on the tensor-core kernels and every depth step on the fused kernel."""
    return (cfg.act == ACT_RELU and not cfg.undirected and lay.E > 0 and h % 4 == 0 and _tc_ok(cfg, h, d_v + d_e, d_v + h)
            and (cfg.depth == 1 or _fused_step_ok(cfg, lay, h)))


def bond_step_bwd_fused(dZ: Tensor, Yact: Tensor | None, dOut: Tensor, h: int, WpkT: Tensor, lay: Layout, act: int,
                        act_param: float, G_out: Tensor | None = None, y_is_preact: bool = False,
                        addends: tuple = ()):
    """dOut = (S.P)(dZ . W_h) [* tau'(Yact)] in one fused launch (WpkT = pack_weight_bf16(W_h.t()));
    G_out also receives (S.P) dZ, the left operand of this step's W_h gradient."""
    lib = _lib.load()
    trp, tap, nt, wf, nw, dr = lay.step_tables()
    rc = lib.dmpnn_bond_step_bwd_fused_bf16(
        dZ.data_ptr(), _ptr(Yact), dOut.data_ptr(), _ld(dZ), dZ.shape[0], h, WpkT.data_ptr(),
        lay.rowptr.data_ptr(), lay.rev_row.data_ptr(), trp.data_ptr(), tap.data_ptr(),
        nt, act, float(act_param), 1 if y_is_preact else 0,
        addends[0].data_ptr() if len(addends) > 0 else None, addends[1].data_ptr() if len(addends) > 1 else None,
        _ptr(G_out), _ptr(wf), _ptr(nw), _ptr(dr), _stream())
    _lib.check(rc, "dmpnn_bond_step_bwd_fused_bf16")


# ---- atom-granular fused step (AtomMessagePassing; the ATOM instantiations of the fused kernel) ------------------------
ATOM_FUSED_ENABLED = os.environ.get("DMPNN_ATOM_FUSED", "1") != "0"      # DMPNN_ATOM_FUSED=0: A/B switch (gather + GEMM launches)
ATOM_TILE_ATOMS, ATOM_TILE_EDGES = 128, 1024


def atom_tables(lay: Layout):
    """(tile_atom_ptr, tile_edge_ptr, n_tiles_dev, n_tiles_max) of the ATOM tiles of a batch: runs of whole molecules with
    <= 128 atoms (and <= 1024 edge rows, what the kernel's staged neighbour table holds), built once per batch on the device
    (dmpnn_tiles_build; the kernel reads the tile count from device memory: no host read-back)."""
    if lay._atom_work is None:
        lib = _lib.load()
        dev = lay.rowptr.device
        i32 = dict(dtype=torch.int32, device=dev)
        ta = torch.empty(lay.B + 2, **i32)
        te = torch.empty(lay.B + 2, **i32)
        info = torch.zeros(4, **i32)
        n = C.c_size_t(0)
        _lib.check(lib.dmpnn_tiles_workspace_bytes(lay.B, C.byref(n)), "dmpnn_tiles_workspace_bytes")
        ws = torch.empty(max(n.value, 16), dtype=torch.uint8, device=dev)
        _lib.check(lib.dmpnn_tiles_build(lay.mol_atom_ptr.data_ptr(), lay.mol_row_ptr.data_ptr(), lay.B, ATOM_TILE_EDGES,
                                         ATOM_TILE_ATOMS, te.data_ptr(), ta.data_ptr(), info.data_ptr(), ws.data_ptr(), _stream()),
                   "dmpnn_tiles_build")
        lay._atom_work = (ta, te, info, max(lay.B, 1))
    return lay._atom_work


def _atom_fused_ok(cfg: MPConfig, lay: Layout, h: int, d_v: int, d_e: int) -> bool:
    """The fused atom step applies: bf16 tier on the tensor-core kernels, directed, depth > 1, no training dropout, and every
    molecule of the batch has <= 128 atoms (an atom tile is a run of whole molecules: max_tile_atoms of the layout exceeds
    128 only for a single oversized molecule)."""
    ok = (ATOM_FUSED_ENABLED and cfg.depth > 1 and not cfg.undirected and cfg.dropout_p == 0 and lay.V > 0 and lay.E > 0
          and _atom_tc_ok(cfg, h, d_v, d_e) and lay.max_tile_atoms <= ATOM_TILE_ATOMS)
    if not ok and ATOM_FUSED_ENABLED and cfg.depth > 1 and lay.E > 0 and _atom_tc_ok(cfg, h, d_v, d_e):
        _warn_once("atom_unfused", "chemprop_b200: this batch leaves the fused atom depth step (" +
                   ("undirected=True" if cfg.undirected else "training dropout" if cfg.dropout_p > 0 else
                    "a molecule with more than 128 atoms") + "): neighbour sum and GEMM run as separate launches")
    return ok


def atom_step_fused(H_prev: Tensor, H0: Tensor, H_next: Tensor, h: int, Wpk: Tensor, bias: Tensor | None, lay: Layout,
                    act: int, act_param: float, first_step: bool, N_out: Tensor | None = None):
    """H_next[v] = act(H0[v] + bias + W . sum_{e in in(v)} g(H_prev[src(e)])) in one launch (dmpnn_atom_step_fused_bf16)."""
    lib = _lib.load()
    ta, te, info, nmax = atom_tables(lay)
    rc = lib.dmpnn_atom_step_fused_bf16(
        H_prev.data_ptr(), H0.data_ptr(), H_next.data_ptr(), _ld(H0), H0.shape[0], h, Wpk.data_ptr(), _ptr(bias),
        lay.rowptr.data_ptr(), lay.src_row.data_ptr(), ta.data_ptr(), te.data_ptr(), info.data_ptr(), nmax, act,
        float(act_param), 1 if first_step else 0, _ptr(N_out), _stream())
    _lib.check(rc, "dmpnn_atom_step_fused_bf16")


def atom_step_bwd_fused(dZ: Tensor, Yact: Tensor | None, dOut: Tensor, h: int, WpkT: Tensor, lay: Layout, act: int,
                        act_param: float, G_out: Tensor | None = None, y_is_preact: bool = False):
    """dOut[v] = ((sum_{e in in(v)} dZ[src(e)]) . W) [* act'(Yact[v])]; G_out also receives the gathered operand."""
    lib = _lib.load()
    ta, te, info, nmax = atom_tables(lay)
    rc = lib.dmpnn_atom_step_bwd_fused_bf16(
        dZ.data_ptr(), _ptr(Yact), dOut.data_ptr(), _ld(dZ), dZ.shape[0], h, WpkT.data_ptr(), lay.rowptr.data_ptr(),
        lay.src_row.data_ptr(), ta.data_ptr(), te.data_ptr(), info.data_ptr(), nmax, act, float(act_param),
        1 if y_is_preact else 0, None, None, _ptr(G_out), _stream())
    _lib.check(rc, "dmpnn_atom_step_bwd_fused_bf16")


def bond_forward(lay: Layout, V: Tensor, E: Tensor, Wi: Tensor, bi, Wh: Tensor, bh, Wo: Tensor, bo,
                 cfg: MPConfig, for_backward: bool = False):
    """BondMessagePassing.forward up to W_o (chemprop/nn/message_passing/base.py:196-212 with
    mixins.py:8-18 and base.py:135-141, 180-182).  Returns (H_v, saved-for-backward)."""
    dev = V.device
    h = Wh.shape[0]
    hp = pad_hidden(h)
    d_v, d_e = V.shape[1], E.shape[1]
    T = cfg.hidden_dtype
    nE, nV = lay.E, lay.V
    a, ap = cfg.act, cfg.act_param
    tc = _tc_ok(cfg, h, d_v + d_e, d_v + h)
    # H_0 = W_i([V[src] || E])   (mixins.py:8-9); rows in dst-sorted order
    if tc and nE > 0:
        kx = (d_v + d_e + 15) // 16 * 16
        X0 = torch.empty((nE, kx), dtype=T, device=dev)
        concat_bf16(V, d_v, X0, nE, idx1=lay.src_row, X2=E, K2=d_e, idx2=lay.perm)
        H0 = _empty_hidden(nE, hp, T, dev)
        linear_tc(X0, d_v + d_e, pack_weight_tc(Wi), h, H0, bias=bi, R=nE)
    elif _x3_ok(cfg, h, d_v + h) and nE > 0:
        # fp32 tier on the tensor cores: [V[src] || E] materialised once in f32 (zero-padded to a multiple of 4 columns),
        # W_i as a 3xTF32 GEMM; the same operand serves the W_i gradient
        X0 = None
        kx4 = (d_v + d_e + 3) // 4 * 4
        X0f = torch.empty((nE, kx4), dtype=torch.float32, device=dev)
        concat_f32(V, d_v, X0f, nE, idx1=lay.src_row, X2=E, K2=d_e, idx2=lay.perm)
        H0 = _hidden(nE, hp, T, dev)
        linear_x3(X0f, kx4, pack_weight_x3(Wi), h, H0, bias=bi, R=nE, pad_to=hp)
    else:
        X0 = None
        H0 = _hidden(nE, hp, T, dev)
        linear_fwd(V, d_v, Wi, H0, h, idx1=lay.src_row, X2=E, K2=d_e, idx2=lay.perm, bias=bi, R=nE, pad_to=hp)
    Hs, Ms, Hbars = [], [], []
    Hprev, first = H0, True  # H^0 = tau(H_0) is applied on load (base.py:200)
    use_fused = cfg.depth > 1 and _fused_step_ok(cfg, lay, h)
    Wpk = pack_weight_bf16(Wh) if use_fused else None
    x3 = _x3_ok(cfg, h, d_v + h)          # fp32 tier: W_h / W_o GEMMs as 3xTF32 on the tensor cores (f32-accurate)
    Wh_x3 = pack_weight_x3(Wh) if (x3 and cfg.depth > 1 and nE > 0) else None
    # bf16 tier off the fused kernel (undirected=True): the W_h GEMM still runs on the tensor cores (k_linear_tc, H_0 residual,
    # bias and tau in its epilogue -- the form AtomMessagePassing's unfused step uses), not on the f32 FMA pipes
    Wh_tc = pack_weight_tc(Wh) if (tc and not use_fused and cfg.depth > 1 and nE > 0) else None
    for _ in range(1, cfg.depth):
        if use_fused:
            Hn = _empty_hidden(nE, hp, T, dev)
            src_in, first_in = Hprev, first
            if cfg.undirected:
                # H~ = (H + H[rev]) / 2 (base.py:202-203) as a prologue pass; the first step's tau(H_0) is applied by it, so the
                # fused step always sees an activation.  H~^{t-1} is kept: it is the right factor of this step's W_h
                # gradient (dZ^T . M^t = ((S.P) dZ)^T . H~^{t-1}, bond_backward).  Zero-filled: the step's TMA boxes read
                # the padding columns up to the 64-column slab edge
                Hbar = _hidden(nE, hp, T, dev)
                rev_average(Hprev, lay, h, Hbar, act=(a if first else ACT_NONE), act_param=ap)
                Hbars.append(Hbar)
                src_in, first_in = Hbar, False
            # training: the first step also stores M^1 (it is tau(H_0)-gathered, which no later kernel can rebuild
            # from a stored activation); the later steps' W_h gradients use (S.P) dZ from the backward kernel instead
            M1 = _empty_hidden(nE, hp, T, dev) if (first_in and for_backward) else None
            # base.py:139 (training-mode dropout): keep bits from Philox, applied in the step's epilogue -- no pass over E x h
            bits = dropout_keep_bits(nE, h, cfg, Hn) if cfg.dropout_p > 0 else None
            with _StepTimer("fused_first" if first else "fused"):
                bond_step_fused(src_in, H0, Hn, h, Wpk, bh, lay, a, ap, first_in, M_out=M1, drop_bits=bits,
                                drop_scale=1.0 / (1.0 - cfg.dropout_p) if bits is not None else 1.0)
            Ms.append(M1)
        else:
            if cfg.dropout_p > 0:
                raise DmpnnError("dropout on the monolithic tier needs the fused depth step (see dropout_fused_ok)")
            src_in, fa = Hprev, (a if first else ACT_NONE)
            if cfg.undirected:  # H = (H + H[rev]) / 2   (base.py:202-203)
                Hbar = _hidden(nE, hp, T, dev)
                rev_average(src_in, lay, h, Hbar, act=fa, act_param=ap)
                Hbars.append(Hbar)
                src_in, fa = Hbar, ACT_NONE
            M = _hidden(nE, hp, T, dev)
            Hn = _hidden(nE, hp, T, dev)
            with _StepTimer("unfused_first" if first else "unfused"):
                bond_message(src_in, lay, h, M, act=fa, act_param=ap)           # mixins.py:11-18
                if Wh_x3 is not None:
                    with _StepTimer("x3_gemm"):
                        linear_x3(M, h, Wh_x3, h, Hn, bias=bh, res=H0, act=a, act_param=ap, R=nE, pad_to=hp)
                elif Wh_tc is not None:
                    linear_tc(M, h, Wh_tc, h, Hn, bias=bh, res=H0, act=a, act_param=ap, R=nE)
                else:
                    linear_fwd(M, h, Wh, Hn, h, bias=bh, res=H0, act=a, act_param=ap, R=nE, pad_to=hp)  # base.py:135-141
            Ms.append(M)
        Hs.append(Hn)
        Hprev, first = Hn, False
    if tc:
        # [V || M_v] assembled once in bf16 (torch.cat of base.py:180), M_v written in place by the segment sum
        hc = (h + 15) // 16 * 16       # zero columns up to pad16(h): 16-byte stores in the segment sum
        ko = (d_v + hc + 1 + 15) // 16 * 16
        XO = torch.empty((max(nV, 1), ko), dtype=T, device=dev)   # columns beyond the K a GEMM asks for are clipped by its TMA descriptor
        concat_bf16(V, d_v, XO, nV, width=d_v)
        Mv = XO[:, d_v:d_v + h]
        segment_sum(Hprev, lay.rowptr, nV, h, Mv, act=(a if first else ACT_NONE), act_param=ap, pad_to=hc)
        ones_col = None
        if for_backward and bo is not None and d_v + hc + 1 <= 448:
            # a column of ones after [V || M_v || 0-pad]: the W_o weight-gradient GEMM over K = d_v + pad16(h) + 1 then delivers
            # the bias gradient (the column sums of dY) as its last column -- no separate column-sum pass over V x h
            ones_col = d_v + hc
            XO[:, ones_col].fill_(1.0)
        Hvp = torch.empty((max(nV, 1), pad_hidden(h)), dtype=T, device=dev)
        linear_tc(XO, d_v + h, pack_weight_tc(Wo), h, Hvp, bias=bo, act=a, act_param=ap, R=nV)
        if cfg.dropout_p > 0:
            _dropout_(Hvp, cfg)                                                    # base.py:182
        Hv = Hvp[:nV, :h]
    else:
        if cfg.dropout_p > 0:
            raise DmpnnError("dropout on the monolithic tier needs the tensor-core path (see dropout_fused_ok)")
        XO = None
        if x3 and nV > 0:
            # [V || M_v] assembled once in f32 (torch.cat of base.py:180): V copied in, M_v written in place by the segment sum
            XO = torch.empty((nV, d_v + h), dtype=T, device=dev)
            XO[:, :d_v].copy_(V)
            Mv = XO[:, d_v:]
            segment_sum(Hprev, lay.rowptr, nV, h, Mv, act=(a if first else ACT_NONE), act_param=ap, pad_to=h)
            Hv = torch.empty((nV, h), dtype=T, device=dev)
            linear_x3(XO, d_v + h, pack_weight_x3(Wo), h, Hv, bias=bo, act=a, act_param=ap, R=nV, pad_to=h)
        else:
            # M_v = sum_{dst(e)=v} H[e]   (base.py:208-211)
            Mv = _hidden(nV, hp, T, dev)
            segment_sum(Hprev, lay.rowptr, nV, h, Mv, act=(a if first else ACT_NONE), act_param=ap, pad_to=hp)
            # H_v = tau(W_o([V || M_v]))   (base.py:180-182)
            Hv = torch.empty((nV, h), dtype=T, device=dev)
            linear_fwd(V, d_v, Wo, Hv, h, X2=Mv, K2=h, bias=bo, act=a, act_param=ap, R=nV, pad_to=h)
    saved = dict(H0=H0, Hs=Hs, Ms=Ms, Hbars=Hbars, Mv=Mv, Hv=Hv, X0=X0, XO=XO, tc=tc, x3=x3, X0f=locals().get("X0f"),
                 ones_col=locals().get("ones_col"))
    return Hv, saved


def bond_backward(lay: Layout, V: Tensor, E: Tensor, Wi: Tensor, Wh: Tensor, Wo: Tensor, cfg: MPConfig,
                  saved: dict, gHv: Tensor, need_bias: tuple[bool, bool, bool]):
    """Hand-written autograd mirror (SURVEY.md 8a-7) of bond_forward.  Returns
    (dWi, dbi, dWh, dbh, dWo, dbo)."""
    dev = V.device
    h = Wh.shape[0]
    hp = pad_hidden(h)
    d_v, d_e = V.shape[1], E.shape[1]
    T = cfg.hidden_dtype
    nE, nV = lay.E, lay.V
    a, ap = cfg.act, cfg.act_param
    H0, Hs, Ms, Hbars, Mv, Hv = saved["H0"], saved["Hs"], saved["Ms"], saved["Hbars"], saved["Mv"], saved["Hv"]
    f32 = dict(dtype=torch.float32, device=dev)
    dWi = torch.zeros_like(Wi, dtype=torch.float32)
    dWh = torch.zeros_like(Wh, dtype=torch.float32)
    dWo = torch.zeros_like(Wo, dtype=torch.float32)
    dbi = torch.zeros(h, **f32) if need_bias[0] else None
    dbh = torch.zeros(h, **f32) if need_bias[1] else None
    dbo = torch.zeros(h, **f32) if need_bias[2] else None
    tc = bool(saved.get("tc"))
    x3 = bool(saved.get("x3")) and saved.get("XO") is not None
    if gHv.stride(1) != 1:
        gHv = gHv.contiguous()
    # readout: dY = g * tau'(Y); dW_o = dY^T [V || M_v]; dM_v = dY . W_o[:, d_v:]
    dY = _hidden(nV, hp, T, dev)
    act_bwd(gHv, Hv, nV, h, act=a, act_param=ap, dZ=dY)
    if tc:
        wgrad_tc(dY, saved["XO"], nV, h, d_v + h, dWo)
        if dbo is not None:
            column_sum(dY, nV, h, dbo)
    elif x3:
        wgrad_x3(dY, saved["XO"], nV, h, d_v + h, dWo)
        if dbo is not None:
            column_sum(dY, nV, h, dbo)
    else:
        linear_wgrad(dY, V, d_v, dWo, h, X2=Mv, K2=h, dbias=dbo, R=nV)
    if tc:
        dMv = _empty_hidden(nV, hp, T, dev)
        linear_tc(dY, h, pack_weight_tc(Wo[:, d_v:], transpose=True), h, dMv, R=nV)
    elif x3:
        dMv = _hidden(nV, hp, T, dev)
        linear_x3(dY, h, pack_weight_x3(Wo[:, d_v:], transpose=True), h, dMv, R=nV, pad_to=hp)
    else:
        WoT = Wo[:, d_v:].t().contiguous()
        dMv = _hidden(nV, hp, T, dev)
        linear_fwd(dY, h, WoT, dMv, h, R=nV, pad_to=hp)
    dH0 = torch.zeros((max(nE, 1), hp), **f32)  # f32 accumulator of dH_0 over all depth steps
    if nE > 0:
        if cfg.depth == 1:
            # dH^0[e] = dM_v[dst(e)];  dH_0 = dH^0 * tau'(H_0)
            act_bwd(dMv, H0, nE, h, act=a, act_param=ap, gidx=lay.dst_row, from_preact=True, acc=dH0)
        else:
            WhT = None if (tc or x3) else Wh.t().contiguous()
            WhT_pk = pack_weight_tc(Wh, transpose=True) if tc else None
            WhT_f = None                                   # W_h^T packed for the fused mirror (undirected fused steps)
            WhT_x3 = pack_weight_x3(Wh, transpose=True) if x3 else None
            dZ = _hidden(nE, hp, T, dev)
            act_bwd(dMv, Hs[-1], nE, h, act=a, act_param=ap, gidx=lay.dst_row, dZ=dZ, acc=dH0)
            for t in range(cfg.depth - 1, 0, -1):
                # inputs of step t: Hin = H^{t-1} (or tau(H_0) when t == 1)
                first = t == 1
                Hin = H0 if first else Hs[t - 2]
                M = Ms[t - 1]
                if M is None and cfg.undirected and tc and _fused_step_ok(cfg, lay, h):
                    # undirected step that ran on the fused kernel: its mirror on the fused kernel too.
                    # dH~^{t-1} = (S.P)(dZ . W_h) = ((S.P) dZ) . W_h, unmasked; the gathered operand G = (S.P) dZ is the left
                    # factor of the W_h gradient (dZ^T . M^t = G^T . H~^{t-1}, H~^{t-1} saved by the forward's prologue);
                    # then the adjoint of the average (self-adjoint) and tau' as in the generic mirror
                    if WhT_f is None:
                        WhT_f = pack_weight_bf16(Wh.t().contiguous())
                    if dbh is not None:
                        column_sum(dZ, nE, h, dbh, accumulate=True)
                    G = _empty_hidden(nE, hp, T, dev)
                    dHbar = _empty_hidden(nE, hp, T, dev)
                    bond_step_bwd_fused(dZ, None, dHbar, h, WhT_f, lay, a, ap, G_out=G)
                    wgrad_tc(G, Hbars[t - 1], nE, h, h, dWh, accumulate=True)
                    dHin = _hidden(nE, hp, T, dev)
                    rev_average(dHbar, lay, h, dHin)
                    if first:
                        act_bwd(dHin, H0, nE, h, act=a, act_param=ap, from_preact=True, acc=dH0)
                    else:
                        dZ = _hidden(nE, hp, T, dev)
                        act_bwd(dHin, Hin, nE, h, act=a, act_param=ap, dZ=dZ, acc=dH0)
                    continue
                if M is None:  # fused forward did not materialise M^t: recompute it
                    M = _hidden(nE, hp, T, dev)
                    if cfg.undirected:
                        bond_message(Hbars[t - 1], lay, h, M)
                    else:
                        bond_message(Hin, lay, h, M, act=(a if first else ACT_NONE), act_param=ap)
                if tc:
                    wgrad_tc(dZ, M, nE, h, h, dWh, accumulate=True)
                    if dbh is not None:
                        column_sum(dZ, nE, h, dbh, accumulate=True)
                elif x3:
                    wgrad_x3(dZ, M, nE, h, h, dWh, accumulate=True)
                    if dbh is not None:
                        column_sum(dZ, nE, h, dbh, accumulate=True)
                else:
                    linear_wgrad(dZ, M, h, dWh, h, dbias=dbh, accumulate=True, R=nE)
                if tc:
                    dM = _empty_hidden(nE, hp, T, dev)
                    linear_tc(dZ, h, WhT_pk, h, dM, R=nE)
                elif x3:
                    dM = _hidden(nE, hp, T, dev)
                    linear_x3(dZ, h, WhT_x3, h, dM, R=nE, pad_to=hp)
                else:
                    dM = _hidden(nE, hp, T, dev)
                    linear_fwd(dZ, h, WhT, dM, h, R=nE, pad_to=hp)
                dHin = _hidden(nE, hp, T, dev)
                bond_message(dM, lay, h, dHin, permute_on_read=True)
                if cfg.undirected:
                    tmp = _hidden(nE, hp, T, dev)
                    rev_average(dHin, lay, h, tmp)
                    dHin = tmp
                if first:
                    act_bwd(dHin, H0, nE, h, act=a, act_param=ap, from_preact=True, acc=dH0)
                else:
                    dZ = _hidden(nE, hp, T, dev)
                    act_bwd(dHin, Hin, nE, h, act=a, act_param=ap, dZ=dZ, acc=dH0)
        if tc and saved.get("X0") is not None:
            dH0b = torch.empty((nE, hp), dtype=T, device=dev)
            concat_bf16(dH0, h, dH0b, nE)                      # f32 accumulator -> bf16 operand
            wgrad_tc(dH0b, saved["X0"], nE, h, d_v + d_e, dWi)
            if dbi is not None:
                column_sum(dH0, nE, h, dbi)
        elif x3 and saved.get("X0f") is not None:
            X0f = saved["X0f"]
            dWi4 = torch.empty((h, X0f.shape[1]), dtype=torch.float32, device=dev)
            wgrad_x3(dH0, X0f, nE, h, X0f.shape[1], dWi4)
            dWi.copy_(dWi4[:, : d_v + d_e])
            if dbi is not None:
                column_sum(dH0, nE, h, dbi)
        else:
            linear_wgrad(dH0, V, d_v, dWi, h, idx1=lay.src_row, X2=E, K2=d_e, idx2=lay.perm, dbias=dbi, R=nE)
    return dWi, dbi, dWh, dbh, dWo, dbo


def bond_backward_tc(lay: Layout, V: Tensor, E: Tensor, Wi: Tensor, Wh: Tensor, Wo: Tensor, cfg: MPConfig,
                     saved: dict, gHv: Tensor, need_bias: tuple[bool, bool, bool]):
    """bf16-tier autograd mirror on the tensor-core kernels (directed bonds).  Differences from the generic
    mirror: every GEMM is tcgen05; tau' is fused into the backward message kernel; dH_0 is never kept as an f32
    read-modify-write accumulator -- the per-step dZ^t stay in bf16 and are summed once, in f32, at the end."""
    dev = V.device
    h = Wh.shape[0]
    hp = pad_hidden(h)
    d_v, d_e = V.shape[1], E.shape[1]
    T = cfg.hidden_dtype
    nE, nV = lay.E, lay.V
    a, ap = cfg.act, cfg.act_param
    # pure streaming passes run over the 16-padded width (16-byte vectors; padding columns only ever feed
    # consumers that clip at h); the gather kernels keep 8-byte lanes (75 of 96 lanes busy beats 38 of 64)
    hc = (h + 15) // 16 * 16
    H0, Hs, Hv = saved["H0"], saved["Hs"], saved["Hv"]
    f32 = dict(dtype=torch.float32, device=dev)
    # every weight gradient is WRITTEN by its first GEMM (no zero fill + accumulate); zeros only where no GEMM runs
    no_e = nE == 0
    dWi = torch.zeros_like(Wi, dtype=torch.float32) if no_e else torch.empty_like(Wi, dtype=torch.float32)
    dWh = torch.zeros_like(Wh, dtype=torch.float32) if (no_e or cfg.depth == 1) else torch.empty_like(Wh, dtype=torch.float32)
    dWo = torch.empty_like(Wo, dtype=torch.float32)
    wh_acc = [False]                                  # has dW_h been written yet?

    def wgrad_h(dYt, Xt):
        wgrad_tc(dYt, Xt, nE, h, h, dWh, accumulate=wh_acc[0])
        wh_acc[0] = True
    dbi = torch.zeros(h, **f32) if need_bias[0] else None
    dbh = torch.zeros(h, **f32) if need_bias[1] else None
    dbo = torch.zeros(h, **f32) if need_bias[2] else None
    if gHv.stride(1) != 1:
        gHv = gHv.contiguous()
    # Training-mode dropout (cfg.dropout_p > 0; ReLU only, dropout_fused_ok): a gradient that crosses a dropout site is
    # multiplied by the keep mask and by s = 1 / (1 - p).  With ReLU the mask is already in tau' of the stored POST-dropout
    # state ([H_post > 0] = mask * [H_pre > 0]), and s, a scalar, folds into the packed weight of the GEMM that produces
    # the gradient arriving at the site (or, for W_o's own gradient, into the result).
    s_drop = 1.0 / (1.0 - cfg.dropout_p) if cfg.dropout_p > 0 else 1.0
    s_v = s_drop                                      # site after W_o (base.py:182)
    s_e = s_drop if cfg.depth > 1 else 1.0            # site on H^{T-1} (base.py:139); H^0 = tau(H_0) has none
    dY = _empty_hidden(nV, hp, T, dev)
    act_bwd(gHv, Hv, nV, h, act=a, act_param=ap, dZ=dY)      # dY / s_v
    oc = saved.get("ones_col")
    if dbo is not None and oc is not None:
        dWo_ext = torch.empty((h, oc + 1), **f32)            # [dW_o | 0 | db_o]: the ones column of XO (bond_forward)
        wgrad_tc(dY, saved["XO"], nV, h, oc + 1, dWo_ext)
        dWo, dbo = dWo_ext[:, : d_v + h], dWo_ext[:, oc]
    else:
        wgrad_tc(dY, saved["XO"], nV, h, d_v + h, dWo)
        if dbo is not None:
            column_sum(dY, nV, h, dbo)
    if s_v != 1.0:
        dWo.mul_(s_v)
        if dbo is not None:
            dbo.mul_(s_v)
    if nE == 0:
        return dWi, dbi, dWh, dbh, dWo, dbo
    dMv = _empty_hidden(nV, hp, T, dev)
    Wo_m = Wo[:, d_v:] if s_v * s_e == 1.0 else Wo[:, d_v:] * (s_v * s_e)
    linear_tc(dY, h, pack_weight_tc(Wo_m, transpose=True), h, dMv, R=nV)
    dH0b = _empty_hidden(nE, hp, T, dev)
    if cfg.depth == 1:
        act_bwd(dMv, H0, nE, hc, act=a, act_param=ap, gidx=lay.dst_row, from_preact=True, dZ=dH0b)
    else:
        fused_bwd = _fused_step_ok(cfg, lay, h)      # the depth step's mirror on the same fused tcgen05 kernel
        if s_drop != 1.0 and not fused_bwd:
            raise DmpnnError("dropout on the monolithic tier needs the fused depth step (see dropout_fused_ok)")
        WhT_pk = None if fused_bwd else pack_weight_tc(Wh, transpose=True)
        WhT_pkf = pack_weight_bf16(Wh.t().contiguous()) if fused_bwd else None
        # mirror steps whose result arrives at a dropout site (every one but the last, which lands on H^0) carry s
        WhT_pkf_s = WhT_pkf if s_drop == 1.0 else pack_weight_bf16((Wh * s_drop).t().contiguous())
        dZ = _empty_hidden(nE, hp, T, dev)
        act_bwd(dMv, Hs[-1], nE, hc, act=a, act_param=ap, gidx=lay.dst_row, dZ=dZ)    # dZ^{T-1}
        dZs, dH_first, fused_sum, dH0_terms = [dZ], None, False, None
        for t in range(cfg.depth - 1, 0, -1):
            first = t == 1
            Hin = H0 if first else Hs[t - 2]
            if dbh is not None:
                column_sum(dZ, nE, h, dbh, accumulate=True)
            if fused_bwd:
                # dH^{t-1} = (S.P)(dZ . W_h) = ((S.P) dZ) . W_h: gather on the A operand, tau' in the epilogue.
                # W_h gradient without recomputing M^t:  dZ^T . M^t = dZ^T . (P.S) H^{t-1} = ((S.P) dZ)^T . H^{t-1};
                # the kernel writes its gathered operand G = (S.P) dZ out.  t = 1 has no stored tau(H_0): it uses
                # the M^1 the forward kernel saved.
                M1 = saved["Ms"][0] if first else None
                if first and M1 is None:
                    M1 = _empty_hidden(nE, hp, T, dev)
                    bond_message(H0, lay, h, M1, act=a, act_param=ap)
                if first:
                    wgrad_h(dZ, M1)
                    if SUM_IN_EPILOGUE and len(dZs) <= 2:
                        # last mirror step writes dH_0 itself: tau'(H_0) mask and the sum over the dZ^t in its epilogue
                        bond_step_bwd_fused(dZ, H0, dH0b, h, WhT_pkf, lay, a, ap, y_is_preact=True, addends=tuple(dZs))
                        fused_sum = True
                    elif not SUM_IN_EPILOGUE:
                        # dH_0 = sum_t dZ^t + dH^0 * tau'(H_0) is only ever contracted with X_0 (and summed for the
                        # bias): keep the terms apart -- the last mirror step applies tau'(H_0) in its epilogue and
                        # the W_i gradient accumulates one GEMM per term instead of a 5-stream summing pass
                        bond_step_bwd_fused(dZ, H0, dH0b, h, WhT_pkf, lay, a, ap, y_is_preact=True)
                        dH0_terms = dZs + [dH0b]
                    else:
                        dH_first = _empty_hidden(nE, hp, T, dev)
                        bond_step_bwd_fused(dZ, None, dH_first, h, WhT_pkf, lay, a, ap)
                else:
                    dZn = _empty_hidden(nE, hp, T, dev)
                    G = _empty_hidden(nE, hp, T, dev)
                    bond_step_bwd_fused(dZ, Hin, dZn, h, WhT_pkf_s, lay, a, ap, G_out=G)
                    wgrad_h(G, Hin)
                    dZ = dZn
                    dZs.append(dZ)
                continue
            M = _empty_hidden(nE, hp, T, dev)                # M^t, recomputed
            bond_message(Hin, lay, h, M, act=(a if first else ACT_NONE), act_param=ap)
            wgrad_h(dZ, M)
            dM = _empty_hidden(nE, hp, T, dev)
            linear_tc(dZ, h, WhT_pk, h, dM, R=nE)
            if first:
                dH_first = _empty_hidden(nE, hp, T, dev)     # dH^0 (tau' from the pre-activation H_0 is applied below)
                bond_message(dM, lay, h, dH_first, permute_on_read=True)
            else:
                dZ = _empty_hidden(nE, hp, T, dev)           # dZ^{t-1} = S.P(dM) * tau'(H^{t-1})
                bond_message_bwd_masked(dM, Hin, lay, h, dZ, act=a, act_param=ap)
                dZs.append(dZ)
        if dH0_terms is not None:
            wgrad_tc_multi(dH0_terms, saved["X0"], nE, h, d_v + d_e, dWi)     # X_0 read once for all terms
            if dbi is not None:
                for i, P in enumerate(dH0_terms):
                    column_sum(P, nE, h, dbi, accumulate=i > 0)
            return dWi, dbi, dWh, dbh, dWo, dbo
        if not fused_sum:
            sum_act_bwd(dZs, dH_first, H0, dH0b, nE, hc, act=a, act_param=ap)
    wgrad_tc(dH0b, saved["X0"], nE, h, d_v + d_e, dWi)
    if dbi is not None:
        column_sum(dH0b, nE, h, dbi)
    return dWi, dbi, dWh, dbh, dWo, dbo


def _refuse_feature_grads(ctx):
    """The hand-written mirrors produce the six parameter gradients only.  chemprop never asks for d/dV or d/dE (features
    come out of the featuriser), but a caller who does (learned atom embeddings, input saliency) must not get a silent
    `None` where the reference's autograd would deliver a gradient."""
    if ctx.needs_input_grad[0] or ctx.needs_input_grad[1]:
        raise DmpnnError(
            "bmg.V / bmg.E require grad: the engine's hand-written backward produces parameter gradients only "
            "(d/dV, d/dE are not implemented); detach the features, or use the reference module for input attribution")


class BondMPFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, V, E, Wi, bi, Wh, bh, Wo, bo, lay, cfg):
        _require_cuda(V, E, Wi, Wh, Wo)
        _refuse_feature_grads(ctx)
        V = V.contiguous().float()
        E = E.contiguous().float()
        Wi_, Wh_, Wo_ = Wi.detach().contiguous().float(), Wh.detach().contiguous().float(), Wo.detach().contiguous().float()
        bi_ = None if bi is None else bi.detach().contiguous().float()
        bh_ = None if bh is None else bh.detach().contiguous().float()
        bo_ = None if bo is None else bo.detach().contiguous().float()
        Hv, saved = bond_forward(lay, V, E, Wi_, bi_, Wh_, bh_, Wo_, bo_, cfg, for_backward=any(ctx.needs_input_grad))
        # `Hv` is the tensor autograd turns into this node's output: keeping THAT object in ctx.saved would be a reference
        # cycle (node -> saved -> Hv -> grad_fn = node) and the step's activations would live until Python's cyclic GC
        # runs (GBs per step, cudaMalloc on every step); a detached alias shares the storage without the back edge
        saved["Hv"] = Hv.detach()
        ctx.lay, ctx.cfg, ctx.saved = lay, cfg, saved
        ctx.VE = (V, E)
        ctx.W = (Wi_, Wh_, Wo_)
        ctx.has_bias = (bi is not None, bh is not None, bo is not None)
        ctx.wdtypes = (Wi.dtype, Wh.dtype, Wo.dtype)
        return Hv

    @staticmethod
    def backward(ctx, gHv):
        V, E = ctx.VE
        Wi, Wh, Wo = ctx.W
        bwd = bond_backward_tc if (ctx.saved.get("tc") and not ctx.cfg.undirected and ctx.saved.get("X0") is not None
                                   and h_is_mult4(Wh)) else bond_backward
        dWi, dbi, dWh, dbh, dWo, dbo = bwd(ctx.lay, V, E, Wi, Wh, Wo, ctx.cfg, ctx.saved, gHv, ctx.has_bias)
        # ctx.saved stays until autograd frees the node: a second backward (retain_graph=True) works like torch's own
        d0, d1, d2 = ctx.wdtypes
        cast = lambda g, d: None if g is None else g.to(d)
        return (None, None, cast(dWi, d0), cast(dbi, d0), cast(dWh, d1), cast(dbh, d1), cast(dWo, d2),
                cast(dbo, d2), None, None)


# ----------------------------------------------------------------------------------------------
# atom message passing (atom-granular: every edge row depends only on its source atom)
# ----------------------------------------------------------------------------------------------
def atom_forward(lay: Layout, V: Tensor, E: Tensor, Wi: Tensor, bi, Wh: Tensor, bh, Wo: Tensor, bo,
                 cfg: MPConfig):
    """AtomMessagePassing.forward up to W_o (base.py:196-212 with mixins.py:22-30), restated on atoms:
    the reference's H[e] equals Ha[src(e)], so M[e] = [sum_{u in N(src e)} Ha[u] || sum_in E]."""
    dev = V.device
    h = Wi.shape[0]
    hp = pad_hidden(h)
    d_v, d_e = V.shape[1], E.shape[1]
    T = cfg.hidden_dtype
    nV = lay.V
    a, ap = cfg.act, cfg.act_param
    H0 = _hidden(nV, hp, T, dev)
    linear_fwd(V, d_v, Wi, H0, h, bias=bi, R=nV, pad_to=hp)                       # mixins.py:22-23
    SE = torch.zeros((max(nV, 1), max(d_e, 1)), dtype=torch.float32, device=dev)   # sum of in-edge bond features
    if d_e > 0:
        segment_sum(E, lay.rowptr, nV, d_e, SE, idx=lay.perm)
    Hs, Ns = [], []
    Hprev, first = H0, True
    for _ in range(1, cfg.depth):
        Nb = _hidden(nV, hp, T, dev)  # sum over in-neighbours u of Ha[u]   (mixins.py:25-30)
        segment_sum(Hprev, lay.rowptr, nV, h, Nb, idx=lay.src_row, act=(a if first else ACT_NONE), act_param=ap,
                    pad_to=hp)
        Hn = _hidden(nV, hp, T, dev)
        linear_fwd(Nb, h, Wh, Hn, h, X2=SE if d_e > 0 else None, K2=d_e, bias=bh, res=H0, act=a, act_param=ap,
                   R=nV, pad_to=hp)                                                  # base.py:135-141
        Hs.append(Hn)
        Ns.append(Nb)
        Hprev, first = Hn, False
    Mv = _hidden(nV, hp, T, dev)
    segment_sum(Hprev, lay.rowptr, nV, h, Mv, idx=lay.src_row, act=(a if first else ACT_NONE), act_param=ap,
                pad_to=hp)                                                           # base.py:208-211
    Hv = torch.empty((nV, h), dtype=T, device=dev)
    linear_fwd(V, d_v, Wo, Hv, h, X2=Mv, K2=h, bias=bo, act=a, act_param=ap, R=nV, pad_to=h)
    return Hv, dict(H0=H0, Hs=Hs, Ns=Ns, SE=SE, Mv=Mv, Hv=Hv)


def atom_backward(lay: Layout, V: Tensor, E: Tensor, Wi: Tensor, Wh: Tensor, Wo: Tensor, cfg: MPConfig,
                  saved: dict, gHv: Tensor, need_bias):
    dev = V.device
    h = Wi.shape[0]
    hp = pad_hidden(h)
    d_v, d_e = V.shape[1], E.shape[1]
    T = cfg.hidden_dtype
    nV = lay.V
    a, ap = cfg.act, cfg.act_param
    H0, Hs, Ns, SE, Mv, Hv = saved["H0"], saved["Hs"], saved["Ns"], saved["SE"], saved["Mv"], saved["Hv"]
    f32 = dict(dtype=torch.float32, device=dev)
    dWi = torch.zeros_like(Wi, dtype=torch.float32)
    dWh = torch.zeros_like(Wh, dtype=torch.float32)
    dWo = torch.zeros_like(Wo, dtype=torch.float32)
    dbi = torch.zeros(h, **f32) if need_bias[0] else None
    dbh = torch.zeros(h, **f32) if need_bias[1] else None
    dbo = torch.zeros(h, **f32) if need_bias[2] else None
    gHv = gHv.contiguous()
    dY = _hidden(nV, hp, T, dev)
    act_bwd(gHv, Hv, nV, h, act=a, act_param=ap, dZ=dY)
    linear_wgrad(dY, V, d_v, dWo, h, X2=Mv, K2=h, dbias=dbo, R=nV)
    WoT = Wo[:, d_v:].t().contiguous()
    dMv = _hidden(nV, hp, T, dev)
    linear_fwd(dY, h, WoT, dMv, h, R=nV, pad_to=hp)
    # d(Ha^{T-1})[u] = sum_{e: src(e)=u} dM_v[dst(e)] = sum_{e' in in(u)} dM_v[src(e')]  (rev is an involution)
    dH0 = torch.zeros((max(nV, 1), hp), **f32)
    dHa = _hidden(nV, hp, T, dev)
    segment_sum(dMv, lay.rowptr, nV, h, dHa, idx=lay.src_row, pad_to=hp)
    WhT = Wh[:, :h].t().contiguous() if cfg.depth > 1 else None
    for t in range(cfg.depth - 1, 0, -1):
        first = t == 1
        dZ = _hidden(nV, hp, T, dev)
        act_bwd(dHa, Hs[t - 1], nV, h, act=a, act_param=ap, dZ=dZ, acc=dH0)
        linear_wgrad(dZ, Ns[t - 1], h, dWh, h, X2=SE if d_e > 0 else None, K2=d_e, dbias=dbh, accumulate=True, R=nV)
        dN = _hidden(nV, hp, T, dev)
        linear_fwd(dZ, h, WhT, dN, h, R=nV, pad_to=hp)
        dHa = _hidden(nV, hp, T, dev)
        segment_sum(dN, lay.rowptr, nV, h, dHa, idx=lay.src_row, pad_to=hp)
    act_bwd(dHa, H0, nV, h, act=a, act_param=ap, from_preact=True, acc=dH0)
    linear_wgrad(dH0, V, d_v, dWi, h, dbias=dbi, R=nV)
    return dWi, dbi, dWh, dbh, dWo, dbo


def _readout_pad(d_v: int, h: int) -> int:
    """Column at which M_v starts inside the read-out operand [V || M_v]: d_v rounded up to 8 columns (16-byte aligned bf16 rows
    for the vectorised segment sum that writes M_v in place; d_v = 106 of the reaction graphs left it on the scalar kernel:
    1.2 ms per step at C4), unless that would exceed the GEMM's K limit."""
    dvp = (d_v + 7) // 8 * 8
    return dvp if dvp + h <= 448 else d_v


def _wo_padded(Wo: Tensor, d_v: int, dvp: int) -> Tensor:
    """W_o with zero columns for the padding between V and M_v"""
    if dvp == d_v:
        return Wo
    return torch.cat([Wo[:, :d_v], Wo.new_zeros((Wo.shape[0], dvp - d_v)), Wo[:, d_v:]], 1)


def _wo_unpadded(dWo_p: Tensor, d_v: int, dvp: int) -> Tensor:
    return dWo_p if dvp == d_v else torch.cat([dWo_p[:, :d_v], dWo_p[:, dvp:]], 1)


def _atom_tc_ok(cfg: MPConfig, h: int, d_v: int, d_e: int) -> bool:
    return _tc_ok(cfg, h, d_v, h + d_e, d_v + h) and h % 4 == 0


def atom_forward_tc(lay: Layout, V: Tensor, E: Tensor, Wi: Tensor, bi, Wh: Tensor, bh, Wo: Tensor, bo, cfg: MPConfig):
    """bf16 tier of atom_forward on the tensor cores: every GEMM is dmpnn_linear_tc_bf16 (the H_0 residual of
    base.py:138 is added in its epilogue), the neighbour sums write straight into the GEMM's A operand."""
    dev = V.device
    h = Wi.shape[0]
    hp = pad_hidden(h)
    hc = (h + 15) // 16 * 16
    d_v, d_e = V.shape[1], E.shape[1]
    T = cfg.hidden_dtype
    nV = lay.V
    a, ap = cfg.act, cfg.act_param
    rows = max(nV, 1)
    kv = (d_v + 15) // 16 * 16
    Xv = torch.empty((rows, kv), dtype=T, device=dev)
    concat_bf16(V, d_v, Xv, nV, width=kv)
    H0 = _empty_hidden(nV, hp, T, dev)
    linear_tc(Xv, d_v, pack_weight_tc(Wi), h, H0, bias=bi, R=nV)                              # mixins.py:22-23
    SE = None
    if d_e > 0:                                                                               # loop-invariant bond term
        SE = torch.zeros((rows, d_e), dtype=torch.float32, device=dev)
        segment_sum(E, lay.rowptr, nV, d_e, SE, idx=lay.perm)
    ka = (h + d_e + 15) // 16 * 16
    Whpk = pack_weight_tc(Wh) if cfg.depth > 1 else None
    Hs, XAs = [], []
    Hprev, first = H0, True
    for _ in range(1, cfg.depth):
        XA = torch.empty((rows, ka), dtype=T, device=dev)   # [sum_{u in N(v)} Ha[u] || sum_in E]   (mixins.py:25-30)
        with _StepTimer("atom_step_first" if first else "atom_step"):
            segment_sum(Hprev, lay.rowptr, nV, h, XA[:, :h], idx=lay.src_row, act=(a if first else ACT_NONE), act_param=ap,
                        pad_to=h)
            if d_e > 0:
                concat_bf16(SE, d_e, XA[:, h:], nV, width=d_e)
            Hn = _empty_hidden(nV, hp, T, dev)
            linear_tc(XA, h + d_e, Whpk, h, Hn, bias=bh, res=H0, act=a, act_param=ap, R=nV)   # base.py:135-141
        Hs.append(Hn)
        XAs.append(XA)
        Hprev, first = Hn, False
    dvp = _readout_pad(d_v, h)
    ko = (dvp + h + 15) // 16 * 16
    XO = torch.empty((rows, ko), dtype=T, device=dev)
    concat_bf16(V, d_v, XO, nV, width=dvp)
    segment_sum(Hprev, lay.rowptr, nV, h, XO[:, dvp:dvp + h], idx=lay.src_row, act=(a if first else ACT_NONE),
                act_param=ap, pad_to=(hc if dvp + hc <= ko else h))                           # base.py:208-211
    Hvp = torch.empty((rows, hp), dtype=T, device=dev)
    linear_tc(XO, dvp + h, pack_weight_tc(_wo_padded(Wo, d_v, dvp)), h, Hvp, bias=bo, act=a, act_param=ap, R=nV)    # base.py:180-182
    Hv = Hvp[:nV, :h]
    return Hv, dict(H0=H0, Hs=Hs, XAs=XAs, XO=XO, Xv=Xv, Hv=Hv, tc=True, dvp=dvp)


def atom_backward_tc(lay: Layout, V: Tensor, E: Tensor, Wi: Tensor, Wh: Tensor, Wo: Tensor, cfg: MPConfig,
                     saved: dict, gHv: Tensor, need_bias):
    """Autograd mirror of atom_forward_tc (tcgen05 GEMMs; dH_0 is kept as separate terms, one W_i GEMM each)."""
    dev = V.device
    h = Wi.shape[0]
    hp = pad_hidden(h)
    hc = (h + 15) // 16 * 16
    d_v, d_e = V.shape[1], E.shape[1]
    T = cfg.hidden_dtype
    nV = lay.V
    a, ap = cfg.act, cfg.act_param
    H0, Hs, XAs, XO, Xv, Hv = saved["H0"], saved["Hs"], saved["XAs"], saved["XO"], saved["Xv"], saved["Hv"]
    f32 = dict(dtype=torch.float32, device=dev)
    dWi = torch.zeros_like(Wi, dtype=torch.float32)
    dWh = torch.zeros_like(Wh, dtype=torch.float32)
    dWo = torch.zeros_like(Wo, dtype=torch.float32)
    dbi = torch.zeros(h, **f32) if need_bias[0] else None
    dbh = torch.zeros(h, **f32) if need_bias[1] else None
    dbo = torch.zeros(h, **f32) if need_bias[2] else None
    if nV == 0:
        return dWi, dbi, dWh, dbh, dWo, dbo
    if gHv.stride(1) != 1:
        gHv = gHv.contiguous()
    dY = _empty_hidden(nV, hp, T, dev)
    act_bwd(gHv, Hv, nV, h, act=a, act_param=ap, dZ=dY)
    dvp = saved.get("dvp", d_v)
    if dvp == d_v:
        wgrad_tc(dY, XO, nV, h, d_v + h, dWo)
    else:
        dWo_p = torch.empty((h, dvp + h), dtype=torch.float32, device=dev)
        wgrad_tc(dY, XO, nV, h, dvp + h, dWo_p)
        dWo = _wo_unpadded(dWo_p, d_v, dvp)
    if dbo is not None:
        column_sum(dY, nV, h, dbo)
    dMv = _empty_hidden(nV, hp, T, dev)
    linear_tc(dY, h, pack_weight_tc(Wo[:, d_v:], transpose=True), h, dMv, R=nV)
    # d(Ha^{T-1})[u] = sum_{e' in in(u)} dM_v[src(e')]   (rev is an involution)
    dHa = _empty_hidden(nV, hp, T, dev)
    segment_sum(dMv, lay.rowptr, nV, h, dHa, idx=lay.src_row, pad_to=hc)
    WhT_pk = pack_weight_tc(Wh[:, :h], transpose=True) if cfg.depth > 1 else None
    terms = []
    for t in range(cfg.depth - 1, 0, -1):
        dZ = _empty_hidden(nV, hp, T, dev)
        act_bwd(dHa, Hs[t - 1], nV, hc, act=a, act_param=ap, dZ=dZ)
        terms.append(dZ)
        wgrad_tc(dZ, XAs[t - 1], nV, h, h + d_e, dWh, accumulate=True)
        if dbh is not None:
            column_sum(dZ, nV, h, dbh, accumulate=True)
        dN = _empty_hidden(nV, hp, T, dev)
        linear_tc(dZ, h, WhT_pk, h, dN, R=nV)
        dHa = _empty_hidden(nV, hp, T, dev)
        segment_sum(dN, lay.rowptr, nV, h, dHa, idx=lay.src_row, pad_to=hc)
    dH0l = _empty_hidden(nV, hp, T, dev)
    act_bwd(dHa, H0, nV, hc, act=a, act_param=ap, from_preact=True, dZ=dH0l)
    terms.append(dH0l)
    wgrad_tc_multi(terms, Xv, nV, h, d_v, dWi)       # dH_0 = sum_t dZ^t + dHa^0 * tau'(H_0), contracted term by term
    if dbi is not None:
        for i, P in enumerate(terms):
            column_sum(P, nV, h, dbi, accumulate=i > 0)
    return dWi, dbi, dWh, dbh, dWo, dbo


def atom_forward_fused(lay: Layout, V: Tensor, E: Tensor, Wi: Tensor, bi, Wh: Tensor, bh, Wo: Tensor, bo, cfg: MPConfig):
    """bf16 tier of atom_forward with ONE launch per depth step (dmpnn_atom_step_fused_bf16).  The reference's update
    (base.py:135-141) on atoms is tau(H_0 + b_h + W_h . [N^t || SE]) with N^t the neighbour sum of the previous state and SE the
    loop-invariant sum of the incoming bond features: W_h[:, h:] . SE + b_h is added to H_0 ONCE (a K = d_e GEMM with H_0 as
    the residual of its epilogue), which gives the step the bond step's shape  tau(H_0' + W_h[:, :h] . N^t)  -- gather, GEMM
    and epilogue in the fused kernel, with the gathered operand of the first step saved for the W_h gradient."""
    dev = V.device
    h = Wi.shape[0]
    hp = pad_hidden(h)
    hc = (h + 15) // 16 * 16
    d_v, d_e = V.shape[1], E.shape[1]
    T = cfg.hidden_dtype
    nV = lay.V
    a, ap = cfg.act, cfg.act_param
    rows = max(nV, 1)
    # [V || sum_in E] side by side in ONE bf16 operand (16-column blocks): W_i reads its first d_v columns, the H_0' GEMM the
    # second block, and the mirror contracts the dZ^t terms with both in one weight-gradient launch
    kv = (d_v + 15) // 16 * 16
    ke = (d_e + 15) // 16 * 16 if d_e > 0 else 0
    Xv = torch.empty((rows, kv + ke), dtype=T, device=dev)
    concat_bf16(V, d_v, Xv, nV, width=kv)
    H0 = _empty_hidden(nV, hp, T, dev)
    linear_tc(Xv, d_v, pack_weight_tc(Wi), h, H0, bias=bi, R=nV)                              # mixins.py:22-23
    SEb, H0p, step_bias = None, H0, bh
    if d_e > 0:                                                                               # loop-invariant bond term
        SE = torch.zeros((rows, d_e), dtype=torch.float32, device=dev)
        segment_sum(E, lay.rowptr, nV, d_e, SE, idx=lay.perm)
        SEb = Xv[:, kv:kv + ke]
        concat_bf16(SE, d_e, SEb, nV, width=ke)
        H0p = _empty_hidden(nV, hp, T, dev)                                                   # H_0 + b_h + W_h[:, h:] . SE
        linear_tc(SEb, d_e, pack_weight_tc(Wh[:, h:]), h, H0p, bias=bh, res=H0, R=nV)
        step_bias = None
    Whpk = pack_weight_bf16(Wh[:, :h].contiguous())
    Hs, N1 = [], None
    Hprev, first = H0, True
    for _ in range(1, cfg.depth):
        Hn = _empty_hidden(nV, hp, T, dev)
        if first:
            N1 = _empty_hidden(nV, hp, T, dev)
        with _StepTimer("atom_fused_first" if first else "atom_fused"):
            atom_step_fused(Hprev, H0p, Hn, h, Whpk, step_bias, lay, a, ap, first, N_out=N1 if first else None)
        Hs.append(Hn)
        Hprev, first = Hn, False
    dvp = _readout_pad(d_v, h)
    ones_col = dvp + hc if (bo is not None and dvp + hc + 1 <= 448) else None   # see bond_forward: db_o rides on dW_o's GEMM
    ko = (dvp + hc + 1 + 15) // 16 * 16 if ones_col is not None else (dvp + h + 15) // 16 * 16
    XO = torch.empty((rows, ko), dtype=T, device=dev)
    concat_bf16(V, d_v, XO, nV, width=dvp)
    segment_sum(Hprev, lay.rowptr, nV, h, XO[:, dvp:dvp + h], idx=lay.src_row, act=ACT_NONE, act_param=ap,
                pad_to=(hc if dvp + hc <= ko else h))                                         # base.py:208-211
    if ones_col is not None:
        XO[:, ones_col].fill_(1.0)
    Hvp = torch.empty((rows, hp), dtype=T, device=dev)
    linear_tc(XO, dvp + h, pack_weight_tc(_wo_padded(Wo, d_v, dvp)), h, Hvp, bias=bo, act=a, act_param=ap, R=nV)    # base.py:180-182
    Hv = Hvp[:nV, :h]
    return Hv, dict(H0=H0, Hs=Hs, N1=N1, SEb=SEb, XO=XO, Xv=Xv, Hv=Hv, tc=True, fused=True, dvp=dvp, ones_col=ones_col)


def atom_backward_fused(lay: Layout, V: Tensor, E: Tensor, Wi: Tensor, Wh: Tensor, Wo: Tensor, cfg: MPConfig,
                        saved: dict, gHv: Tensor, need_bias):
    """Autograd mirror of atom_forward_fused.  With A the (symmetric) atom adjacency, N^t = A H^{t-1}:
    dH^{t-1} = ((A dZ^t) . W_h[:, :h]) * tau'(H^{t-1}) -- the mirror mode of the fused kernel, whose gathered operand
    G^t = A dZ^t is also the left factor of the step's weight gradient (dZ^T . N^t = G^T . H^{t-1}); t = 1 uses the N^1 the
    forward saved.  dW_h[:, h:] = (sum_t dZ^t)^T . SE and dW_i = (sum_t dZ^t + dH^0 tau'(H_0))^T . V as multi-term GEMMs."""
    dev = V.device
    h = Wi.shape[0]
    hp = pad_hidden(h)
    hc = (h + 15) // 16 * 16
    d_v, d_e = V.shape[1], E.shape[1]
    T = cfg.hidden_dtype
    nV = lay.V
    a, ap = cfg.act, cfg.act_param
    H0, Hs, N1, SEb, XO, Xv, Hv = (saved[k] for k in ("H0", "Hs", "N1", "SEb", "XO", "Xv", "Hv"))
    f32 = dict(dtype=torch.float32, device=dev)
    dWi = torch.empty_like(Wi, dtype=torch.float32)
    dWh = torch.empty_like(Wh, dtype=torch.float32)
    dWo = torch.empty_like(Wo, dtype=torch.float32)
    dbi = torch.zeros(h, **f32) if need_bias[0] else None
    dbh = torch.zeros(h, **f32) if need_bias[1] else None
    dbo = torch.zeros(h, **f32) if need_bias[2] else None
    if gHv.stride(1) != 1:
        gHv = gHv.contiguous()
    dY = _empty_hidden(nV, hp, T, dev)
    act_bwd(gHv, Hv, nV, h, act=a, act_param=ap, dZ=dY)
    dvp = saved.get("dvp", d_v)
    oc = saved.get("ones_col")
    if dbo is not None and oc is not None:
        dWo_p = torch.empty((h, oc + 1), dtype=torch.float32, device=dev)      # [dW_o (padded) | 0 | db_o]
        wgrad_tc(dY, XO, nV, h, oc + 1, dWo_p)
        dWo, dbo = _wo_unpadded(dWo_p[:, :dvp + h], d_v, dvp), dWo_p[:, oc]
    else:
        if dvp == d_v:
            wgrad_tc(dY, XO, nV, h, d_v + h, dWo)
        else:
            dWo_p = torch.empty((h, dvp + h), dtype=torch.float32, device=dev)
            wgrad_tc(dY, XO, nV, h, dvp + h, dWo_p)
            dWo = _wo_unpadded(dWo_p, d_v, dvp)
        if dbo is not None:
            column_sum(dY, nV, h, dbo)
    # dZ^{T-1} = (A (dY . W_o[:, d_v:])) * tau'(H^{T-1}) = ((A dY) . W_o[:, d_v:]) * tau'(H^{T-1}): the read-out GEMM, the
    # neighbour gather of its result and the tau' pass are ONE mirror launch of the fused kernel on dY (three launches before)
    dZ = _empty_hidden(nV, hp, T, dev)
    atom_step_bwd_fused(dY, Hs[-1], dZ, h, pack_weight_bf16(Wo[:, d_v:].t().contiguous()), lay, a, ap)
    WhT = pack_weight_bf16(Wh[:, :h].t().contiguous())
    dWhN = dWh[:, :h]
    terms, wrote = [dZ], False
    dH0l = _empty_hidden(nV, hp, T, dev)
    for t in range(cfg.depth - 1, 0, -1):
        if dbh is not None:
            column_sum(dZ, nV, h, dbh, accumulate=True)
        if t == 1:
            wgrad_tc(dZ, N1, nV, h, h, dWhN, accumulate=wrote)
            atom_step_bwd_fused(dZ, H0, dH0l, h, WhT, lay, a, ap, y_is_preact=True)           # dH^0 * tau'(H_0)
        else:
            Hin = Hs[t - 2]
            dZn = _empty_hidden(nV, hp, T, dev)
            G = _empty_hidden(nV, hp, T, dev)
            atom_step_bwd_fused(dZ, Hin, dZn, h, WhT, lay, a, ap, G_out=G)
            wgrad_tc(G, Hin, nV, h, h, dWhN, accumulate=wrote)
            dZ = dZn
            terms.append(dZ)
        wrote = True
    if d_e > 0:
        # one pass over the dZ^t terms for both [V || sum_in E] blocks of Xv, then the dH^0 term for the V block alone
        kv = (d_v + 15) // 16 * 16
        dWx = torch.empty((h, kv + d_e), **f32)
        wgrad_tc_multi(terms, Xv, nV, h, kv + d_e, dWx)
        wgrad_tc(dH0l, Xv, nV, h, d_v, dWx[:, :d_v], accumulate=True)
        dWi = dWx[:, :d_v]
        dWh[:, h:].copy_(dWx[:, kv:kv + d_e])
    else:
        wgrad_tc_multi(terms + [dH0l], Xv, nV, h, d_v, dWi)
    if dbi is not None:
        for i, P in enumerate(terms + [dH0l]):
            column_sum(P, nV, h, dbi, accumulate=i > 0)
    return dWi, dbi, dWh, dbh, dWo, dbo


class AtomMPFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, V, E, Wi, bi, Wh, bh, Wo, bo, lay, cfg):
        _require_cuda(V, E, Wi, Wh, Wo)
        _refuse_feature_grads(ctx)
        V = V.contiguous().float()
        E = E.contiguous().float()
        Wi_, Wh_, Wo_ = Wi.detach().contiguous().float(), Wh.detach().contiguous().float(), Wo.detach().contiguous().float()
        bi_ = None if bi is None else bi.detach().contiguous().float()
        bh_ = None if bh is None else bh.detach().contiguous().float()
        bo_ = None if bo is None else bo.detach().contiguous().float()
        fwd = atom_forward_tc if (_atom_tc_ok(cfg, Wi_.shape[0], V.shape[1], E.shape[1]) and lay.V > 0) else atom_forward
        if fwd is atom_forward_tc and _atom_fused_ok(cfg, lay, Wi_.shape[0], V.shape[1], E.shape[1]):
            fwd = atom_forward_fused
        Hv, saved = fwd(lay, V, E, Wi_, bi_, Wh_, bh_, Wo_, bo_, cfg)
        # `Hv` is the tensor autograd turns into this node's output: keeping THAT object in ctx.saved would be a reference
        # cycle (node -> saved -> Hv -> grad_fn = node) and the step's activations would live until Python's cyclic GC
        # runs (GBs per step, cudaMalloc on every step); a detached alias shares the storage without the back edge
        saved["Hv"] = Hv.detach()
        ctx.lay, ctx.cfg, ctx.saved = lay, cfg, saved
        ctx.VE = (V, E)
        ctx.W = (Wi_, Wh_, Wo_)
        ctx.has_bias = (bi is not None, bh is not None, bo is not None)
        ctx.wdtypes = (Wi.dtype, Wh.dtype, Wo.dtype)
        return Hv

    @staticmethod
    def backward(ctx, gHv):
        V, E = ctx.VE
        Wi, Wh, Wo = ctx.W
        bwd = atom_backward_fused if ctx.saved.get("fused") else atom_backward_tc if ctx.saved.get("tc") else atom_backward
        dWi, dbi, dWh, dbh, dWo, dbo = bwd(ctx.lay, V, E, Wi, Wh, Wo, ctx.cfg, ctx.saved, gHv, ctx.has_bias)
        # ctx.saved stays until autograd frees the node: a second backward (retain_graph=True) works like torch's own
        d0, d1, d2 = ctx.wdtypes
        cast = lambda g, d: None if g is None else g.to(d)
        return (None, None, cast(dWi, d0), cast(dbi, d0), cast(dWh, d1), cast(dbh, d1), cast(dWo, d2),
                cast(dbo, d2), None, None)


# ----------------------------------------------------------------------------------------------
# aggregation
# ----------------------------------------------------------------------------------------------
class SegmentAggFunction(torch.autograd.Function):
    """Mean / Sum / Norm aggregation over molecules (chemprop/nn/agg.py:73-78, 90-95, 112-113)."""

    @staticmethod
    def forward(ctx, H, mol_atom_ptr, atom_mol, n_mols, scale_mode, scale):
        _require_cuda(H)
        Hc = H if H.stride(1) == 1 else H.contiguous()
        # molecule-level output is always f32 (b x d is tiny): whatever follows -- the reference's BatchNorm / FFN heads
        # (models/model.py:126-161) -- holds f32 parameters, so a bf16-tier encoder drops in without a cast by the caller
        out = torch.empty((n_mols, H.shape[1]), dtype=torch.float32, device=H.device)
        segment_sum(Hc, mol_atom_ptr, n_mols, H.shape[1], out, scale_mode=scale_mode, scale=scale,
                    pad_to=H.shape[1])
        ctx.ptr, ctx.atom_mol, ctx.mode, ctx.scale = mol_atom_ptr, atom_mol, scale_mode, scale
        ctx.nV, ctx.in_dtype = H.shape[0], H.dtype
        return out

    @staticmethod
    def backward(ctx, g):
        g = g.contiguous()
        if g.dtype not in (torch.float32, torch.bfloat16):
            g = g.float()
        dH = torch.empty((ctx.nV, g.shape[1]), dtype=ctx.in_dtype, device=g.device)
        segment_bcast(g, ctx.atom_mol, ctx.ptr, ctx.nV, g.shape[1], dH, scale_mode=ctx.mode, scale=ctx.scale,
                      n_seg=g.shape[0])
        return dH, None, None, None, None, None


class SegmentBcastFunction(torch.autograd.Function):
    """rows <- their segment's row (`Z[batch]` of chemprop/nn/agg.py:127, nn/ffn.py:127): dmpnn_segment_bcast; the mirror
    is the segment sum."""

    @staticmethod
    def forward(ctx, G, mol_atom_ptr, atom_mol, n_rows):
        _require_cuda(G)
        Gc = G if G.stride(1) == 1 else G.contiguous()
        out = torch.empty((n_rows, G.shape[1]), dtype=G.dtype, device=G.device)
        segment_bcast(Gc, atom_mol, mol_atom_ptr, n_rows, G.shape[1], out, n_seg=G.shape[0])
        ctx.ptr, ctx.n_seg = mol_atom_ptr, G.shape[0]
        return out

    @staticmethod
    def backward(ctx, g):
        g = g.contiguous()
        dG = torch.empty((ctx.n_seg, g.shape[1]), dtype=g.dtype, device=g.device)
        segment_sum(g, ctx.ptr, ctx.n_seg, g.shape[1], dG, pad_to=g.shape[1])
        return dG, None, None, None
