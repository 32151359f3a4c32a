#!/usr/bin/env python
"""Benchmark of the D-MPNN hot path (BASELINE.json): molecules/sec, forward+backward, of the message-passing encoder +
aggregation on synthetic molecule batches.

    python bench.py [--config C2|C3|C4|C5] [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

Configurations (BASELINE.json `configs`; C1 is the reference's CPU plumbing case and lives in the tests):
  C2  10 k ~25-atom molecules / GPU, BondMessagePassing h=300 depth=3, bf16 tier, fused depth step   (default, weak scaling)
  C3  50 k molecules, h=600 depth=6, fp32 tier (3xTF32 tensor-core GEMMs)
  C4  10 k ~80-atom condensed-reaction graphs (d_v=106, d_e=28), AtomMessagePassing h=300 depth=3, bf16 tier
  C5  1 M molecules, global batch 200 k = 8 micro-batches of 25 k, sharded over the ranks by the loader
      (DistributedSampler semantics), gradient accumulation + ONE all-reduce per step                     (strong scaling)

One process per GPU (torchrun for N>1, NCCL).  A "step" is one pass of the hot path over one batch: device layout build,
forward, dummy scalar loss on the b x h output, backward (all weight gradients), and for N>1 the gradient all-reduce.
Prints ONE JSON line (rank 0):

 value         whole-job molecules/s, the batch's tensors already resident in HBM when the timed region starts
 e2e           same metric through the public loader API (`PackedBatchLoader` over a `PackedMolGraphDataset` resident in
               HBM): every step the host draws the batch's molecule ids, uploads ids + offsets from pinned memory (24 B per
               molecule), the batch is assembled by one gather launch, and the step's loss is copied back and read by the host
 e2e_host_batch  (C2, N = 1) the same step fed with a complete host batch per step (bf16 features + int32 indices, 57 MB H2D)
 roofline      the dominant kernel: algorithmic bytes or flops / its CUDA-event duration vs the measured peak
 cpu_baseline  the oracle port (the reference's own op sequence on torch CPU) on the host cores, bounded sample

`--dump-outputs DIR` writes the results of the last timed step of the path `value` measures: the per-atom hidden states
`H` and the per-molecule aggregates `agg` (a fixed, seeded sample of rows when larger than 16 MB), the `loss` and every
weight gradient `grad.<name>`, as float32 .npy files.  Inputs and weights are seeded, so two builds run with the same
arguments can be compared array for array.

`--impl reference` times that CPU implementation on the SAME workload (full batch per step) on the host's cores.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CONFIGS = {
    "C2": dict(kind="bond", n_mols=10_000, d_h=300, depth=3, precision="bf16", gen="mol", d_v=72, d_e=14, pool=3,
               scaling="weak", desc="10000 synthetic mols/GPU (~25 atoms), BondMessagePassing h=300 depth=3 + MeanAggregation"),
    "C3": dict(kind="bond", n_mols=50_000, d_h=600, depth=6, precision="fp32", gen="mol", d_v=72, d_e=14, pool=1,
               scaling="weak", graph=False,      # ~100 GB of activations per step: no room for a graph's private pool beside it
               desc="50000 synthetic mols/GPU (~25 atoms), BondMessagePassing h=600 depth=6 fp32 + MeanAggregation"),
    "C4": dict(kind="atom", n_mols=10_000, d_h=300, depth=3, precision="bf16", gen="cgr", d_v=106, d_e=28, pool=2,
               scaling="weak", desc="10000 synthetic condensed reaction graphs/GPU (~80 atoms, d_v=106 d_e=28), "
                                    "AtomMessagePassing h=300 depth=3 + MeanAggregation"),
    "C5": dict(kind="bond", n_mols=25_000, d_h=300, depth=3, precision="bf16", gen="mol", d_v=72, d_e=14, pool=0,
               scaling="strong", total=1_000_000, global_batch=200_000, unique=100_000,
               desc="1M synthetic mols (~25 atoms) data-parallel, global batch 200000 = 8 micro-batches of 25000, "
                    "BondMessagePassing h=300 depth=3 + MeanAggregation"),
}
FALLBACK_HBM_GBS = 6650.0
FALLBACK_BF16_TFLOPS = 1400.0


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    out = {"hbm": FALLBACK_HBM_GBS, "bf16": FALLBACK_BF16_TFLOPS, "src": "fallback"}
    if os.path.exists(p):
        try:
            j = json.load(open(p))
            out = {"hbm": float(j["hbm_gbs"]), "bf16": float(j.get("bf16_tflops_sustained", j.get("bf16_tflops", FALLBACK_BF16_TFLOPS))),
                   "src": "measured"}
        except Exception:
            pass
    return out


def workload_config(name: str, cfg: dict, world: int) -> dict:
    """The workload, stated identically by both arms (`--impl reference` runs exactly this on the host cores)."""
    return {
        "workload": f"{name}: {cfg['desc']}, fwd+bwd",
        "molecules_per_step": cfg["global_batch"] if cfg["scaling"] == "strong" else cfg["n_mols"] * world,
        "d_h": cfg["d_h"], "depth": cfg["depth"], "kind": cfg["kind"],
        "parallelism": f"dp{world}",
        "l2": "working set (hidden buffers >= 0.15 GB each) exceeds the 126 MB L2; no explicit flush",
    }


class ClockSampler:
    """Samples SM clock + throttle reasons during the timed region (nvidia-smi fields via NVML)."""

    def __init__(self, index: int):
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop = threading.Event()
        self._t = None
        self._nv = self._h = None
        try:                                    # NVML is initialised here, outside the timed region
            import pynvml as nv

            nv.nvmlInit()
            self._nv, self._h = nv, nv.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(self._h, nv.NVML_CLOCK_SM)
        except Exception as e:  # noqa: BLE001
            self.reasons.add(f"nvml_unavailable:{type(e).__name__}")

    def _sample(self):
        nv, h = self._nv, self._h
        names = {
            "hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
            "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
            "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
            "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4),
            "hw_power_brake": getattr(nv, "nvmlClocksThrottleReasonHwPowerBrakeSlowdown", 0x80),
        }
        self.samples.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
        r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
        for k, bit in names.items():
            if r & bit:
                self.reasons.add(k)

    def _run(self):
        if self._nv is None:
            return
        try:
            while not self._stop.is_set():
                self._sample()
                time.sleep(0.002)
        except Exception as e:  # noqa: BLE001
            self.reasons.add(f"nvml_unavailable:{type(e).__name__}")

    def __enter__(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        try:
            if self._nv is not None:
                self._sample()
        except Exception:  # noqa: BLE001
            pass
        self._stop.set()
        self._t.join(timeout=2)

    def summary(self):
        return {"sm_mhz": statistics.median(self.samples) if self.samples else None,
                "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


def bind_to_gpu_numa(index: int) -> str:
    """Pin this rank's host threads to the CPUs next to its GPU (NVML's ideal affinity = the GPU's NUMA node): the loader's
    pinned staging memory and the H2D copies then stay on the local memory controller and PCIe root."""
    try:
        import pynvml as nv

        nv.nvmlInit()
        h = nv.nvmlDeviceGetHandleByIndex(index)
        words = nv.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = [64 * w + b for w, word in enumerate(words) for b in range(64) if (word >> b) & 1]
        cpus = [c for c in cpus if c in os.sched_getaffinity(0)]
        if cpus:
            os.sched_setaffinity(0, cpus)
            return f"{len(cpus)} cpus of the GPU's NUMA node ({cpus[0]}..{cpus[-1]})"
    except Exception as e:  # noqa: BLE001
        return f"unbound ({type(e).__name__})"
    return "unbound"


def gen_mols(cfg: dict, n: int, seed: int):
    from chemprop_b200.data import make_cgr_graphs, make_molecules

    if cfg["gen"] == "cgr":
        return make_cgr_graphs(n, seed=seed, d_v=cfg["d_v"], d_e=cfg["d_e"])
    return make_molecules(n, seed=seed, mean_atoms=25.0)


# ------------------------------------------------------------------------------------------------
# CPU arm: the oracle port (the reference's op sequence on torch CPU), all useful host threads
# ------------------------------------------------------------------------------------------------
def cpu_step_fn(cfg: dict, n_mols: int, seed: int):
    """One fwd+bwd step of the path on the host cores, and what ran it: the UNMODIFIED reference's own modules
    (`chemprop.nn.{Bond,Atom}MessagePassing` + `MeanAggregation` on a `chemprop.data.BatchMolGraph`, imported from the
    reference tree through oracle/ref_shim.py) where that tree is reachable -- i.e. in the build container -- and otherwise
    (the GPU box: the tree does not travel) the oracle restatement of the same op sequence.  -> (step, kind)"""
    torch.manual_seed(seed)
    mgs = gen_mols(cfg, n_mols, seed)
    h, d_v, d_e = cfg["d_h"], cfg["d_v"], cfg["d_e"]
    try:
        from oracle.ref_shim import import_reference, reference_available

        if os.environ.get("DMPNN_BENCH_CPU_KIND", "") != "port" and reference_available():
            import_reference()
            import chemprop.nn as ref_nn
            from chemprop.data import BatchMolGraph as RefBMG
            from chemprop.data.molgraph import MolGraph as RefMG

            cls = ref_nn.BondMessagePassing if cfg["kind"] == "bond" else ref_nn.AtomMessagePassing
            mp = cls(d_v=d_v, d_e=d_e, d_h=h, depth=cfg["depth"])
            agg = ref_nn.MeanAggregation()
            bmg = RefBMG([RefMG(*m) for m in mgs])

            def step_ref():
                mp.zero_grad(set_to_none=True)
                loss = agg(mp(bmg), bmg.batch).square().mean()
                loss.backward()
                return loss.item()

            return step_ref, "reference"
    except Exception as e:  # noqa: BLE001 -- the port below is always available
        print(f"[bench] reference modules not usable ({type(e).__name__}: {e}); timing the oracle port", file=sys.stderr)

    from oracle import restatement as R

    V, E, ei, rev, batch = (torch.from_numpy(x) for x in R.collate(mgs))
    lin = lambda o, i: torch.nn.Linear(i, o).weight.detach().requires_grad_(True)  # noqa: E731
    if cfg["kind"] == "bond":
        Wi, Wh = lin(h, d_v + d_e), lin(h, h)
    else:
        Wi, Wh = lin(h, d_v), lin(h, d_e + h)
    Wo = lin(h, d_v + h)
    bo = torch.zeros(h, requires_grad=True)

    def step():
        for p in (Wi, Wh, Wo, bo):
            p.grad = None
        H = R.message_passing_forward(cfg["kind"], V, E, ei, rev, Wi, None, Wh, None, Wo, bo, cfg["depth"])
        loss = R.aggregate(H, batch, "mean").square().mean()
        loss.backward()
        return loss.item()

    return step, "port"


def run_cpu(cfg: dict, n_mols: int, steps: int, warmup: int):
    """torch's CPU scatter / index kernels stop scaling (and regress) well before 128 threads, so the thread count is
    probed (8, 16, 32, all cores: one step each on a small sample) and the fastest is used for the timed steps."""
    ncpu = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    probe, _ = cpu_step_fn(cfg, min(n_mols, 500), seed=1)
    best_t, best_dt = ncpu, float("inf")
    for nt in sorted({min(8, ncpu), min(16, ncpu), min(32, ncpu), ncpu}):
        torch.set_num_threads(nt)
        probe()
        t0 = time.perf_counter()
        probe()
        dt = time.perf_counter() - t0
        if dt < best_dt:
            best_t, best_dt = nt, dt
    torch.set_num_threads(best_t)
    step, kind = cpu_step_fn(cfg, n_mols, seed=1)
    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = (time.perf_counter() - t0) / max(steps, 1)
    return n_mols / dt, dt, best_t, ncpu, kind


def main_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    name, cfg = args.config, CONFIGS[args.config]
    world = args.gpus
    # the full batch of the configuration per step, unless that cannot finish in minutes (C3 / C5 per-step batches)
    per_step = cfg["n_mols"] if name == "C2" else {"C3": 1_000, "C4": 1_500, "C5": 10_000}[name]
    v, dt, cores, ncpu, kind = run_cpu(cfg, per_step, args.steps, args.warmup)
    what = ("the unmodified reference's modules (imported from its source tree)" if kind == "reference" else
            "oracle restatement of the reference's op sequence")
    full = per_step == cfg["n_mols"]
    line = {
        "impl": "reference", "metric": f"molecules/sec fwd+bwd (h={cfg['d_h']} d={cfg['depth']})", "value": v,
        "unit": "molecules/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3,
        "higher_is_better": True, "scaling": cfg["scaling"], "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(name, cfg, world),
        "cpu_baseline": {"value": v, "unit": "molecules/s", "cores": cores, "kind": kind,
                         "sample": (f"{per_step} molecules per step" + (" = the configuration's full per-GPU batch" if full else
                                    f" (bounded sample of the {cfg['n_mols']}-molecule batch)") +
                                    f" x {args.steps} steps, {what} on torch CPU, {cores} threads "
                                    f"(fastest of 8/16/32/{ncpu})")},
        "e2e": {"value": v, "unit": "molecules/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def main_gpu(args):
    import torch.distributed as dist

    from chemprop_b200 import _lib, engine
    from chemprop_b200.data import BatchMolGraph, PackedBatchLoader, PackedMolGraphDataset, tile_packing_order_of
    from chemprop_b200.nn import AtomMessagePassing, BondMessagePassing, MeanAggregation
    from chemprop_b200.parallel import FlatGradAllReducer

    name, cfg = args.config, CONFIGS[args.config]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = bind_to_gpu_numa(local) if world > 1 else "single process (not bound)"
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.load()
    assert lib.dmpnn_device_ok() == 1, "bench needs an sm_100 device"

    n_mols = args.mols or cfg["n_mols"]
    precision = args.precision or cfg["precision"]
    torch.manual_seed(0)  # identical weights on every rank
    cls = BondMessagePassing if cfg["kind"] == "bond" else AtomMessagePassing
    mp = cls(d_v=cfg["d_v"], d_e=cfg["d_e"], d_h=cfg["d_h"], depth=cfg["depth"], precision=precision).to(dev)
    mp.fused = not args.no_fused
    agg = MeanAggregation()
    params = list(mp.parameters())
    reducer = FlatGradAllReducer(params)
    if world > 1:
        reducer.attach()           # p.grad = views of the flat bucket; NCCL AVG on a side stream behind the backward
    strong = cfg["scaling"] == "strong"

    def zero_grads():
        if world > 1:
            reducer.wait()         # the previous step's all-reduce has to be done before its bucket is cleared
            reducer.zero_()
        else:
            for p in params:
                p.grad = None

    # ---- data: a packed data set resident in HBM + the loader over it -------------------------------------------
    if strong:
        total, gb = cfg["total"], cfg["global_batch"]
        if gb % (n_mols * world) != 0:
            raise SystemExit(f"C5: {world} ranks x {n_mols}-molecule micro-batches do not divide the global batch {gb}")
        uniq = min(cfg["unique"], total)
        base = PackedMolGraphDataset.from_molgraphs(gen_mols(cfg, uniq, seed=11))
        ds = base.replicate(total // uniq).to(dev)           # every rank holds the whole (logical) data set, sharded by the sampler
        micro_per_step = gb // (n_mols * world)
        mols_per_step = gb
        pool_note = f"{total} molecules = {total // uniq} x {uniq} unique synthetic molecules"
    else:
        pool = max(1, cfg["pool"]) * n_mols
        ds = PackedMolGraphDataset.from_molgraphs(gen_mols(cfg, pool, seed=1 + rank)).to(dev)
        micro_per_step = 1
        mols_per_step = world * n_mols
        pool_note = f"{pool} molecules per rank"
    loader = PackedBatchLoader(ds, batch_size=n_mols, shuffle=True, seed=5, rank=rank if strong else 0,
                               world=world if strong else 1, drop_last=True, pack_tiles=not args.no_pack)

    def batches():
        return loader.stream()          # epoch after epoch, plans prefetched across the epoch boundaries

    first_ids = np.arange(n_mols, dtype=np.int64)
    resident = ds.batch(first_ids if args.no_pack else ds.packed_order(first_ids))
    V_atoms, E_rows = resident.V.shape[0], resident.E.shape[0]
    n_tiles = resident._meta_host[_lib.META_N_TILES] if resident._meta_host else None

    last = {}                                    # --dump-outputs: the latest step's results (static outputs under a graph)

    def fwd_bwd(bmg):
        bmg._layout = None                       # the device layout build is part of every step
        H = mp(bmg)
        a = agg(H, bmg.batch)
        loss = a.float().square().mean()
        loss.backward()
        if args.dump_outputs:
            last.update(H=H.detach(), agg=a.detach(), loss=loss.detach())   # no autograd graph kept alive
        return loss

    def snapshot():
        """Host copies of what the timed path computed in its last step (taken after the timed region)."""
        torch.cuda.synchronize()
        out = {"H": sample_rows(last["H"]), "agg": sample_rows(last["agg"]),
               "loss": last["loss"].detach().float().reshape(1).cpu().numpy()}
        for k, p in mp.named_parameters():
            out["grad." + k] = p.grad.detach().float().cpu().numpy()
        return out

    def step_resident():
        zero_grads()
        loss = None
        for _ in range(micro_per_step):
            loss = fwd_bwd(resident)
        reducer.allreduce_()
        return loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for _ in range(steps):
            fn()
        reducer.wait()             # the last step's gradient all-reduce is part of the timed region
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    # ---- device-resident throughput --------------------------------------------------------
    # Eager first (per-kernel CUDA events for the roofline), then -- the product's way to run a fixed-signature batch -- the
    # same step as ONE CUDA graph (chemprop_b200.graph.CudaGraphStep: layout build + forward + loss + backward captured once,
    # replayed per step; the gradient all-reduce stays outside the graph on its side stream).  `value` is the graph figure
    # when the capture works (it does wherever the step is sync-free), the eager one otherwise; both are reported.
    W = max(args.warmup, 3)
    for _ in range(W):
        step_resident()
    engine.STEP_EVENTS = []
    l0 = lib.dmpnn_launch_count()
    with ClockSampler(local) as clocks:
        ms = timed(step_resident, args.steps)
    launches = lib.dmpnn_launch_count() - l0
    step_events, engine.STEP_EVENTS = engine.STEP_EVENTS, None
    dump = snapshot() if args.dump_outputs else None
    ms_per_step = ms / args.steps
    value = mols_per_step / (ms_per_step * 1e-3)
    eager = {"value": value, "ms_per_step": ms_per_step, "gpu_launches": int(launches)}
    graph_info = {"used": False}
    if not args.no_graph and cfg.get("graph", True):
        try:
            from chemprop_b200.graph import CudaGraphStep

            if world == 1:
                for p in params:
                    p.grad = torch.zeros_like(p)

            def graph_body(b):
                if world > 1:
                    reducer.zero_()
                else:
                    for p in params:
                        p.grad.zero_()
                loss = None
                for _ in range(micro_per_step):
                    loss = fwd_bwd(b)
                return loss

            gstep = CudaGraphStep(graph_body)

            def step_graph():
                reducer.wait()
                loss = gstep(resident)
                reducer.allreduce_()
                return loss

            for _ in range(W):
                step_graph()
            with ClockSampler(local) as clocks_g:
                ms_g = timed(step_graph, args.steps)
            if gstep.captures == 1 and ms_g > 0:
                ms_per_step = ms_g / args.steps
                value = mols_per_step / (ms_per_step * 1e-3)
                launches = gstep.last_launches * args.steps
                clocks = clocks_g
                graph_info = {"used": True, "kernels_per_replay": gstep.last_launches, "graph_launches_per_step": 1}
                if args.dump_outputs:
                    dump = snapshot()
            if world == 1:
                for p in params:
                    p.grad = None
        except Exception as e:  # noqa: BLE001 -- the eager figures stand
            graph_info = {"used": False, "error": f"{type(e).__name__}: {e}"[:300]}
            try:
                torch.cuda.synchronize()
            except Exception:  # noqa: BLE001
                pass
        finally:
            gstep = None            # release the graph and its private memory pool before the loader-driven phases
            import gc

            gc.collect()
            torch.cuda.empty_cache()

    # ---- end to end through the loader: ids in (pinned host -> device), loss out ---------------------------------
    loss_host = torch.empty(2, dtype=torch.float32).pin_memory()
    stream_it = batches()

    def e2e_loop(k):
        # The loss of step i is copied to pinned host memory right after its backward is queued and READ by the host one
        # step later (as a logging training loop does): the GPU queue never drains on the read.  All k batches are drawn
        # from the loader (ids uploaded, batch gathered on the device) and all k losses are read inside the timed region.
        pending, losses = None, []
        for i in range(k):
            zero_grads()
            loss = None
            for _ in range(micro_per_step):
                loss = fwd_bwd(next(stream_it).bmg)
            reducer.allreduce_()
            slot = loss_host[i & 1:(i & 1) + 1]
            slot.copy_(loss.detach().float().reshape(1), non_blocking=True)
            done = torch.cuda.Event()
            done.record()
            if pending is not None:
                pending[0].synchronize()
                losses.append(float(pending[1][0]))
            pending = (done, slot)
        pending[0].synchronize()
        losses.append(float(pending[1][0]))
        assert len(losses) == k and all(np.isfinite(losses))

    e2e_loop(2)
    ms_e2e = timed(lambda: e2e_loop(args.steps), 1) / args.steps
    e2e_value = mols_per_step / (ms_e2e * 1e-3)
    h2d_loader = micro_per_step * 8 * (3 * n_mols + 2)

    # ---- (C2) end to end from complete host batches: 57 MB of features + indices per step ------------------------
    e2e_host = None
    if name == "C2" and not strong and not args.no_host_batch and world == 1:
        mgs = gen_mols(cfg, n_mols, seed=1 + rank)
        if not args.no_pack:
            mgs = [mgs[i] for i in tile_packing_order_of(mgs)]
        host_bmg = BatchMolGraph(mgs, pin_memory=True, transfer_dtype=torch.bfloat16 if precision == "bf16" else None)
        del mgs
        copy_stream = torch.cuda.Stream(device=dev)

        def issue_copy():
            with torch.cuda.stream(copy_stream):
                b = host_bmg.cuda_copy(dev, non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(copy_stream)
            return b, ev

        def host_loop(k):
            nxt, pending, losses = issue_copy(), None, []
            for i in range(k):
                bmg, ev = nxt
                torch.cuda.current_stream().wait_event(ev)
                for t in (bmg.V, bmg.E, bmg.edge_index, bmg.rev_edge_index, bmg.batch):
                    t.record_stream(torch.cuda.current_stream())
                if i + 1 < k:
                    nxt = issue_copy()
                zero_grads()
                loss = fwd_bwd(bmg)
                reducer.allreduce_()
                slot = loss_host[i & 1:(i & 1) + 1]
                slot.copy_(loss.detach().float().reshape(1), non_blocking=True)
                done = torch.cuda.Event()
                done.record()
                if pending is not None:
                    pending[0].synchronize()
                    losses.append(float(pending[1][0]))
                pending = (done, slot)
            pending[0].synchronize()
            losses.append(float(pending[1][0]))
            assert len(losses) == k and all(np.isfinite(losses))

        host_loop(2)
        ms_h = timed(lambda: host_loop(args.steps), 1) / args.steps
        e2e_host = {"value": mols_per_step / (ms_h * 1e-3), "unit": "molecules/s", "ms_per_step": ms_h,
                    "h2d_bytes_per_step": host_bmg.transfer_nbytes(), "d2h_bytes_per_step": 4,
                    "host_format": "complete host batch per step: bf16 features + int32 indices "
                                   "(BatchMolGraph(transfer_dtype=bfloat16)), copied on a side stream"}

    # ---- roofline of the dominant kernel -------------------------------------------------------------------------
    pk = peaks()
    s = 2 if precision == "bf16" else 4
    h = cfg["d_h"]
    by_tag = {}
    for tag, a, b in step_events:
        by_tag.setdefault(tag, []).append(a.elapsed_time(b))
    roofline = None
    if "fused" in by_tag:
        dur_ms = statistics.mean(by_tag["fused"])
        alg = 3 * E_rows * h * s + 12 * E_rows + 4 * V_atoms
        ach = alg / (dur_ms * 1e-3) / 1e9
        traffic = None
        tp = os.path.join(ROOT, "profiles", "fused_step_traffic.json")
        if os.path.exists(tp):
            try:
                tj = json.load(open(tp))
                if int(tj.get("directed_edges", -1)) == E_rows and tj.get("precision") == precision:
                    traffic = tj["dram_bytes_per_launch"]
            except Exception:
                pass
        roofline = {"bound": "hbm", "achieved": ach, "peak": pk["hbm"], "unit": "GB/s", "frac": ach / pk["hbm"],
                    "traffic": traffic, "kernel": "k_bond_step_fused: bond depth step t>=2 (message + W_h GEMM + H_0 + tau, one launch)",
                    "launch_ms": dur_ms, "algorithmic_bytes": alg, "peak_source": pk["src"],
                    "traffic_source": "profiles/fused_step_traffic.json (ncu --set full of this kernel on this workload)" if traffic else None,
                    "first_step_ms": statistics.mean(by_tag.get("fused_first", [float("nan")]))}
    elif "x3_gemm" in by_tag:
        # fp32 tier: the depth step is bond_message (HBM-bound) + the 3xTF32 W_h GEMM (tensor-bound); the GEMM dominates
        dur_ms = statistics.mean(by_tag["x3_gemm"])
        flops = 2.0 * E_rows * h * h
        ach = flops / (dur_ms * 1e-3) / 1e12
        alg_b = 3 * E_rows * h * 4
        roofline = {"bound": "tensor", "achieved": ach, "peak": pk["bf16"], "unit": "TFLOP/s", "frac": ach / pk["bf16"],
                    "traffic": None, "kernel": "k_linear_x3: W_h GEMM of the fp32 depth step (3 x tcgen05 kind::tf32 passes per product)",
                    "launch_ms": dur_ms, "algorithmic_flops": flops, "peak_source": pk["src"],
                    "note": ("algorithmic flops 2*E*h*h; the f32-accurate product costs 3 tf32 MMAs = 6 bf16-equivalents, so the "
                             "ceiling of this scheme is peak/6; peak = measured dense bf16 (MEASURED_PEAKS.json, sustained)"),
                    "frac_of_x3_ceiling": ach / (pk["bf16"] / 6.0),
                    "hbm_bound": {"algorithmic_bytes": alg_b, "achieved_gbs": alg_b / (dur_ms * 1e-3) / 1e9, "peak_gbs": pk["hbm"],
                                  "frac": alg_b / (dur_ms * 1e-3) / 1e9 / pk["hbm"]}}
    elif "atom_fused" in by_tag:
        dur_ms = statistics.mean(by_tag["atom_fused"])
        alg = 3 * V_atoms * h * s + 4 * E_rows + 4 * V_atoms          # H_prev, H_0', H_next rows + neighbour table + row pointers
        ach = alg / (dur_ms * 1e-3) / 1e9
        roofline = {"bound": "hbm", "achieved": ach, "peak": pk["hbm"], "unit": "GB/s", "frac": ach / pk["hbm"], "traffic": None,
                    "kernel": "k_bond_step_fused<ATOM>: atom depth step t>=2 (neighbour gather + W_h GEMM + H_0' + tau, one launch)",
                    "launch_ms": dur_ms, "algorithmic_bytes": alg, "peak_source": pk["src"],
                    "first_step_ms": statistics.mean(by_tag.get("atom_fused_first", [float("nan")]))}
    elif "atom_step" in by_tag:
        dur_ms = statistics.mean(by_tag["atom_step"])
        alg = 3 * V_atoms * h * s
        ach = alg / (dur_ms * 1e-3) / 1e9
        roofline = {"bound": "hbm", "achieved": ach, "peak": pk["hbm"], "unit": "GB/s", "frac": ach / pk["hbm"], "traffic": None,
                    "kernel": "atom depth step: neighbour segment sum + k_linear_tc (W_h GEMM + H_0 residual + tau)",
                    "launch_ms": dur_ms, "algorithmic_bytes": alg, "peak_source": pk["src"]}
    elif "unfused" in by_tag:
        dur_ms = statistics.mean(by_tag["unfused"])
        alg = 3 * E_rows * h * s + 12 * E_rows + 4 * V_atoms
        ach = alg / (dur_ms * 1e-3) / 1e9
        roofline = {"bound": "hbm", "achieved": ach, "peak": pk["hbm"], "unit": "GB/s", "frac": ach / pk["hbm"], "traffic": None,
                    "kernel": "bond depth step (unfused: bond_message + GEMM)", "launch_ms": dur_ms, "algorithmic_bytes": alg,
                    "peak_source": pk["src"]}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- CPU baseline (rank 0, N=1 only; bounded sample) ---------------------------------------
    cpu = None
    if world == 1 and not args.no_cpu:
        sample = 1000 if cfg["d_h"] <= 300 and cfg["gen"] == "mol" else 300
        v, dt, cores, ncpu, kind = run_cpu(cfg, sample, 3, 1)
        cpu = {"value": v, "unit": "molecules/s", "cores": cores, "kind": kind,
               "sample": f"{sample} molecules x 3 steps (1 warm-up), "
                         + ("the reference's own modules" if kind == "reference" else "oracle restatement") +
                         f" on torch CPU, {cores} threads (fastest of 8/16/32/{ncpu})"}

    config = workload_config(name, cfg, world)
    line = {
        "metric": f"molecules/sec fwd+bwd (h={cfg['d_h']} d={cfg['depth']})", "value": value, "unit": "molecules/s",
        "n_gpus": world, "steps": args.steps, "warmup": W, "ms_per_step": ms_per_step, "higher_is_better": True,
        "scaling": cfg["scaling"], "vs_baseline": None, "dtype": "bf16" if precision == "bf16" else "f32",
        "data": "synthetic", "config": config,
        "details": {"atoms_per_batch": V_atoms, "directed_edges_per_batch": E_rows, "precision": precision,
                    "tensor_core_fp32": bool(precision == "fp32" and engine.X3_ENABLED and not args.no_fused),
                    "fused_depth_step": ("fused" in by_tag or "atom_fused" in by_tag), "micro_batches_per_step_per_rank": micro_per_step,
                    "molecule_order": ("loader tile packing (best-fit decreasing on edge counts, dmpnn_tile_pack_order)"
                                       if not args.no_pack else "sampler order"),
                    "tiles": n_tiles, "tile_fill": (E_rows / (128.0 * n_tiles)) if n_tiles else None,
                    "step_sync_free": bool(engine.HOST_META), "dataset": pool_note + ", packed, resident in HBM",
                    "dataset_bytes_in_hbm": ds.nbytes(), "host_affinity": numa},
        "clocks": clocks.summary(),
        "e2e": {"value": e2e_value, "unit": "molecules/s", "ms_per_step": ms_e2e, "h2d_bytes_per_step": h2d_loader,
                "d2h_bytes_per_step": 4,
                "path": "PackedBatchLoader over the HBM-resident PackedMolGraphDataset: per step the sampler's molecule ids + "
                        "output offsets go host -> device from pinned memory, one gather launch assembles the BatchMolGraph, "
                        "the loss comes back to the host"},
        "e2e_host_batch": e2e_host,
        "eager": eager,
        "cuda_graph": graph_info,
        "gpu_launches": int(launches),
        "roofline": roofline,
        "cpu_baseline": cpu,
    }
    print(json.dumps(line))
    if dump is not None:
        write_outputs(args.dump_outputs, dump)
    if world > 1:
        dist.destroy_process_group()


DUMP_ARRAY_BYTES = 16 << 20      # per sampled array (H, agg); with the weight gradients the dump stays under 64 MB


def sample_rows(x: torch.Tensor) -> np.ndarray:
    """All rows of `x` as float32, or a fixed, seeded, sorted sample of them when they exceed DUMP_ARRAY_BYTES."""
    x = x.detach().float()
    cap = max(1, DUMP_ARRAY_BYTES // (4 * max(1, x.shape[1])))
    if x.shape[0] > cap:
        idx = np.sort(np.random.default_rng(0).choice(x.shape[0], size=cap, replace=False))
        x = x[torch.from_numpy(idx).to(x.device)]
    return x.cpu().numpy()


def write_outputs(out_dir: str, arrays: dict):
    os.makedirs(out_dir, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(out_dir, f"{k}.npy"), np.ascontiguousarray(v, dtype=np.float32))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="C2", choices=sorted(CONFIGS))
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--mols", type=int, default=0, help="override the per-GPU (micro-)batch size of the configuration")
    ap.add_argument("--precision", default=None, choices=["bf16", "fp32"])
    ap.add_argument("--no-fused", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-host-batch", action="store_true", help="skip the complete-host-batch e2e figure (C2)")
    ap.add_argument("--no-dataset", action="store_true", help="(kept for old command lines; no effect)")
    ap.add_argument("--no-pack", action="store_true", help="keep the sampler's molecule order (no tile packing)")
    ap.add_argument("--no-graph", action="store_true", help="do not run the resident step as a CUDA graph")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step computed (H, agg, loss, grad.<param>) "
                         "as DIR/<name>.npy in float32")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    if args.impl == "reference":
        main_reference(args)
    else:
        main_gpu(args)


if __name__ == "__main__":
    main()
