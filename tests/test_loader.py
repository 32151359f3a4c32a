"""CPU tier: PackedBatchLoader -- the reference's build_dataloader + SeededSampler + DistributedSampler semantics
(chemprop/data/dataloader.py:24-96, samplers.py:8-27) over the packed data set."""
import time

import numpy as np
import pytest
import torch

from chemprop_b200.data import BatchMolGraph, PackedBatchLoader, PackedMolGraphDataset, make_molecules
from chemprop_b200.data.loader import epoch_shard
from tests.util import load_golden

N = 203


@pytest.fixture(scope="module")
def data():
    mgs = make_molecules(N, seed=31, mean_atoms=9, std_atoms=3, shuffle_edges=True, min_atoms=1)
    return mgs, PackedMolGraphDataset.from_molgraphs(mgs)


def _check_batch(b, mgs):
    ref = BatchMolGraph([mgs[i] for i in b.ids])
    for k in ("V", "E", "edge_index", "rev_edge_index", "batch"):
        assert torch.equal(getattr(b.bmg, k), getattr(ref, k)), k
    assert b.bmg._meta_host == ref._meta_host and len(b.bmg) == len(b.ids)


def test_seeded_order_is_the_references_seeded_sampler(data):
    mgs, ds = data
    loader = PackedBatchLoader(ds, batch_size=32, shuffle=True, seed=1234, pack_tiles=False)
    rg, idxs = np.random.default_rng(1234), np.arange(N)          # samplers.py:16-21, restated
    for epoch in range(3):
        rg.shuffle(idxs)
        got = np.concatenate([b.ids for b in loader])
        assert np.array_equal(got, idxs), epoch
    assert len(loader) == 7                                        # 203 = 6 * 32 + 11
    ref = load_golden("fixture_seeded_sampler")                    # the reference's SeededSampler(203, 99), two epochs
    assert int(ref["n"]) == N and int(ref["seed"]) == 99
    ours = PackedBatchLoader(ds, batch_size=50, shuffle=True, seed=99, pack_tiles=False)
    for epoch in range(2):
        assert np.array_equal(ref["order"][epoch], np.concatenate([b.ids for b in ours])), epoch


@pytest.mark.parametrize("prefetch,compact", [(2, False), (3, True)])
def test_batches_are_the_collate_of_their_ids_even_with_a_slow_consumer(data, prefetch, compact):
    mgs, ds = data
    loader = PackedBatchLoader(ds, batch_size=24, shuffle=True, seed=5, prefetch=prefetch,
                               transfer_dtype=torch.bfloat16 if compact else None)
    seen = 0
    for i, b in enumerate(loader):
        if i % 3 == 0:
            time.sleep(0.02)            # let the producer run ahead into the other staging buffers
        _check_batch(b, mgs)
        if compact:
            assert torch.equal(b.bmg._xfer[0], b.bmg.V.bfloat16()) and b.bmg._xfer[2].dtype == torch.int32
        seen += len(b.ids)
    assert seen == N


def test_drop_last_rule_and_unshuffled_order(data):
    mgs, ds = data
    assert [len(b.ids) for b in PackedBatchLoader(ds, batch_size=101, shuffle=False)] == [101, 101]      # 203 % 101 == 1
    assert [len(b.ids) for b in PackedBatchLoader(ds, batch_size=101, shuffle=False, drop_last=False)] == [101, 101, 1]
    assert [len(b.ids) for b in PackedBatchLoader(ds, batch_size=100, shuffle=False)] == [100, 100, 3]
    assert len(PackedBatchLoader(ds, batch_size=101)) == 2 and len(PackedBatchLoader(ds, batch_size=100)) == 3
    got = np.concatenate([b.ids for b in PackedBatchLoader(ds, batch_size=64, shuffle=False, pack_tiles=False)])
    assert np.array_equal(got, np.arange(N))
    a = np.concatenate([b.ids for b in PackedBatchLoader(ds, batch_size=64, shuffle=True)])                # unseeded
    assert np.array_equal(np.sort(a), np.arange(N))


def test_ranks_partition_the_epoch_like_distributed_sampler(data):
    mgs, ds = data
    world = 4
    per_rank = [np.concatenate([b.ids for b in PackedBatchLoader(ds, batch_size=16, shuffle=True, seed=7, rank=r, world=world,
                                                                   pack_tiles=False)])
                for r in range(world)]
    assert {len(x) for x in per_rank} == {51}                                                              # ceil(203 / 4)
    order = np.arange(N)
    np.random.default_rng(7).shuffle(order)
    padded = np.concatenate([order, order[:1]])
    for r in range(world):
        assert np.array_equal(per_rank[r], padded[r::world])
    assert np.array_equal(epoch_shard(np.arange(5), 1, 2), [1, 3, 0]) and np.array_equal(epoch_shard(np.arange(5), 0, 1), np.arange(5))
    torch_ds = torch.utils.data.distributed.DistributedSampler(list(range(N)), num_replicas=world, rank=2, shuffle=False)
    ours = np.concatenate([b.ids for b in PackedBatchLoader(ds, batch_size=16, shuffle=False, rank=2, world=world,
                                                            pack_tiles=False)])
    assert np.array_equal(ours, np.fromiter(iter(torch_ds), dtype=np.int64))


def test_side_arrays_and_early_exit(data):
    mgs, ds = data
    Y = np.arange(N, dtype=np.float32)[:, None] * 2.0
    w = np.ones(N, dtype=np.float32)
    loader = PackedBatchLoader(ds, batch_size=20, shuffle=True, seed=3, arrays={"Y": Y, "w": w})
    for i, b in enumerate(loader):
        assert torch.equal(b.extras["Y"][:, 0], torch.from_numpy(b.ids.astype(np.float32) * 2.0)) and b.extras["w"].shape == (len(b.ids),)
        if i == 2:
            break                       # abandoning the iterator must not leave the producer thread hanging
    t0 = time.time()
    assert sum(len(b.ids) for b in loader) == N and time.time() - t0 < 10
    with pytest.raises(ValueError):
        PackedBatchLoader(ds, arrays={"Y": Y[:-1]})
    with pytest.raises(ValueError):
        PackedBatchLoader(ds, prefetch=1)


def test_tile_packing_keeps_batch_membership_and_fills_tiles():
    from chemprop_b200 import _lib
    from chemprop_b200.data import tile_packing_order, tile_packing_order_of

    mgs = make_molecules(4000, seed=1)
    ds = PackedMolGraphDataset.from_molgraphs(mgs)
    plain = PackedBatchLoader(ds, batch_size=2000, shuffle=True, seed=2, pack_tiles=False)
    packed = PackedBatchLoader(ds, batch_size=2000, shuffle=True, seed=2)
    for a, b in zip(plain, packed):
        assert np.array_equal(np.sort(a.ids), np.sort(b.ids)) and not np.array_equal(a.ids, b.ids)
        ta, tb = a.bmg._meta_host[_lib.META_N_TILES], b.bmg._meta_host[_lib.META_N_TILES]
        rows = b.bmg.E.shape[0]
        assert tb < 0.9 * ta and rows / (128 * tb) > 0.9, (ta, tb)
        assert b.bmg._meta_host[_lib.META_MAX_TILE_ROWS] <= 128
        _check_batch(b, mgs)
    order = tile_packing_order_of(mgs[:500])
    assert np.array_equal(np.sort(order), np.arange(500))
    # degenerate inputs: empty, single-atom molecules (no edges: bounded by the 128-atom cap), an oversized molecule
    assert tile_packing_order([], []).shape == (0,)
    o = tile_packing_order([1] * 300, [0] * 300)
    assert np.array_equal(np.sort(o), np.arange(300))
    o = tile_packing_order([90, 10, 10, 70], [200, 20, 20, 108])
    assert np.array_equal(np.sort(o), np.arange(4)) and o[0] == 0          # the oversized one sits alone, first
    with pytest.raises(ValueError):
        tile_packing_order([1, 2], [1])


def test_plan_prefetch_thread_of_the_resident_path(data):
    """The resident data set's loader path (`_resident_batches`: plans made `prefetch` batches ahead on a thread, batches
    assembled by the consumer) driven over the HOST data set, where `batch(ids, plan=...)` takes the same plan: same batches as
    the host path, epoch boundaries crossed by `epochs=None`, and a consumer that leaves early (bounded queue full, producer
    already past its last batch) neither hangs nor leaves the thread behind."""
    import threading

    mgs, ds = data
    a = PackedBatchLoader(ds, batch_size=32, shuffle=True, seed=8, prefetch=2)
    b = PackedBatchLoader(ds, batch_size=32, shuffle=True, seed=8, prefetch=2)
    host = [x.ids for x in a] + [x.ids for x in a]
    it = b._resident_batches(epochs=None)                       # two epochs and a bit, without a drain in between
    got = [next(it) for _ in range(len(host) + 2)]
    for x in got:
        _check_batch(x, mgs)
    assert all(np.array_equal(x.ids, y) for x, y in zip(got, host))
    it.close()

    c = PackedBatchLoader(ds, batch_size=64, shuffle=False, prefetch=2)          # 4 batches: the queue (2) fills up at once
    it = c._resident_batches(epochs=1)
    first = next(it)
    _check_batch(first, mgs)
    time.sleep(0.3)                                             # producer: all plans made, blocked on the full queue
    t0 = time.perf_counter()
    it.close()                                                  # the consumer goes away
    assert time.perf_counter() - t0 < 2.0
    assert not [t for t in threading.enumerate() if t.name == "packed-batch-planner" and t.is_alive()]
