"""CPU tests of how a multi-rank push splits a DataLoader: the shard plan (batches per rank, global offsets, the owner of a
global clip index), the batch list rank 0 draws and broadcasts (gloo world of 2), the per-rank loaders built from it,
which fetch only their own batches, and the argument checks of the winner side-data capture (pasn_push_capture)."""
import os

import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from protoasnet_b200 import _lib
from protoasnet_b200 import push as pushmod


class _Indexed(torch.utils.data.Dataset):
    def __init__(self, n, log=None):
        self.n, self.log = n, log

    def __len__(self):
        return self.n

    def __getitem__(self, i):
        if self.log is not None:
            self.log.append(int(i))
        return {"cine": torch.full((2,), float(i)), "target_AS": i % 3, "filename": f"clip_{i}"}


def _plan(loader, world):
    return pushmod.ShardPlan([len(b) for b in pushmod.loader_batches(loader)], world)


def _owners(plan):
    return [plan.owner(i) for i in range(plan.n_total)]


def test_plan_batch_count_not_divisible_by_world():
    plan = _plan(torch.utils.data.DataLoader(_Indexed(33), batch_size=5), 2)      # 7 batches: 5 x 6 + 3
    assert plan.sizes == [5] * 6 + [3]
    assert plan.bounds == [(0, 4), (4, 7)]
    assert plan.starts == [0, 20] and plan.counts == [20, 13] and plan.n_total == 33
    assert _owners(plan) == [0] * 20 + [1] * 13
    plan3 = pushmod.ShardPlan(plan.sizes, 3)                                      # per = 3: 3 + 3 + 1 batches
    assert plan3.bounds == [(0, 3), (3, 6), (6, 7)] and plan3.starts == [0, 15, 30] and plan3.counts == [15, 15, 3]


def test_plan_drop_last():
    plan = _plan(torch.utils.data.DataLoader(_Indexed(33), batch_size=5, drop_last=True), 4)
    assert plan.sizes == [5] * 6
    assert plan.bounds == [(0, 2), (2, 4), (4, 6), (6, 6)]
    assert plan.starts == [0, 10, 20, 30] and plan.counts == [10, 10, 10, 0]
    assert _owners(plan) == [0] * 10 + [1] * 10 + [2] * 10
    for bad in (30, 32, -1):                                                     # dropped clips are not in the push set
        try:
            plan.owner(bad)
        except ValueError:
            continue
        raise AssertionError(f"owner({bad}) should raise")


def test_plan_more_ranks_than_batches():
    plan = _plan(torch.utils.data.DataLoader(_Indexed(7), batch_size=4), 4)       # 2 batches, 4 ranks
    assert plan.bounds == [(0, 1), (1, 2), (2, 2), (2, 2)]
    assert plan.starts == [0, 4, 7, 7] and plan.counts == [4, 3, 0, 0]
    assert _owners(plan) == [0] * 4 + [1] * 3
    empty = pushmod.ShardPlan([], 3)                                              # an empty loader
    assert empty.bounds == [(0, 0)] * 3 and empty.n_total == 0


def test_loaders_without_a_batch_sampler_keep_the_iterate_and_skip_path():
    class _Stream(torch.utils.data.IterableDataset):
        def __iter__(self):
            return iter(range(5))

    assert pushmod.loader_batches(torch.utils.data.DataLoader(_Stream(), batch_size=2)) is None
    assert pushmod.loader_batches(torch.utils.data.DataLoader(_Indexed(5), batch_size=None)) is None
    assert pushmod.loader_batches([{"cine": torch.zeros(1, 2)}]) is None


class _ShuffledBatches(torch.utils.data.Sampler):
    """A custom batch sampler of uneven batches whose order depends on its seed: ranks given different seeds would
    disagree unless the batch list is drawn once and broadcast."""

    def __init__(self, n, seed):
        self.n, self.seed = n, seed

    def __iter__(self):
        g = torch.Generator().manual_seed(self.seed)
        perm = torch.randperm(self.n, generator=g).tolist()
        cuts = [0, 3, 4, 9, 11, 12, self.n]
        return iter([perm[a:b] for a, b in zip(cuts[:-1], cuts[1:])])

    def __len__(self):
        return 6


def _collate(samples):
    out = torch.utils.data.default_collate(samples)
    out["collated_by"] = "custom"
    return out


def _worker(rank, world, port, ret):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        log = []
        loader = torch.utils.data.DataLoader(_Indexed(17, log), batch_sampler=_ShuffledBatches(17, seed=100 + rank),
                                             collate_fn=_collate)
        batches = pushmod.loader_batches(loader)
        lo, hi = pushmod.shard_bounds(len(batches), rank, world)
        seen = []
        for data in pushmod.shard_loader(loader, batches[lo:hi]):
            assert data["collated_by"] == "custom"
            seen.append([int(v) for v in data["cine"][:, 0]])
        ret[rank] = {"batches": batches, "seen": seen, "fetched": log}
    finally:
        dist.destroy_process_group()


def test_custom_batch_sampler_is_broadcast_and_each_rank_fetches_its_slice_gloo():
    ret = mp.Manager().dict()
    mp.spawn(_worker, args=(2, 29541, ret), nprocs=2, join=True)
    b0, b1 = ret[0]["batches"], ret[1]["batches"]
    assert b0 == b1 == list(_ShuffledBatches(17, seed=100))                      # rank 0's draw, on every rank
    plan = pushmod.ShardPlan([len(b) for b in b0], 2)
    assert plan.bounds == [(0, 3), (3, 6)] and plan.starts == [0, 9] and plan.counts == [9, 8]
    for r in range(2):
        lo, hi = plan.bounds[r]
        assert ret[r]["seen"] == b0[lo:hi]                                        # its batches, in loader order
        assert sorted(ret[r]["fetched"]) == sorted(i for b in b0[lo:hi] for i in b)   # and nothing else was loaded
    assert sorted(ret[0]["fetched"] + ret[1]["fetched"]) == list(range(17))     # every clip exactly once overall


def test_capture_rejects_bad_arguments_without_gpu():
    lib = _lib.load()
    fake = 1 << 20                                   # never dereferenced: every call below returns before any launch

    def slots(n, **kw):
        arr = (_lib.PasnCaptureSlot * max(n, 1))()
        for s in arr:
            s.src, s.dst, s.row_bytes, s.clip_stride_bytes, s.proto_stride_bytes = fake, fake, 16, 16, 0
            for k, v in kw.items():
                setattr(s, k, v)
        return arr

    ok = slots(2)
    assert lib.pasn_push_capture(fake, 4, 0, 0, ok, 2, None) == 0                # no clips: nothing to do
    assert lib.pasn_push_capture(fake, 4, 0, 3, slots(1, row_bytes=0), 1, None) == 0   # empty rows: nothing to do
    bad = [
        (None, 4, 0, 3, ok, 2),                      # no keys
        (fake, 0, 0, 3, ok, 2),                      # P = 0
        (fake, 4, -1, 3, ok, 2),                     # negative global offset
        (fake, 4, 0, -1, ok, 2),                     # negative N
        (fake, 4, (1 << 32) - 2, 3, ok, 2),          # clip indices beyond the 32 bits a key holds
        (fake, 4, 0, 3, None, 2),                    # no slots
        (fake, 4, 0, 3, ok, 0),                      # zero slots
        (fake, 4, 0, 3, slots(9), 9),                # more than PASN_CAPTURE_MAX_SLOTS
        (fake, 4, 0, 3, slots(1, row_bytes=-16), 1),
        (fake, 4, 0, 3, slots(1, clip_stride_bytes=-1), 1),
        (fake, 4, 0, 3, slots(1, proto_stride_bytes=-1), 1),
        (fake, 4, 0, 3, slots(1, src=None), 1),
        (fake, 4, 0, 3, slots(1, dst=None), 1),
    ]
    for args in bad:
        assert lib.pasn_push_capture(*args, None) == -1, args
