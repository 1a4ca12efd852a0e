"""push_prototypes over a data loader on the GPU: the device-side winner capture (pasn_push_capture) against torch
indexing, no host synchronisation per batch, and a push on several ranks (2 gloo ranks sharing one GPU; 2 / 4 / 8 NCCL
ranks where the node has the GPUs) that loads each clip once, on the rank that owns its batch, and writes one
prototypes_info.pickle equal to the single-process one."""
import glob
import os
import pickle
import warnings

import numpy as np
import pytest
import torch

from protoasnet_b200 import _lib, synth
from protoasnet_b200 import push as pushmod
from tests.test_push_dist_cpu import _NONE, _pack
from tests.util import build_model

pytestmark = pytest.mark.gpu


def test_capture_kernel_matches_torch_indexing():
    lib = _lib.load()
    dev = torch.device("cuda")
    P, N, off = 11, 6, 100
    # per prototype: winner clip (global index) or None = no candidate; 99, 106 and 200 lie outside this call's clips
    win = [100, 105, 103, None, 99, 106, 100, 200, 102, None, 105]
    keys = np.array([_NONE if i is None else _pack(0.25 + 0.01 * p, i) for p, i in enumerate(win)], dtype=np.uint64)
    key = torch.from_numpy(keys.view(np.int64).copy()).to(dev)
    g = torch.Generator(device=dev).manual_seed(3)

    def rnd(*shape, dtype=torch.float32):
        return torch.randn(shape, device=dev, generator=g).to(dtype)

    odd = rnd(N * P * 8 + 1, dtype=torch.float16)[1:].view(N, P, 8)      # source 2 bytes off 16-byte alignment
    cases = [  # (source, per-prototype rows?)
        (rnd(N, P, 5), True),                                  # fp32 occurrence rows of 20 bytes
        (rnd(N, P, 1, 2, 3, dtype=torch.bfloat16), True),      # bf16, 12-byte rows
        (rnd(N, P, 8, dtype=torch.float16), True),             # fp16, 16-byte rows: vector copy
        (odd, True),                                           # fp16 at a misaligned address: byte copy
        (rnd(N, 4), False),                                    # fp32 logits (per clip)
        (rnd(N, 3, 5, 7, dtype=torch.bfloat16), False),        # bf16 clip, 210-byte rows
        (rnd(N, 3, 4, 4, 4, dtype=torch.float16), False),      # fp16 clip
        (rnd(N, 3, 16, 32, 32), False),                        # fp32 clip of 192 KB: split over several blocks
    ]
    assert len(cases) == _lib.PASN_CAPTURE_MAX_SLOTS
    dsts, slots = [], (_lib.PasnCaptureSlot * len(cases))()
    for s, (src, per_proto) in zip(slots, cases):
        row_shape = src.shape[2:] if per_proto else src.shape[1:]
        dst = rnd(P, *row_shape, dtype=src.dtype)
        dsts.append((dst, dst.clone()))
        row = dst[0].numel() * dst.element_size()
        s.src, s.dst, s.row_bytes = src.data_ptr(), dst.data_ptr(), row
        s.clip_stride_bytes = src.stride(0) * src.element_size()
        s.proto_stride_bytes = src.stride(1) * src.element_size() if per_proto else 0
    st = torch.cuda.current_stream().cuda_stream
    _lib.check(lib.pasn_push_capture(key.data_ptr(), P, off, N, slots, len(cases), st), "pasn_push_capture")
    _lib.check(lib.pasn_push_capture(key.data_ptr(), P, off, 0, slots, len(cases), st), "pasn_push_capture (N = 0)")
    torch.cuda.synchronize()
    for (src, per_proto), (dst, before) in zip(cases, dsts):
        exp = before.clone()
        for p, i in enumerate(win):
            if i is not None and off <= i < off + N:
                exp[p] = src[i - off, p] if per_proto else src[i - off]
        assert torch.equal(dst, exp), (src.dtype, tuple(src.shape), per_proto)
    assert lib.pasn_debug_fault() == 0


class _ToBF16(torch.nn.Module):
    """Backbone stand-in: the loader yields fp32 clips (what the pickle stores), the head runs in bf16 mode."""

    def __init__(self, c):
        super().__init__()
        self.out_channels = c

    def forward(self, x):
        return x.bfloat16()


def _model(cfg, device="cuda"):
    dims = synth.CONFIGS[cfg]
    sd = synth.make_head_params(dims, seed=11, bias_scale=0.05, bf16_round=(cfg != "tiny_video"))
    m = build_model(dims, sd, device=device)
    if cfg != "tiny_video":
        m.cnn_backbone = _ToBF16(dims.C)
    return m


class _WindowSet(torch.utils.data.Dataset):
    """Like the reference's train_push set (src/data/as_dataloader.py:246-255): every __getitem__ draws a random window,
    here seeded by the index so that two runs over the same set see the same clips.  Fetched indices are appended to
    ``log_path``."""

    def __init__(self, cfg, n, log_path=None):
        dims = synth.CONFIGS[cfg]
        self.x = torch.from_numpy(synth.make_features(dims, n, seed=4))
        self.y = torch.from_numpy(synth.push_labels(n, dims.K - 1, seed=9))
        self.log_path = log_path

    def __len__(self):
        return self.x.shape[0]

    def __getitem__(self, i):
        g = torch.Generator().manual_seed(1000 + i)
        clip = self.x[i] * (0.5 + torch.rand(self.x[i].shape, generator=g))
        if self.log_path is not None:
            with open(self.log_path, "a") as f:
                f.write(f"{i}\n")
        return {"cine": clip, "target_AS": self.y[i], "filename": f"clip_{i}"}


def _count_syncs(m, cfg, n_batches, batch, out_dir):
    loader = torch.utils.data.DataLoader(_WindowSet(cfg, n_batches * batch), batch_size=batch, pin_memory=True)
    with warnings.catch_warnings(record=True) as caught:
        warnings.simplefilter("always")
        torch.cuda.set_sync_debug_mode("warn")
        try:
            pushmod.push_prototypes(loader, m, root_dir_for_saving_prototypes=out_dir, log=lambda *a: None,
                                    replace_prototypes=False)
        finally:
            torch.cuda.set_sync_debug_mode("default")
    return [str(w.message).splitlines()[0] for w in caught if "synchroniz" in str(w.message)]


@pytest.mark.parametrize("cfg", ["tiny_video", "cfg3_video_b1024"])
def test_push_with_side_data_makes_no_host_sync_per_batch(cfg, tmp_path):
    m = _model(cfg)
    _count_syncs(m, cfg, 2, 4, str(tmp_path / "warm"))          # first call: weight packing, workspace, CUDA context
    few = _count_syncs(m, cfg, 4, 4, str(tmp_path / "a"))
    many = _count_syncs(m, cfg, 16, 4, str(tmp_path / "b"))
    assert len(few) == len(many), f"syncs grow with the batch count: 4 batches {few}, 16 batches {many}"
    assert os.path.exists(str(tmp_path / "b" / "prototypes_info.pickle"))


# ------------------------------------------------------------------------------------------------------------------------
# several ranks
# ------------------------------------------------------------------------------------------------------------------------
_CFG = "cfg3_video_b1024"
_CASES = [(37, 8), (6, 8)]   # (clips, batch): 5 batches, an odd count; 1 batch, so ranks >= 1 get none


def _case_dir(root, n, batch, peer):
    return os.path.join(root, f"n{n}_b{batch}_peer{peer}")


def _worker(rank, world, port, root, backend, peers):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dev = torch.device("cuda", rank if backend == "nccl" else 0)
    torch.cuda.set_device(dev)
    if backend == "nccl":
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    else:
        dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        for peer in peers:
            os.environ["PASN_PUSH_PEER"] = peer
            for n, batch in _CASES:
                d = _case_dir(root, n, batch, peer)
                ds = _WindowSet(_CFG, n, log_path=os.path.join(d, f"fetched.{rank}.txt"))
                m = _model(_CFG, device=dev)
                res = pushmod.push_prototypes(torch.utils.data.DataLoader(ds, batch_size=batch), m,
                                              root_dir_for_saving_prototypes=d, log=lambda *a: None)
                used_peer = any(v is not None for v in m.__dict__.get("_pasn_peer_records", {}).values())
                np.savez(os.path.join(d, f"rank{rank}.npz"), vec=m.prototype_vectors.data.cpu().numpy(),
                         index=res["index"].cpu().numpy(), n_side=len(res["side"]), used_peer=used_peer)
                dist.barrier()
    finally:
        dist.destroy_process_group()


def _check_multi_rank(world, backend, peers, port, tmp_path):
    import torch.multiprocessing as mp
    root = str(tmp_path)
    for peer in peers:
        for n, batch in _CASES:
            os.makedirs(_case_dir(root, n, batch, peer))
    mp.spawn(_worker, args=(world, port, root, backend, peers), nprocs=world, join=True)
    for n, batch in _CASES:
        ref_dir = str(tmp_path / f"single_n{n}")
        m = _model(_CFG)
        ref = pushmod.push_prototypes(torch.utils.data.DataLoader(_WindowSet(_CFG, n), batch_size=batch), m,
                                      root_dir_for_saving_prototypes=ref_dir, log=lambda *a: None)
        ref_info = pickle.load(open(os.path.join(ref_dir, "prototypes_info.pickle"), "rb"))
        ref_vec = m.prototype_vectors.data.cpu().numpy()
        plan = pushmod.ShardPlan([min(batch, n - i) for i in range(0, n, batch)], world)
        for peer in peers:
            d = _case_dir(root, n, batch, peer)
            what = f"{backend} world {world}, {n} clips in batches of {batch}, PASN_PUSH_PEER={peer}"
            fetched = []
            for r in range(world):
                f = os.path.join(d, f"fetched.{r}.txt")
                got = [int(v) for v in open(f).read().split()] if os.path.exists(f) else []
                assert sorted(got) == list(range(plan.starts[r], plan.starts[r] + plan.counts[r])), (what, r)
                fetched += got
            assert sorted(fetched) == list(range(n)), what                 # every clip fetched exactly once overall
            assert sorted(os.path.basename(p) for p in glob.glob(os.path.join(d, "prototypes_info*"))) == \
                ["prototypes_info.pickle"], what
            info = pickle.load(open(os.path.join(d, "prototypes_info.pickle"), "rb"))
            assert sorted(info) == sorted(ref_info), what
            for k in ref_info:
                assert ref_info[k].dtype == info[k].dtype and np.array_equal(ref_info[k], info[k]), (what, k)
            for r in range(world):
                z = np.load(os.path.join(d, f"rank{r}.npz"))
                assert np.array_equal(z["index"], ref["index"].cpu().numpy()), (what, r)
                assert np.array_equal(z["vec"], ref_vec), (what, r)            # prototype_vectors as one process pushes them
                assert int(z["n_side"]) == (len(info["prototype_ids"]) if r == 0 else 0), (what, r)
                assert bool(z["used_peer"]) == (peer == "1"), (what, r)


@pytest.mark.parametrize("world", [2, 4, 8])
def test_multi_rank_loader_push_matches_single_process(world, tmp_path):
    """NCCL ranks on separate GPUs, the merge over peer memory and over the all-gather."""
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs on one node")
    _check_multi_rank(world, "nccl", ("1", "0"), 29561 + world, tmp_path)


def test_two_rank_loader_push_on_one_gpu_gloo(tmp_path):
    """The same push with two gloo ranks sharing one GPU (all-gather merge): sharded loading, barrier, merge and the one
    pickle on a machine with a single GPU."""
    _check_multi_rank(2, "gloo", ("0",), 29571, tmp_path)
