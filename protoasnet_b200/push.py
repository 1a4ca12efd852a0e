"""Push / prototype projection on device, sharded across ranks.

Mirrors ``push_prototypes`` of the reference (src/utils/push_abs_revision.py:181-348) and the agent wrapper
``XProtoNet_Base.push`` (src/agents/XProtoNet_Base.py:149-167), re-designed for B200:

  load    a map-style DataLoader's batches are drawn once on rank 0 from its batch sampler and broadcast; rank r loads only
          its contiguous slice of them (``shard_bounds``), through a DataLoader over the same dataset with the same
          collation and workers.  Batches keep their single-process composition and global offsets.  A loader without a
          batch sampler (IterableDataset) is walked whole by every rank, each computing on its own slice.
  scan    per batch ONE fused launch pair computes the head, folds the class-restricted running argmin into packed keys
          ``orderable(fp32 dist) << 32 | global index`` AND keeps the winner's ``features_extracted`` row -- both in one
          device record ``[keys P x u64 | vectors P x D x f32]``.  The winner is captured in the pass that saw it, as the
          reference does (push_abs_revision.py:299-307): its push loader draws a random window per ``__getitem__``
          (src/data/as_dataloader.py:246-255), so a clip cannot be fetched a second time.  No per-batch D2H of features,
          distances, occurrence maps or input clips (push_abs_revision.py:278-285).
  side    with a save directory, the data the reference pickles (occurrence map, logits, input clip;
          push_abs_revision.py:301-325) is copied on the device by ``pasn_push_capture`` right after the scan of each
          batch, into per-prototype stashes; labels and file names stay on the host.  No host synchronisation per batch.
  merge   ONE collective: all-gather of the records (41 KB per rank at P=40, D=256), or one kernel over peer memory;
          every rank then picks, per prototype, the record with the smallest key (lowest distance, ties -> lowest global
          index) and overwrites ``prototype_vectors`` identically (push_abs_revision.py:342-346).  The loader path waits
          at a barrier first, so loader skew between ranks is absorbed there.
  pickle  the host reads the winners' indices once; the rank whose shard holds a winner copies its side rows to the host,
          one gather_object brings them to rank 0 (copied, never summed: bit-identical), and rank 0 writes the one
          ``prototypes_info.pickle``, identical to a single-process push over the same batches.

Defined behaviour where the reference crashes: a class-specific prototype whose class never occurs keeps its old
vector and reports index -1 (SURVEY.md section 7 'Empty class').  Rendering of prototype images / mp4s
(push_abs_revision.py:13-178, :329-340) is out of scope; the pickle with the same keys is written when a save
directory is given.
"""
from __future__ import annotations

import os
import pickle
import time
from typing import Dict, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _lib

_SIGN = -(1 << 63)


def proto_class_restriction(model, class_specific: bool = True, abstain_class: bool = True) -> torch.Tensor:
    """int32 [P]: class each prototype is restricted to, -1 = unrestricted.  push_abs_revision.py:226-239."""
    P = model.num_prototypes
    cls = torch.argmax(model.prototype_class_identity, dim=1).to(torch.int32)
    spec = torch.full((P,), bool(class_specific))
    if abstain_class:
        K = model.num_classes - 1
        assert K >= 2, "Abstention-push must have >= 2 classes not including abstain"
        per = P // model.num_classes
        spec[K * per: P] = False
    return torch.where(spec, cls, torch.full_like(cls, -1))


def new_best_key(P: int, device) -> torch.Tensor:
    key = torch.empty(P, dtype=torch.int64, device=device)  # storage for uint64 keys
    _init_key(key)
    return key


def _init_key(key: torch.Tensor) -> None:
    lib = _lib.load()
    dev = key.device
    with torch.cuda.device(dev):
        _lib.check(lib.pasn_push_init(key.data_ptr(), key.numel(), torch.cuda.current_stream(dev).cuda_stream), "pasn_push_init")


class PushRecord:
    """One rank's running push state in ONE device buffer ``[keys: P x u64 | vectors: P x D x f32]`` (include/pasn.h,
    ``pasn_push_record_bytes``): ``key`` and ``vec`` are views, ``buf`` is what the all-gather moves."""

    def __init__(self, P: int, D: int, device, buf: Optional[torch.Tensor] = None):
        self.P, self.D = int(P), int(D)
        nbytes = self.P * 8 + self.P * self.D * 4
        # ``buf``: caller-provided storage (a slice of peer-mapped symmetric memory, see PeerRecords)
        self.buf = torch.zeros(nbytes, dtype=torch.uint8, device=device) if buf is None else buf[:nbytes]
        self.peer = None   # (PeerRecords, buffer index, epoch) when the merge runs over peer memory
        self.key = self.buf[: self.P * 8].view(torch.int64)
        self.vec = self.buf[self.P * 8:].view(torch.float32).view(self.P, self.D)
        if self.buf.is_cuda:
            _init_key(self.key)
        else:   # host-side bookkeeping only (gloo tests of the merge logic)
            self.key.fill_(_KEY_NONE)


_KEY_NONE = (1 << 63) - 1   # INT64_MAX: no candidate


class PeerRecords:
    """Push records of all ranks of one node in peer-mapped (symmetric) memory, so that the merge is ONE kernel that reads the
    peers' records over NVLink (``pasn_push_merge_peers``) instead of a collective call.  Per rank: two record buffers
    (alternating from push to push: a rank that starts its next push never overwrites what a slower peer is still reading)
    and one epoch flag.  Built once per (model, device, P, D, group): the rendezvous is collective and not cheap."""

    def __init__(self, P: int, D: int, device, group=None):
        import torch.distributed as dist
        import torch.distributed._symmetric_memory as symm

        self.P, self.D = int(P), int(D)
        rec = self.P * 8 + self.P * self.D * 4
        self.stride = (rec + 255) // 256 * 256
        self.mem = symm.empty(2 * self.stride + 256, dtype=torch.uint8, device=device)
        self.mem.zero_()
        pg = group if group is not None else dist.group.WORLD
        self.handle = symm.rendezvous(self.mem, pg)
        self.rank, self.world = int(self.handle.rank), int(self.handle.world_size)
        ptrs = [int(q) for q in self.handle.buffer_ptrs]
        self.rec_ptrs = [torch.tensor([q + b * self.stride for q in ptrs], dtype=torch.int64, device=device) for b in (0, 1)]
        self.flag_ptrs = torch.tensor([q + 2 * self.stride for q in ptrs], dtype=torch.int64, device=device)
        self.epoch = 0
        torch.cuda.synchronize(device)
        dist.barrier(group=group)      # every rank's flags are zero before anybody can poll them

    def next_record(self) -> "PushRecord":
        self.epoch += 1
        b = self.epoch & 1
        rec = PushRecord(self.P, self.D, self.mem.device, buf=self.mem[b * self.stride: (b + 1) * self.stride])   # keys reset
        rec.peer = (self, b, self.epoch)
        return rec


def _peer_records(model, P: int, D: int, device, group=None) -> Optional[PeerRecords]:
    """PeerRecords for this model (cached), or None when the merge has to go through the all-gather: single rank, CPU
    bookkeeping, ``PASN_PUSH_PEER=0``, or symmetric memory not available for this group (decided once, by all ranks alike)."""
    import torch.distributed as dist

    _, world = _world(group)
    if world == 1 or torch.device(device).type != "cuda" or os.environ.get("PASN_PUSH_PEER", "1") == "0":
        return None
    cache = model.__dict__.setdefault("_pasn_peer_records", {})
    ck = (P, D, str(device), id(group))
    if ck not in cache:
        ok = torch.ones(1, dtype=torch.int32, device=device)
        pr = None
        try:
            pr = PeerRecords(P, D, device, group)
        except Exception as e:   # noqa: BLE001 -- any failure means "use the collective"; all ranks must agree
            ok.zero_()
            if os.environ.get("PASN_PUSH_PEER_VERBOSE"):
                print(f"[protoasnet_b200] peer-memory push merge unavailable: {e!r}")
        dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=group)
        cache[ck] = pr if int(ok.item()) == 1 else None
    return cache[ck]


def merge_keys(best_key: torch.Tensor, group=None) -> torch.Tensor:
    """All-reduce(MIN) of packed keys alone (kept for callers that only need indices).  Keys are stored with the top bit
    flipped (include/pasn.h), so the signed int64 order NCCL / gloo reduce with is the key order."""
    import torch.distributed as dist

    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(best_key, op=dist.ReduceOp.MIN, group=group)
    return best_key


def decode_keys(best_key: torch.Tensor):
    """-> (index int64 [P] (-1 = no candidate), distance fp32 [P])."""
    if not best_key.is_cuda:  # host-side bookkeeping only (gloo tests of the merge logic); no head compute here
        none = best_key == _KEY_NONE
        ku = best_key ^ _SIGN                      # back to the unsigned key bit pattern (held in an int64)
        o = (ku >> 32) & 0xFFFFFFFF
        u = torch.where((o & 0x80000000) != 0, o & 0x7FFFFFFF, (~o) & 0xFFFFFFFF)
        u = torch.where(u >= (1 << 31), u - (1 << 32), u).to(torch.int32)
        d = torch.where(none, torch.full_like(u, 0x7F800000), u).view(torch.float32)
        return torch.where(none, torch.full_like(best_key, -1), ku & 0xFFFFFFFF), d
    lib = _lib.load()
    P = best_key.numel()
    idx = torch.empty(P, dtype=torch.int64, device=best_key.device)
    d = torch.empty(P, dtype=torch.float32, device=best_key.device)
    with torch.cuda.device(best_key.device):
        _lib.check(lib.pasn_push_decode(best_key.data_ptr(), P, idx.data_ptr(), d.data_ptr(),
                                        torch.cuda.current_stream(best_key.device).cuda_stream), "pasn_push_decode")
    return idx, d


def _world(group=None):
    import torch.distributed as dist

    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(group), dist.get_world_size(group)
    return 0, 1


def gather_records(rec: PushRecord, group=None) -> Tuple[torch.Tensor, int]:
    """The one collective of a push: all-gather of the ranks' records -> (R records back to back, R)."""
    import torch.distributed as dist

    _, world = _world(group)
    if world == 1:
        return rec.buf, 1
    out = torch.empty(world * rec.buf.numel(), dtype=torch.uint8, device=rec.buf.device)
    if rec.buf.is_cuda:
        dist.all_gather_into_tensor(out, rec.buf, group=group)
    else:
        dist.all_gather(list(out.view(world, -1).unbind(0)), rec.buf, group=group)
    return out, world


def reduce_records(gathered: torch.Tensor, R: int, P: int, D: int):
    """Per prototype the record with the smallest key wins -> (index, distance, valid int32, vec [P,D])."""
    dev = gathered.device
    if not gathered.is_cuda:   # host-side bookkeeping only (gloo tests of the merge logic)
        recs = gathered.view(R, -1)
        keys = torch.stack([recs[r, : P * 8].view(torch.int64) for r in range(R)])
        vecs = torch.stack([recs[r, P * 8:].view(torch.float32).view(P, D) for r in range(R)])
        best, who = keys.min(dim=0)
        idx, d = decode_keys(best)
        valid = (idx >= 0).to(torch.int32)
        vec = vecs[who, torch.arange(P)] * valid[:, None]
        return idx, d, valid, vec
    lib = _lib.load()
    idx = torch.empty(P, dtype=torch.int64, device=dev)
    d = torch.empty(P, dtype=torch.float32, device=dev)
    valid = torch.empty(P, dtype=torch.int32, device=dev)
    vec = torch.zeros((P, D), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        _lib.check(lib.pasn_push_reduce(gathered.data_ptr(), R, P, D, idx.data_ptr(), d.data_ptr(), valid.data_ptr(),
                                        vec.data_ptr(), torch.cuda.current_stream(dev).cuda_stream), "pasn_push_reduce")
    return idx, d, valid, vec


def finish_push(model, rec: PushRecord, replace_prototypes=True, group=None):
    """One all-gather of the records, per-prototype minimum, prototype overwrite.  No host synchronisation.
    Returns dict(index, distance, features (P,D), valid)."""
    lib = _lib.load()
    if rec.peer is not None:
        # exchange + merge in one kernel over NVLink peer memory
        pr, b, epoch = rec.peer
        dev = rec.buf.device
        idx = torch.empty(rec.P, dtype=torch.int64, device=dev)
        dmin = torch.empty(rec.P, dtype=torch.float32, device=dev)
        valid = torch.empty(rec.P, dtype=torch.int32, device=dev)
        vec = torch.empty((rec.P, rec.D), dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            _lib.check(lib.pasn_push_merge_peers(pr.rec_ptrs[b].data_ptr(), pr.flag_ptrs.data_ptr(), pr.world, pr.rank,
                                                 epoch & 0xFFFFFFFF, rec.P, rec.D, idx.data_ptr(), dmin.data_ptr(),
                                                 valid.data_ptr(), vec.data_ptr(), torch.cuda.current_stream(dev).cuda_stream),
                       "pasn_push_merge_peers")
    else:
        gathered, R = gather_records(rec, group)
        idx, dmin, valid, vec = reduce_records(gathered, R, rec.P, rec.D)
    if replace_prototypes:
        pv = model.prototype_vectors.data
        dev = pv.device
        with torch.cuda.device(dev):
            _lib.check(lib.pasn_push_write_prototypes(pv.data_ptr(), vec.data_ptr(), valid.data_ptr(), rec.P, rec.D,
                                                      torch.cuda.current_stream(dev).cuda_stream),
                       "pasn_push_write_prototypes")
    return {"index": idx, "distance": dmin, "features": vec, "valid": valid, "side": {}}


def push_resident(model, features: torch.Tensor, labels: torch.Tensor, global_offset: int = 0, n_total: Optional[int] = None,
                  chunk: int = 8192, class_specific=True, abstain_class=True, replace_prototypes=True, group=None):
    """Push over backbone feature maps already resident on this rank's GPU (``features`` [n_local,C,*spatial],
    ``labels`` int64 [n_local]); ``global_offset`` = global index of local clip 0.  This is the path bench.py times."""
    dev = features.device
    P, D = model.num_prototypes, model.prototype_shape[1]
    # the class restriction only depends on the (fixed) prototype_class_identity buffer: built once per model / device, so a
    # push issues no host->device copy of its own (at 8 GPUs the fixed cost of a push is what limits its scaling)
    ck = (bool(class_specific), bool(abstain_class), str(dev))
    cache = model.__dict__.setdefault("_pasn_push_pc", {})
    pc = cache.get(ck)
    if pc is None:
        pc = cache[ck] = proto_class_restriction(model, class_specific, abstain_class).to(dev)
    peers = _peer_records(model, P, D, dev, group)
    rec = peers.next_record() if peers is not None else PushRecord(P, D, dev)
    n_local = features.shape[0]
    for i in range(0, n_local, chunk):
        model.push_scan(features[i:i + chunk], labels[i:i + chunk], pc, global_offset + i, rec.key, backbone=False,
                        best_vec=rec.vec)
    return finish_push(model, rec, replace_prototypes, group)


def shard_bounds(n_batches: int, rank: int, world: int) -> Tuple[int, int]:
    """Batches [lo, hi) of rank ``rank``: contiguous slices of ceil(n_batches / world) batches, so every batch has the
    composition it has in a single-process run (the trailing ranks get an empty slice when there are fewer batches)."""
    per = -(-n_batches // world)
    return min(rank * per, n_batches), min((rank + 1) * per, n_batches)


class ShardPlan:
    """Who pushes which clips: from the sizes of ALL batches in loader order, rank r takes the batches
    ``bounds[r]`` (``shard_bounds``) and so the global clips [starts[r], starts[r] + counts[r])."""

    def __init__(self, sizes: Sequence[int], world: int):
        self.sizes = [int(b) for b in sizes]
        self.world = int(world)
        cum = [0]
        for b in self.sizes:
            cum.append(cum[-1] + b)
        self.n_total = cum[-1]
        self.bounds = [shard_bounds(len(self.sizes), r, self.world) for r in range(self.world)]
        self.starts = [cum[lo] for lo, _ in self.bounds]
        self.counts = [cum[hi] - cum[lo] for lo, hi in self.bounds]

    def owner(self, index: int) -> int:
        """Rank whose shard holds global clip ``index``."""
        if not 0 <= index < self.n_total:
            raise ValueError(f"clip index {index} outside the push set [0, {self.n_total})")
        return next(r for r in range(self.world) if self.starts[r] <= index < self.starts[r] + self.counts[r])


def loader_batches(dataloader, group=None) -> Optional[list]:
    """The batches (lists of dataset indices) a map-style DataLoader yields, drawn once from its batch sampler on rank 0
    and broadcast, so that every rank agrees on them whatever the sampler.  None for a loader that has no batch sampler
    to draw from (an IterableDataset, ``batch_size=None``, or any other iterable)."""
    import torch.distributed as dist

    if not isinstance(dataloader, torch.utils.data.DataLoader) or dataloader.batch_sampler is None or \
            isinstance(dataloader.dataset, torch.utils.data.IterableDataset):
        return None
    rank, world = _world(group)
    obj = [[list(b) for b in dataloader.batch_sampler] if rank == 0 else None]
    if world > 1:
        src = 0 if group is None else dist.get_global_rank(group, 0)
        dist.broadcast_object_list(obj, src=src, group=group)
    return obj[0]


def shard_loader(dataloader, batches):
    """A DataLoader over ``dataloader.dataset`` that yields exactly ``batches``, with the original's collation, workers
    and memory pinning."""
    kw = dict(collate_fn=dataloader.collate_fn, num_workers=dataloader.num_workers, pin_memory=dataloader.pin_memory,
              worker_init_fn=dataloader.worker_init_fn, timeout=dataloader.timeout,
              multiprocessing_context=dataloader.multiprocessing_context, persistent_workers=dataloader.persistent_workers)
    if dataloader.num_workers > 0:
        kw["prefetch_factor"] = dataloader.prefetch_factor
    return torch.utils.data.DataLoader(dataloader.dataset, batch_sampler=batches, **kw)


class _SideCapture:
    """The side data the reference pickles for each prototype's winner (push_abs_revision.py:301-325), captured on the
    device in the pass that produced the minimum: after each batch's scan, ``pasn_push_capture`` copies the rows of the
    clips that improved a prototype into per-prototype stashes -- occurrence-map row [1,*spatial] (map dtype), logits [K]
    (fp32), input clip (loader dtype).  Labels and file names are host data the loader hands over anyway; they are kept
    per shard, by global position.  Nothing here waits for the device."""

    def __init__(self, P: int, dev):
        self.P, self.dev = P, dev
        self.stash = None           # [occurrence rows, logits, clips], allocated at the first batch
        self.start = None           # global index of this rank's first clip
        self.targets, self.names = [], []

    def batch(self, best_key, offset: int, x: torch.Tensor, out: dict, data_sample) -> None:
        occ, logits = out["occurrence_map"], out["logits"]
        x = x.contiguous()
        N = int(x.shape[0])
        if self.stash is None:
            self.start = offset
            self.stash = [torch.empty((self.P,) + tuple(t.shape[k:]), dtype=t.dtype, device=self.dev)
                          for t, k in ((occ, 2), (logits, 1), (x, 1))]
        elif tuple(x.shape[1:]) != tuple(self.stash[2].shape[1:]) or x.dtype != self.stash[2].dtype:
            raise _lib.PasnError(f"push with a save directory needs clips of one shape and dtype: got {tuple(x.shape[1:])} "
                                 f"{x.dtype} after {tuple(self.stash[2].shape[1:])} {self.stash[2].dtype}")
        slots = (_lib.PasnCaptureSlot * 3)()
        for s, src, dst, per_proto in zip(slots, (occ, logits, x), self.stash, (True, False, False)):
            row = dst[0].numel() * dst.element_size()
            s.src, s.dst, s.row_bytes = src.data_ptr(), dst.data_ptr(), row
            s.clip_stride_bytes, s.proto_stride_bytes = (row * self.P, row) if per_proto else (row, 0)
        lib = _lib.load()
        with torch.cuda.device(self.dev):
            _lib.check(lib.pasn_push_capture(best_key.data_ptr(), self.P, offset, N, slots, 3,
                                             torch.cuda.current_stream(self.dev).cuda_stream), "pasn_push_capture")
        self.targets.append(data_sample["target_AS"])
        names = data_sample.get("filename", None)
        self.names.extend(names[a] if names is not None else str(offset + a) for a in range(N))

    def rows(self, index, protos) -> Dict[int, tuple]:
        """Host copies of the side data of ``protos`` (winners in this rank's shard): p -> (occurrence-map row, logits,
        clip, gt, file name).  Copied, never computed on, so they carry the captured bits (-0.0 included)."""
        if not protos:
            return {}
        sel = torch.tensor(protos, dtype=torch.int64, device=self.dev)
        occ, logits, clips = (t.index_select(0, sel) for t in self.stash)
        occ, logits, clips = occ.float().cpu().numpy(), logits.cpu().numpy(), clips.cpu().numpy()
        gts = torch.cat(self.targets).tolist()
        return {p: (occ[t], logits[t], clips[t], int(gts[index[p] - self.start]), self.names[index[p] - self.start])
                for t, p in enumerate(protos)}


def _collect_side(cap: _SideCapture, res, plan: ShardPlan, group=None) -> Optional[Dict[int, tuple]]:
    """Side data of every winner, on rank 0 (None on the other ranks): each rank takes the rows of the winners in its
    shard off the device, and one gather_object brings them to rank 0, so the result is bit-identical to what a single
    process captures."""
    import torch.distributed as dist

    rank, world = _world(group)
    index = res["index"].cpu().tolist()                       # the one host read of the push
    protos = [p for p in range(cap.P) if index[p] >= 0]
    part = cap.rows(index, [p for p in protos if plan.owner(index[p]) == rank])
    if world == 1:
        return part
    gathered = [None] * world if rank == 0 else None
    with torch.cuda.device(cap.dev):
        dist.gather_object(part, gathered, dst=0 if group is None else dist.get_global_rank(group, 0), group=group)
    return {p: v for g in gathered for p, v in g.items()} if rank == 0 else None


def push_prototypes(
    dataloader,
    model,
    class_specific=True,
    abstain_class=True,
    preprocess_input_function=None,
    root_dir_for_saving_prototypes=None,
    epoch_number=None,
    log=print,
    prototype_img_filename_prefix=None,
    prototype_self_act_filename_prefix=None,
    proto_bound_boxes_filename_prefix=None,
    replace_prototypes=True,
    group=None,
):
    """Same signature and effect as the reference's ``push_prototypes`` (push_abs_revision.py:181-196).

    ``dataloader`` yields dicts with ``"cine"`` [B,3,(T),H,W], ``"target_AS"`` [B] and ``"filename"``, unshuffled
    (src/data/as_dataloader.py:65).  Every clip is seen exactly once: the winners' vectors and side data are captured
    on the device from the batch that produced them, so a loader whose ``__getitem__`` is random (as the reference's
    is) is fine, and no batch waits for the host.
    Under torch.distributed every rank calls this with the SAME loader.  A map-style DataLoader's batches are drawn on
    rank 0 and broadcast; rank r then loads only its contiguous slice of them (``shard_bounds``).  A loader without a
    batch sampler is iterated whole by every rank, each computing its slice.  Rank 0 writes the one
    ``prototypes_info.pickle`` and holds ``res["side"]``; it is ``{}`` on the other ranks.
    """
    model.eval()
    log(f"############## push at epoch {epoch_number} #################")
    start = time.time()
    proto_epoch_dir = None
    if root_dir_for_saving_prototypes is not None:
        proto_epoch_dir = root_dir_for_saving_prototypes if epoch_number is None else \
            os.path.join(root_dir_for_saving_prototypes, "epoch-" + str(epoch_number))
        os.makedirs(proto_epoch_dir, exist_ok=True)

    dev = model.prototype_vectors.device
    P, D = model.num_prototypes, model.prototype_shape[1]
    pc = proto_class_restriction(model, class_specific, abstain_class).to(dev)
    peers = _peer_records(model, P, D, dev, group)
    rec = peers.next_record() if peers is not None else PushRecord(P, D, dev)
    rank, world = _world(group)
    batches = None
    if world > 1:
        with torch.cuda.device(dev):
            batches = loader_batches(dataloader, group)
    if batches is not None:            # sharded loading: this rank fetches its own batches only
        sizes = [len(b) for b in batches]
        b_lo, b_hi = shard_bounds(len(sizes), rank, world)
        source = enumerate(shard_loader(dataloader, batches[b_lo:b_hi]), start=b_lo)
        offset = sum(sizes[:b_lo])
    else:                              # every rank walks the whole loader and computes on its slice
        sizes = []
        b_lo, b_hi = shard_bounds(len(dataloader), rank, world)
        source = enumerate(dataloader)
        offset = 0

    cap = _SideCapture(P, dev) if proto_epoch_dir is not None else None
    with torch.no_grad():
        for bi, data_sample in source:
            x = data_sample["cine"]
            B = x.shape[0]
            if batches is None:
                sizes.append(B)
            elif B != sizes[bi]:
                raise _lib.PasnError(f"batch {bi} holds {B} clips but its batch sampler listed {sizes[bi]} indices: "
                                     f"the collate_fn must keep one clip per index")
            if b_lo <= bi < b_hi:
                if preprocess_input_function is not None:
                    x = preprocess_input_function(x)
                xd = x.to(dev, non_blocking=True)
                y = data_sample["target_AS"].to(dev, non_blocking=True).to(torch.int64)
                fmap = model.cnn_backbone(xd)
                out = model.push_scan(fmap, y, pc, offset, rec.key, backbone=False, best_vec=rec.vec,
                                      want_occ=cap is not None)
                if cap is not None:
                    cap.batch(rec.key, offset, xd, out, data_sample)
            offset += B

    if world > 1:
        # ranks finish their shards at different times: wait here rather than in the merge, whose peer-memory wait is short
        import torch.distributed as dist
        with torch.cuda.device(dev):
            dist.barrier(group=group)
    with torch.no_grad():
        res = finish_push(model, rec, replace_prototypes, group)

    if cap is not None:
        side = _collect_side(cap, res, ShardPlan(sizes, world), group)
        if side:
            protos = sorted(side)
            occ, logits, clips, gts, names = (np.array([side[j][k] for j in protos]) for k in range(5))
            # the reference's pickle schema (push_abs_revision.py:309-325)
            info = {
                "prototype_ids": np.asarray(protos),
                "prototypes_filenames": names,
                "prototypes_src_imgs": clips,
                "prototypes_gts": gts,
                "prototypes_preds": logits,
                "prototypes_occurrence_maps": occ,
                "prototypes_similarity_to_src_ROIs": 1 - res["distance"][protos].double().cpu().numpy(),
            }
            with open(os.path.join(proto_epoch_dir, "prototypes_info.pickle"), "wb") as f:
                pickle.dump(info, f)
            res["side"] = {j: dict(zip(("occurrence_map", "logits", "image", "gt", "filename"), side[j])) for j in protos}
    log("\tpush time: \t{0}".format(time.time() - start))
    return res


def agent_push(agent, replace_prototypes=True):
    """``XProtoNet_Base.push`` (src/agents/XProtoNet_Base.py:149-167) for an agent-like object exposing
    ``current_epoch``, ``data_loaders['train_push']``, ``model`` and ``config``."""
    epoch = f"{agent.current_epoch}_pushed"
    return push_prototypes(
        dataloader=agent.data_loaders["train_push"], model=agent.model, abstain_class=agent.config["abstain_class"],
        preprocess_input_function=None,
        root_dir_for_saving_prototypes=os.path.join(agent.config["save_dir"], "img"), epoch_number=epoch,
        prototype_img_filename_prefix="prototype-img", prototype_self_act_filename_prefix="prototype-self-act",
        proto_bound_boxes_filename_prefix="bb", replace_prototypes=replace_prototypes)
