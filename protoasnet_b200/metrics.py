"""Loss / metric consumers of the head outputs, evaluated on the device (SURVEY.md section 8(f) row 3).

Same class names, constructor arguments and ``compute`` signatures as the reference (src/loss/loss.py) for the three
terms that only read the head's outputs, plus the prototype diversity counters the agents keep per epoch:

  ``ClusterRoiFeat``      src/loss/loss.py:99-138       -sum_n max_{j in class y_n} similarity[n, j]
  ``SeparationRoiFeat``   src/loss/loss.py:141-187      sum_n sum_{k != y_n, k not abstention} max_{j in class k} similarity[n, j]
  ``L_norm``              src/loss/loss.py:229-250      occurrence maps, p in {1, 2}, norm over the trailing spatial dims
  ``DiversityCounters``   src/agents/Video_XProtoNet_e2e.py:158-173 (torch.sort on the CPU + np.add.at every step)

Each forward is one small kernel of libpasn_b200.so; nothing leaves the GPU until ``.item()`` / ``result()`` is asked
for.  Gradients (these terms sit inside the training loss) are provided by autograd Functions whose backward is a
scatter / an elementwise product of what the kernel already produced (arg-max indices, row norms).
"""
from __future__ import annotations

import ctypes as C
import logging
from typing import Optional

import numpy as np
import torch

from . import _lib


def _stream(dev):
    return torch.cuda.current_stream(dev).cuda_stream


def _check_sim(similarities: torch.Tensor):
    if not similarities.is_cuda:
        raise _lib.PasnError("protoasnet_b200.metrics needs CUDA tensors: there is no CPU implementation of this path")
    if similarities.dim() != 2:
        raise _lib.PasnError("similarities must be [N, P]")


class _ClassMax(torch.autograd.Function):
    """similarities [N,P] fp32, labels [N] int64 -> (cluster_sum, separation_sum) as float64 scalars on the device."""

    @staticmethod
    def forward(ctx, similarities, target, num_classes, abstain):
        _check_sim(similarities)
        lib = _lib.load()
        s = similarities.detach().to(torch.float32).contiguous()
        t = target.detach().to(device=s.device, dtype=torch.int64).contiguous()
        n, p = s.shape
        sums = torch.zeros(2, dtype=torch.float64, device=s.device)
        arg = torch.empty((n, num_classes), dtype=torch.int32, device=s.device)
        with torch.cuda.device(s.device):
            _lib.check(lib.pasn_similarity_stats(s.data_ptr(), t.data_ptr(), n, p, num_classes, int(abstain), 0, 0, 0,
                                                 None, arg.data_ptr(), sums.data_ptr(), None, None, _stream(s.device)),
                       "pasn_similarity_stats")
        ctx.save_for_backward(arg, t)
        ctx.shape, ctx.num_classes, ctx.abstain, ctx.dtype = (n, p), num_classes, bool(abstain), similarities.dtype
        return sums[0], sums[1]

    @staticmethod
    def backward(ctx, g_cluster, g_sep):
        arg, t = ctx.saved_tensors
        n, p = ctx.shape
        k = ctx.num_classes
        onehot = torch.nn.functional.one_hot(t, num_classes=k).to(torch.float64)        # [N,K]
        w = torch.zeros((n, k), dtype=torch.float64, device=arg.device)
        if g_cluster is not None:
            w = w - g_cluster.to(torch.float64) * onehot
        if g_sep is not None:
            neg = 1.0 - onehot
            if ctx.abstain:
                neg[:, -1] = 0.0
            w = w + g_sep.to(torch.float64) * neg
        grad = torch.zeros((n, p), dtype=torch.float64, device=arg.device)
        grad.scatter_add_(1, arg.to(torch.int64), w)
        return grad.to(ctx.dtype), None, None, None


def _reduce(total: torch.Tensor, n: int, reduction: str) -> torch.Tensor:
    # 'mean' in the reference is loss.mean(dim=0).sum(): the batch sum divided by N
    if reduction == "mean":
        return total / max(n, 1)
    if reduction == "sum":
        return total
    raise ValueError(f"reduction must be 'mean' or 'sum', got {reduction!r}")


class ClusterRoiFeat(object):
    """Cluster cost on the similarity scores (reference: src/loss/loss.py:99-138)."""

    def __init__(self, loss_weight, num_classes=4, reduction="sum"):
        self.num_classes, self.loss_weight, self.reduction = num_classes, loss_weight, reduction
        logging.info(f"setup ROI-Based Cluster Loss with loss_weight:{loss_weight}, for num_classes:{num_classes}, "
                     f"and reduction:{reduction}")

    def compute(self, similarities, target):
        if self.loss_weight == 0:
            return torch.tensor(0, device=target.device)
        cluster, _ = _ClassMax.apply(similarities, target, self.num_classes, False)
        return (self.loss_weight * _reduce(cluster, similarities.shape[0], self.reduction)).to(torch.float32)


class SeparationRoiFeat(object):
    """Separation cost on the similarity scores (reference: src/loss/loss.py:141-187)."""

    def __init__(self, loss_weight, num_classes=4, reduction="sum", abstain_class=True):
        self.num_classes, self.loss_weight, self.reduction = num_classes, loss_weight, reduction
        self.abstain_class = abstain_class
        logging.info(f"setup ROI-Based Separation Loss with loss_weight:{loss_weight}, for num_classes:{num_classes}, "
                     f"and reduction:{reduction}")

    def compute(self, similarities, target):
        if self.loss_weight == 0:
            return torch.tensor(0, device=target.device)
        _, sep = _ClassMax.apply(similarities, target, self.num_classes, self.abstain_class)
        return (self.loss_weight * _reduce(sep, similarities.shape[0], self.reduction)).to(torch.float32)


class _OccNorm(torch.autograd.Function):
    """occurrence maps [N,P,1,(T),H,W] -> sum over (n,p) of the p-norm over the spatial dims (float64 device scalar)."""

    @staticmethod
    def forward(ctx, occ, p):
        if not occ.is_cuda:
            raise _lib.PasnError("protoasnet_b200.metrics needs CUDA tensors: there is no CPU implementation of this path")
        lib = _lib.load()
        o = occ.detach()
        if o.dtype not in _lib.DTYPES:
            o = o.to(torch.float32)
        o = o.contiguous()
        rows = int(o.shape[0] * o.shape[1])
        s = int(o.numel() // max(rows, 1))
        total = torch.zeros(1, dtype=torch.float64, device=o.device)
        norms = torch.empty(rows, dtype=torch.float32, device=o.device)
        with torch.cuda.device(o.device):
            _lib.check(lib.pasn_occurrence_lnorm(o.data_ptr(), _lib.DTYPES[o.dtype],
                                                 rows, s, int(p), total.data_ptr(), norms.data_ptr(), _stream(o.device)),
                       "pasn_occurrence_lnorm")
        ctx.save_for_backward(occ, norms)
        ctx.p = int(p)
        return total[0]

    @staticmethod
    def backward(ctx, g):
        occ, norms = ctx.saved_tensors
        o = occ.detach().to(torch.float32)
        if ctx.p == 1:
            grad = torch.sign(o)
        else:
            nrm = norms.reshape(occ.shape[0], occ.shape[1], *([1] * (occ.dim() - 2)))
            grad = torch.where(nrm > 0, o / nrm.clamp_min(1e-38), torch.zeros_like(o))
        return (g.to(torch.float32) * grad).to(occ.dtype), None


class L_norm(object):
    """L1 / L2 regulariser (reference: src/loss/loss.py:229-250).  The occurrence-map use -- ``compute(occurrence_map,
    dim=<all trailing spatial dims>)``, src/agents/XProtoNet_Base.py:355, Video_XProtoNet_e2e.py:96 -- runs in the
    library; any other call (e.g. the masked last-layer term, a [K,P] tensor) is a handful of elements and stays a
    plain PyTorch expression on the device."""

    def __init__(self, mask=None, p=1, loss_weight=1e-4, reduction="sum"):
        self.mask, self.p, self.loss_weight, self.reduction = mask, p, loss_weight, reduction
        logging.info(f"setup L{p}-Norm Loss with loss_weight:{loss_weight}, with reduction:{reduction}")

    def compute(self, tensor, dim=None):
        if self.loss_weight == 0:
            return torch.tensor(0, device=tensor.device)
        spatial = None
        nd = tensor.dim()
        if dim is not None and nd in (5, 6) and tensor.shape[2] == 1:      # [N,P,1,(T),H,W], norm over (T),H,W
            dims = sorted(d % nd for d in (dim if isinstance(dim, (tuple, list)) else (dim,)))
            if dims == list(range(3, nd)):
                spatial = dims
        if spatial is not None and self.mask is None and self.p in (1, 2) and tensor.is_cuda:
            total = _OccNorm.apply(tensor, self.p)
            return (self.loss_weight * _reduce(total, tensor.shape[0], self.reduction)).to(torch.float32)
        t = tensor if self.mask is None else self.mask.to(tensor.device) * tensor
        loss = t.norm(p=self.p, dim=dim)
        loss = loss.mean(dim=0).sum() if self.reduction == "mean" else loss.sum()
        return self.loss_weight * loss


class DiversityCounters:
    """Per-epoch prototype usage statistics kept on the device (reference: Video_XProtoNet_e2e.py:158-173 sorts the
    similarities on the CPU and updates a numpy array every step)."""

    def __init__(self, num_prototypes: int, n_specific: int = 30, top_specific: int = 5, top_rest: int = 2,
                 abstain_class: bool = True, device="cuda"):
        self.P, self.n_specific = int(num_prototypes), int(n_specific)
        self.top_specific, self.top_rest = int(top_specific), int(top_rest if abstain_class else 0)
        self.count = torch.zeros(self.P, dtype=torch.int64, device=device)
        self.simscore_cumsum = torch.zeros(self.P, dtype=torch.float64, device=device)

    @torch.no_grad()
    def update(self, similarities: torch.Tensor):
        _check_sim(similarities)
        lib = _lib.load()
        s = similarities.detach().to(torch.float32).contiguous()
        n, p = s.shape
        if p != self.P:
            raise _lib.PasnError("similarity width does not match the counters")
        with torch.cuda.device(s.device):
            _lib.check(lib.pasn_similarity_stats(s.data_ptr(), None, n, p, 1, 0, self.n_specific, self.top_specific,
                                                 self.top_rest, None, None, None, self.count.data_ptr(),
                                                 self.simscore_cumsum.data_ptr(), _stream(s.device)),
                       "pasn_similarity_stats")

    def result(self):
        """(count_array [P] int64, simscore_cumsum [P] float64) as numpy arrays."""
        return self.count.cpu().numpy(), self.simscore_cumsum.cpu().numpy()
