"""Drop-in prototype-head models: same class names, constructor kwargs, sub-module / parameter names,
``state_dict`` layout and method signatures as the reference, with the head computed by libpasn_b200.so.

Reference interface being mirrored (paths relative to the reference checkout):
  * ``Video_XProtoNet``            src/models/Video_XProtoNet.py:8-130
  * ``XProtoNet``                  src/models/XProtoNet.py:8-106   (PPNet 'regular' add-on minus Sigmoid, ProtoPNet.py:117-130)
  * ``construct_Video_XProtoNet``  src/models/Video_XProtoNet.py:154-178
  * ``construct_XProtoNet``        src/models/XProtoNet.py:132-159
  * ``MODELS`` / ``build``         src/models/model_builder.py:7-25

The backbone stays PyTorch (north_star); everything from its feature map to the logits runs in the CUDA
library.  There is NO PyTorch/CPU fallback for inference: a CPU tensor, or a missing library, raises.
Training through the head (SURVEY.md section 8f row 2): ``autograd_mode='kernel'`` runs ``requires_grad`` calls
through the library as well (forward as usual, backward = ``pasn_head_backward``, fp32 CUDA-core kernels that
recompute the forward intermediates); ``'composite'`` opts in to a differentiable PyTorch composite of the same maths
on the GPU; the default ``'error'`` refuses instead of silently switching.
"""
from __future__ import annotations

import ctypes as C
from copy import deepcopy
from typing import Dict, Optional, Tuple

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import _lib
from ._lib import PasnDims, PasnGrads, PasnPushArgs, PasnWeights


import os as _os

_DEBUG_SYNC = bool(int(_os.environ.get("PASN_DEBUG_SYNC", "0")))  # tests: surface kernel-internal fault codes


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


class _HeadRuntime:
    """Per-module launcher: owns the scratch buffer and the derived bf16 weight cache (never saved)."""

    def __init__(self, owner: "PrototypeHeadMixin"):
        self.owner = owner
        self._ws: Optional[torch.Tensor] = None
        self._packed: Dict = {}

    def _weights_struct(self, m) -> Tuple[PasnWeights, list]:
        a, o = m.add_on_layers, m.occurrence_module
        tensors = [a[0].weight, a[0].bias, a[2].weight, a[2].bias, o[0].weight, o[0].bias, o[2].weight, o[2].bias,
                   o[4].weight, m.prototype_vectors, m.last_layer.weight]
        for t in tensors:
            if t.dtype != torch.float32 or not t.is_contiguous():
                raise _lib.PasnError("head parameters must be contiguous fp32 (the state_dict layout of the reference)")
        w = PasnWeights(*[t.data_ptr() for t in tensors])
        return w, tensors

    def _workspace(self, lib, dims: PasnDims, device) -> torch.Tensor:
        need = int(lib.pasn_head_workspace_bytes(C.byref(dims)))
        if self._ws is None or self._ws.device != device or self._ws.numel() < need:
            self._ws = torch.empty(max(need, 256), dtype=torch.uint8, device=device)
        return self._ws

    def _packed_weights(self, lib, dims: PasnDims, w: PasnWeights, tensors, device, stream) -> Optional[torch.Tensor]:
        """Derived bf16 weight cache of the tensor-core path that serves ``dims`` (fused stage images or tiled planes),
        one entry per (shape, dtype, path); re-packed when a parameter's version counter or storage changes."""
        if not lib.pasn_tcgen05_supported(C.byref(dims)):
            return None
        slot = (str(device), dims.C, dims.D, dims.P, dims.dtype, dims.path)
        key = tuple((t.data_ptr(), t._version) for t in tensors[:9])
        ent = self._packed.get(slot)
        if ent is None or ent[0] != key:
            nbytes = int(lib.pasn_packed_weights_bytes(C.byref(dims)))
            buf = ent[1] if ent is not None and ent[1].numel() == nbytes else torch.empty(nbytes, dtype=torch.uint8, device=device)
            _lib.check(lib.pasn_pack_weights(C.byref(w), C.byref(dims), buf.data_ptr(), stream), "pasn_pack_weights")
            self._packed[slot] = (key, buf)
            ent = self._packed[slot]
        return ent[1]

    def make_dims(self, x: torch.Tensor, path: int) -> Tuple[PasnDims, torch.Tensor, Tuple[int, ...]]:
        m = self.owner
        if not x.is_cuda:
            raise _lib.PasnError("protoasnet_b200 head needs a CUDA tensor: there is no CPU implementation of this path")
        if x.dtype not in _lib.DTYPES:
            raise _lib.PasnError(f"unsupported feature dtype {x.dtype} (fp32, bf16 or fp16)")
        nd = x.dim() - 2
        if nd not in (2, 3):
            raise _lib.PasnError("feature map must be [N,C,H,W] or [N,C,T,H,W]")
        spatial = tuple(x.shape[2:])
        cl = torch.channels_last_3d if nd == 3 else torch.channels_last
        if x.is_contiguous():
            layout = _lib.PASN_LAYOUT_NCS
        elif x.is_contiguous(memory_format=cl):
            layout = _lib.PASN_LAYOUT_NSC
        else:
            x = x.contiguous()
            layout = _lib.PASN_LAYOUT_NCS
        S = 1
        for v in spatial:
            S *= int(v)
        P, D = int(m.prototype_shape[0]), int(m.prototype_shape[1])
        dims = PasnDims(int(x.shape[0]), int(x.shape[1]), D, P, int(m.num_classes), S, _lib.DTYPES[x.dtype], layout,
                        _lib.PASN_OCC_ABS, path)
        if dims.dtype == _lib.PASN_F16 and not _lib.load().pasn_tcgen05_supported(C.byref(dims)):
            raise _lib.PasnError(
                f"fp16 feature maps run on the tensor-core paths only (fused: D = 256, C % 64 == 0, C <= 1024, P <= 48, "
                f"S % 4 == 0, S >= 128; tiled: C % 64 == 0, D % 128 == 0; kernel_path not GENERIC), and this head "
                f"(C = {dims.C}, D = {D}, P = {P}, S = {S}, kernel_path = {path}) takes neither: pass x.float() or "
                f"x.bfloat16()")
        return dims, x, spatial

    def run(self, x: torch.Tensor, want_occ=True, want_feats=False, want_dist=False, push: Optional[dict] = None):
        """x: backbone feature map.  Returns dict(logits, similarity, occurrence_map, features_extracted, distance)."""
        lib = _lib.load()
        m = self.owner
        dims, x, spatial = self.make_dims(x, m.kernel_path)
        dev = x.device
        N, P, D, K = dims.N, dims.P, dims.D, dims.K
        if x.shape[1] != m.add_on_layers[0].weight.shape[1]:
            raise _lib.PasnError("feature map channel count does not match add_on_layers[0]")
        with torch.cuda.device(dev):
            stream = torch.cuda.current_stream(dev).cuda_stream
            w, tensors = self._weights_struct(m)
            for t in tensors:
                if t.device != dev:
                    raise _lib.PasnError("parameters and feature map live on different devices")
            logits = torch.empty((N, K), dtype=torch.float32, device=dev)
            sim = torch.empty((N, P), dtype=torch.float32, device=dev)
            occ = torch.empty((N, P, 1) + spatial, dtype=x.dtype, device=dev) if want_occ else None
            feats = torch.empty((N, P, D), dtype=torch.float32, device=dev) if want_feats else None
            dist = torch.empty((N, P), dtype=torch.float32, device=dev) if want_dist else None
            if N > 0:
                packed = self._packed_weights(lib, dims, w, tensors, dev, stream) if dims.path != _lib.PASN_PATH_GENERIC else None
                ws = self._workspace(lib, dims, dev)
                pa = None
                if push is not None:
                    pa = PasnPushArgs(push["labels"].data_ptr(), push["proto_class"].data_ptr(),
                                      int(push["global_offset"]), push["best_key"].data_ptr(), _ptr(push.get("best_vec")))
                st = lib.pasn_head_forward(x.data_ptr(), C.byref(w), _ptr(packed), C.byref(dims), logits.data_ptr(),
                                           sim.data_ptr(), _ptr(occ), _ptr(feats), _ptr(dist),
                                           C.byref(pa) if pa is not None else None, ws.data_ptr(), ws.numel(), stream)
                _lib.check(st, "pasn_head_forward")
                if _DEBUG_SYNC:
                    code = lib.pasn_debug_sm100_error(ws.data_ptr(), C.byref(dims), stream) if packed is not None else 0
                    torch.cuda.synchronize(dev)
                    if code != 0:
                        raise _lib.PasnError(f"fused tcgen05 kernel reported internal pipeline fault {code}")
        return {"logits": logits, "similarity": sim, "occurrence_map": occ, "features_extracted": feats, "distance": dist}

    def occurrence_only(self, x: torch.Tensor) -> torch.Tensor:
        """compute_occurence_map: served by the kernel family forward() uses for this shape (fused token kernel alone, the
        occurrence branch of the tiled chain, or the generic path)."""
        lib = _lib.load()
        m = self.owner
        dims, x, spatial = self.make_dims(x, m.kernel_path)
        dev = x.device
        with torch.cuda.device(dev):
            stream = torch.cuda.current_stream(dev).cuda_stream
            w, tensors = self._weights_struct(m)
            occ = torch.empty((dims.N, dims.P, 1) + spatial, dtype=x.dtype, device=dev)
            if dims.N > 0:
                packed = self._packed_weights(lib, dims, w, tensors, dev, stream) if dims.path != _lib.PASN_PATH_GENERIC else None
                ws = self._workspace(lib, dims, dev)
                _lib.check(lib.pasn_occurrence_only(x.data_ptr(), C.byref(w), _ptr(packed), C.byref(dims), occ.data_ptr(),
                                                    ws.data_ptr(), ws.numel(), stream), "pasn_occurrence_only")
        return occ


def _library_backward(ctx_rt, x, g_logits, g_sim, g_occ, want_gx):
    """pasn_head_backward on (x, head parameters): returns (grad_x or None, [11 parameter gradients]).  With g_logits and
    g_sim both None only the occurrence branch is differentiated (compute_occurence_map)."""
    rt = ctx_rt
    lib = _lib.load()
    m = rt.owner
    dims, xc, spatial = rt.make_dims(x, m.kernel_path)   # GENERIC keeps the CUDA-core backward, anything else lets the
    dev = xc.device                                       # library pick the tensor-core chain when the shape qualifies
    with torch.cuda.device(dev), torch.no_grad():
        stream = torch.cuda.current_stream(dev).cuda_stream
        w, tensors = rt._weights_struct(m)
        grads = [torch.zeros_like(t) for t in tensors]
        gw = PasnGrads(*[g.data_ptr() for g in grads])
        gx = torch.empty((dims.N, dims.C, dims.S), dtype=torch.float32, device=dev) if want_gx else None

        def prep(g, shape):
            if g is None:
                return None
            return g.to(torch.float32).reshape(shape).contiguous()

        gl = prep(g_logits, (dims.N, dims.K))
        gs = prep(g_sim, (dims.N, dims.P))
        go = prep(g_occ, (dims.N, dims.P, dims.S))
        if dims.N > 0:
            need = int(lib.pasn_head_backward_workspace_bytes(C.byref(dims)))
            ws = torch.empty(max(need, 256), dtype=torch.uint8, device=dev)
            st = lib.pasn_head_backward(xc.data_ptr(), C.byref(w), C.byref(dims), _ptr(gl), _ptr(gs), _ptr(go),
                                        C.byref(gw), _ptr(gx), ws.data_ptr(), ws.numel(), stream)
            _lib.check(st, "pasn_head_backward")
        elif gx is not None:
            gx.zero_()
    if gx is not None:
        gx = gx.reshape((dims.N, dims.C) + spatial).to(x.dtype)
    return gx, grads


class _OccFunction(torch.autograd.Function):
    """(features, occurrence_module parameters) -> occurrence_map with gradients: compute_occurence_map under grad, which
    the reference's TransformLoss calls once more per training step (src/loss/loss.py:302).  Forward = the library's
    occurrence-only path, backward = pasn_head_backward with no logits / similarity gradient (occurrence branch only)."""

    @staticmethod
    def forward(ctx, rt, x, *params):
        with torch.no_grad():
            occ = rt.occurrence_only(x)
        ctx.rt = rt
        ctx.save_for_backward(x, *params)
        return occ

    @staticmethod
    def backward(ctx, g_occ):
        x, *params = ctx.saved_tensors
        gx, grads = _library_backward(ctx.rt, x, None, None, g_occ, ctx.needs_input_grad[1])
        out = [None, gx]
        for i in range(5):   # occ_w1, occ_b1, occ_w2, occ_b2, occ_w3 = entries 4..8 of the weight struct
            out.append(grads[4 + i].reshape(params[i].shape) if ctx.needs_input_grad[2 + i] else None)
        return tuple(out)


class _HeadFunction(torch.autograd.Function):
    """(features, 11 head parameters) -> (logits, similarity, occurrence_map): forward through the library's usual path,
    backward through ``pasn_head_backward`` (fp32 CUDA-core kernels, forward intermediates recomputed)."""

    @staticmethod
    def forward(ctx, rt, x, *params):
        with torch.no_grad():
            r = rt.run(x, want_occ=True)
        ctx.rt = rt
        ctx.save_for_backward(x, *params)
        return r["logits"], r["similarity"], r["occurrence_map"]

    @staticmethod
    def backward(ctx, g_logits, g_sim, g_occ):
        x, *params = ctx.saved_tensors
        gx, grads = _library_backward(ctx.rt, x, g_logits, g_sim, g_occ, ctx.needs_input_grad[1])
        tensors = grads
        out = [None, gx]
        for i, t in enumerate(tensors):
            out.append(grads[i].reshape(params[i].shape) if ctx.needs_input_grad[2 + i] else None)
        return tuple(out)


class HostPipeline:
    """Head forward for batches that live in pinned host memory: the batch is cut into ``chunks`` pieces, each piece's
    host->device copy runs on a copy stream while the previous piece is in the kernels, and logits / similarities
    (optionally occurrence maps) go back into pinned host buffers.  Device staging and host result buffers are
    allocated once and reused, so a steady-state call does no allocation.  The step then costs about one H2D copy of
    the batch instead of copy + compute.

        pipe = HostPipeline(model, chunks=4)
        logits, sim = pipe(x_host_pinned)          # pinned host tensors, complete on return, valid until the next call

    Stream contract: the staging buffers are reused across calls, so the "kernels that read staging buffer i are done"
    events persist from call to call (the next call's first copies wait for the previous call's last kernels).  With
    ``sync=True`` (default) the call returns after the last device->host copy has completed; with ``sync=False`` it
    returns immediately and ``pipe.done`` (a CUDA event) marks the point after which the host buffers may be read.
    """

    def __init__(self, model, chunks: int = 4, device=None, want_occ: bool = False, sync: bool = True):
        self.model, self.chunks, self.want_occ, self.sync = model, max(1, int(chunks)), want_occ, sync
        self.device = torch.device(device) if device is not None else next(model.parameters()).device
        self.copy_stream = torch.cuda.Stream(device=self.device)
        self._stage = None
        self._host = None
        self._free = [None, None]    # event per staging buffer: kernels that read it are done (persists across calls)
        self.done = None

    @torch.no_grad()
    def __call__(self, x_host: torch.Tensor):
        m, dev = self.model, self.device
        n = int(x_host.shape[0])
        bounds = [(i * n) // self.chunks for i in range(self.chunks + 1)]
        pieces = [(bounds[i], bounds[i + 1]) for i in range(self.chunks) if bounds[i + 1] > bounds[i]]
        cmax = max((b - a for a, b in pieces), default=0)
        key = (tuple(x_host.shape[1:]), x_host.dtype, cmax, n)
        main = torch.cuda.current_stream(dev)
        if self._stage is None or self._stage[0] != key:
            if self.done is not None:
                self.done.synchronize()          # nothing may still be using the buffers we are about to replace
            bufs = [torch.empty((cmax,) + tuple(x_host.shape[1:]), dtype=x_host.dtype, device=dev) for _ in range(2)]
            self._stage = (key, bufs)
            self._free = [None, None]
            P, K = int(m.prototype_shape[0]), int(m.num_classes)
            host = {"logits": torch.empty((n, K), dtype=torch.float32).pin_memory(),
                    "similarity": torch.empty((n, P), dtype=torch.float32).pin_memory()}
            if self.want_occ:
                host["occurrence_map"] = torch.empty((n, P, 1) + tuple(x_host.shape[2:]), dtype=x_host.dtype).pin_memory()
            self._host = host
        bufs, host = self._stage[1], self._host
        free = self._free
        for i, (a, b) in enumerate(pieces):
            buf = bufs[i & 1][: b - a]
            with torch.cuda.stream(self.copy_stream):
                if free[i & 1] is not None:
                    self.copy_stream.wait_event(free[i & 1])
                buf.copy_(x_host[a:b], non_blocking=True)
                ready = torch.cuda.Event()
                ready.record(self.copy_stream)
            main.wait_event(ready)
            logits, sim, occ = m(buf)
            host["logits"][a:b].copy_(logits, non_blocking=True)
            host["similarity"][a:b].copy_(sim, non_blocking=True)
            if self.want_occ:
                host["occurrence_map"][a:b].copy_(occ, non_blocking=True)
            done = torch.cuda.Event()
            done.record(main)
            free[i & 1] = done
            self.done = done
        if self.sync and self.done is not None:
            self.done.synchronize()
        if self.want_occ:
            return host["logits"], host["similarity"], host["occurrence_map"]
        return host["logits"], host["similarity"]


def get_prototype_class_identity(num_prototypes: int, num_classes: int) -> torch.Tensor:
    """One-hot (P, K), prototype j -> class j // (P/K).  Reference: src/models/ProtoPNet.py:326-340."""
    assert num_prototypes % num_classes == 0
    ident = torch.zeros(num_prototypes, num_classes)
    per = num_prototypes // num_classes
    ident[torch.arange(num_prototypes), torch.arange(num_prototypes) // per] = 1
    return ident


def backbone_out_channels(backbone: nn.Module) -> int:
    """Same rule as PPNet.get_cnn_backbone_out_channels (src/models/ProtoPNet.py:152-162), extended so that any
    module exposing ``out_channels`` (e.g. an identity stub feeding precomputed features) also works."""
    if hasattr(backbone, "out_channels") and isinstance(getattr(backbone, "out_channels"), int):
        return backbone.out_channels
    name = str(backbone).upper()
    if "RESNET2P1D" in name or "R2PLUS1D" in name or "VIDEORESNET" in name:
        return [m for m in backbone.modules() if isinstance(m, nn.Conv3d)][-1].out_channels
    if name.startswith("VGG") or name.startswith("RES") or "RESNET" in name:
        return [m for m in backbone.modules() if isinstance(m, nn.Conv2d)][-1].out_channels
    if name.startswith("DENSE"):
        return [m for m in backbone.modules() if isinstance(m, nn.BatchNorm2d)][-1].num_features
    convs = [m for m in backbone.modules() if isinstance(m, (nn.Conv2d, nn.Conv3d))]
    if convs:
        return convs[-1].out_channels
    raise Exception("other base base_architecture NOT implemented")


class FeatureInput(nn.Module):
    """Identity 'backbone' for callers that already hold the backbone feature map (benchmarks, tests, push over
    precomputed features)."""

    def __init__(self, out_channels: int):
        super().__init__()
        self.out_channels = int(out_channels)

    def forward(self, x):
        return x


class PrototypeHeadMixin:
    """forward / push_forward / compute_occurence_map shared by the video and image models."""

    kernel_path: int = _lib.PASN_PATH_AUTO   # PASN_PATH_* selector (AUTO: tcgen05 when the shape qualifies)
    autograd_mode: str = "error"             # 'error' | 'kernel' | 'composite'

    def _init_head(self, cnn_backbone, img_size, prototype_shape, proto_layer_rf_info, num_classes, init_weights, conv):
        self.img_size = img_size
        self.prototype_shape = tuple(prototype_shape)
        self.num_prototypes = self.prototype_shape[0]
        self.num_classes = num_classes
        self.prototype_class_identity = get_prototype_class_identity(self.num_prototypes, self.num_classes)
        self.proto_layer_rf_info = proto_layer_rf_info
        self.epsilon = 1e-4
        self.cnn_backbone = cnn_backbone
        C_in = backbone_out_channels(cnn_backbone)
        D, P = self.prototype_shape[1], self.prototype_shape[0]
        self.add_on_layers = nn.Sequential(conv(C_in, D, kernel_size=1), nn.ReLU(), conv(D, D, kernel_size=1))
        self.occurrence_module = nn.Sequential(
            conv(C_in, D, kernel_size=1), nn.ReLU(), conv(D, D // 2, kernel_size=1), nn.ReLU(),
            conv(D // 2, P, kernel_size=1, bias=False))
        self.om_softmax = nn.Softmax(dim=-1)
        self.cosine_similarity = nn.CosineSimilarity(dim=2)
        self.prototype_vectors = nn.Parameter(torch.rand(self.prototype_shape), requires_grad=True)
        self.ones = nn.Parameter(torch.ones(self.prototype_shape), requires_grad=False)
        self.last_layer = nn.Linear(self.num_prototypes, self.num_classes, bias=False)
        if init_weights:
            self._initialize_weights(self.add_on_layers)
            self._initialize_weights(self.occurrence_module)
            self.set_last_layer_incorrect_connection(incorrect_strength=0)
        self._rt = _HeadRuntime(self)

    # ---- reference helpers (src/models/ProtoPNet.py:299-324) ----
    def set_last_layer_incorrect_connection(self, incorrect_strength):
        pos = torch.t(self.prototype_class_identity)
        self.last_layer.weight.data.copy_(1 * pos + incorrect_strength * (1 - pos))

    def _initialize_weights(self, layer):
        for m in layer.modules():
            if isinstance(m, (nn.Conv2d, nn.Conv3d)):
                nn.init.kaiming_normal_(m.weight, mode="fan_out", nonlinearity="relu")
                if m.bias is not None:
                    nn.init.constant_(m.bias, 0)

    def get_prototype_class_identity(self):
        return get_prototype_class_identity(self.num_prototypes, self.num_classes)

    # ---- dispatch ----
    def _needs_grad(self, x) -> bool:
        if not torch.is_grad_enabled():
            return False
        if x.requires_grad:
            return True
        return any(p.requires_grad for p in self.add_on_layers.parameters()) or \
            any(p.requires_grad for p in self.occurrence_module.parameters()) or \
            self.prototype_vectors.requires_grad or self.last_layer.weight.requires_grad

    def _composite(self, x):
        """Differentiable PyTorch composite of the head (opt-in, GPU, training only)."""
        fmap = self.add_on_layers(x)
        occ = torch.abs(self.occurrence_module(x))
        n = x.shape[0]
        feats = torch.einsum("nps,nds->npd", occ.reshape(n, occ.shape[1], -1), fmap.reshape(n, fmap.shape[1], -1))
        sim = self.cosine_similarity(feats, self.prototype_vectors.reshape(self.num_prototypes, -1).unsqueeze(0))
        sim = (sim + 1) / 2.0
        return feats, sim, occ.unsqueeze(2), self.last_layer(sim)

    def _grad_guard(self, x):
        if self._needs_grad(x):
            if self.autograd_mode in ("composite", "kernel"):
                return True
            raise NotImplementedError(
                "protoasnet_b200: this call needs gradients. Call under torch.no_grad() (eval / push / explain), or set "
                "model.autograd_mode = 'kernel' (backward through the library) or 'composite' (explicit PyTorch "
                "composite of the head) to train.")
        return False

    def _kernel_autograd(self, x):
        """(logits, similarity, occurrence_map) with gradients flowing through pasn_head_backward."""
        a, o = self.add_on_layers, self.occurrence_module
        params = (a[0].weight, a[0].bias, a[2].weight, a[2].bias, o[0].weight, o[0].bias, o[2].weight, o[2].bias,
                  o[4].weight, self.prototype_vectors, self.last_layer.weight)
        return _HeadFunction.apply(self._rt, x, *params)

    # ---- reference API ----
    def forward(self, x):
        """-> (logits [N,K], similarity [N,P], occurrence_map [N,P,1,(T),H,W]).  Video_XProtoNet.py:82-98."""
        x = self.cnn_backbone(x)
        if self._grad_guard(x):
            if self.autograd_mode == "kernel":
                return self._kernel_autograd(x)
            _, sim, occ, logits = self._composite(x)
            return logits, sim, occ
        r = self._rt.run(x, want_occ=True)
        return r["logits"], r["similarity"], r["occurrence_map"]

    def compute_occurence_map(self, x):
        """-> occurrence_map [N,P,1,(T),H,W].  Video_XProtoNet.py:100-109."""
        x = self.cnn_backbone(x)
        if self._grad_guard(x):
            if self.autograd_mode == "kernel":
                o = self.occurrence_module
                return _OccFunction.apply(self._rt, x, o[0].weight, o[0].bias, o[2].weight, o[2].bias, o[4].weight)
            return torch.abs(self.occurrence_module(x)).unsqueeze(2)
        return self._rt.occurrence_only(x)

    def get_occurence_map_absolute_val(self, x):
        if self._grad_guard(x):
            return torch.abs(self.occurrence_module(x)).unsqueeze(2)
        return self._rt.occurrence_only(x)

    def push_forward(self, x):
        """-> (features_extracted [N,P,D], 1 - similarity [N,P], occurrence_map, logits).  Video_XProtoNet.py:111-130."""
        x = self.cnn_backbone(x)
        if self._grad_guard(x):
            feats, sim, occ, logits = self._composite(x)
            return feats, 1 - sim, occ, logits
        r = self._rt.run(x, want_occ=True, want_feats=True, want_dist=True)
        return r["features_extracted"], r["distance"], r["occurrence_map"], r["logits"]

    # ---- B200 extension used by push (no per-batch D2H; the occurrence map is stored only on request) ----
    def push_scan(self, x, labels, proto_class, global_offset, best_key, backbone=True, best_vec=None, want_occ=False):
        """Fused similarity + class-restricted running argmin over one batch; updates ``best_key`` (and, when given,
        the winners' ``features_extracted`` rows ``best_vec`` [P,D] fp32) in place.  Returns the batch's ``logits``
        (and ``occurrence_map`` with ``want_occ``) from the same pass, for the winners' side data."""
        if backbone:
            x = self.cnn_backbone(x)
        if best_vec is not None and (best_vec.dtype != torch.float32 or not best_vec.is_contiguous()):
            raise _lib.PasnError("best_vec must be a contiguous fp32 [P,D] tensor")
        return self._rt.run(x, want_occ=want_occ, push=dict(labels=labels, proto_class=proto_class,
                                                              global_offset=global_offset, best_key=best_key,
                                                              best_vec=best_vec))

    def __repr__(self):
        rep = ("PPNet(\n\tcnn_backbone: {},\n\timg_size: {},\n\tprototype_shape: {},\n\tproto_layer_rf_info: {},\n"
               "\tnum_classes: {},\n)")
        return rep.format(self.cnn_backbone, self.img_size, self.prototype_shape, self.proto_layer_rf_info,
                          self.num_classes)


class Video_XProtoNet(PrototypeHeadMixin, nn.Module):
    def __init__(self, cnn_backbone, img_size, prototype_shape, proto_layer_rf_info, num_classes, init_weights=True,
                 **kwargs):
        nn.Module.__init__(self)
        assert len(prototype_shape) == 5, "video prototype_shape is (P, D, 1, 1, 1)"
        self._init_head(cnn_backbone, img_size, prototype_shape, proto_layer_rf_info, num_classes, init_weights, nn.Conv3d)


class XProtoNet(PrototypeHeadMixin, nn.Module):
    def __init__(self, features, img_size, prototype_shape, proto_layer_rf_info, num_classes, init_weights=True,
                 prototype_activation_function="log", add_on_layers_type="regular", **kwargs):
        nn.Module.__init__(self)
        assert len(prototype_shape) == 4, "image prototype_shape is (P, D, 1, 1)"
        if add_on_layers_type != "regular":
            raise NotImplementedError("only add_on_layers_type='regular' (the ProtoASNet image config) is supported")
        self.prototype_activation_function = prototype_activation_function
        self._init_head(features, img_size, prototype_shape, proto_layer_rf_info, num_classes, init_weights, nn.Conv2d)


# ---------------------------------------------------------------------------------------------
# constructors / registry (src/models/model_builder.py)
# ---------------------------------------------------------------------------------------------
def _video_backbone(base_architecture, pretrained, last_layer_num):
    if base_architecture == "features":
        raise ValueError("pass a module, not 'features'")
    if base_architecture != "resnet2p1d_18":
        raise Exception("other base base_architecture NOT implemented")
    if pretrained:
        raise RuntimeError("pretrained backbone weights need a download; pass pretrained=False and load a checkpoint")
    from torchvision.models.video import r2plus1d_18

    class Resnet2p1dFeatures(nn.Module):
        """torchvision r2plus1d_18 children[:last_layer_num] under ``.backbone`` -- the module layout (and hence the
        checkpoint keys ``cnn_backbone.backbone.<i>...``) of the reference's wrapper, src/models/resnet_features.py:307-327."""

        def __init__(self):
            super().__init__()
            self.backbone = nn.Sequential(*list(r2plus1d_18(weights=None).children())[:last_layer_num])

        def forward(self, x):
            return self.backbone(x)

    return Resnet2p1dFeatures()


def _image_backbone(base_architecture, pretrained):
    if base_architecture != "resnet18":
        raise Exception("other base base_architecture NOT implemented")
    if pretrained:
        raise RuntimeError("pretrained backbone weights need a download; pass pretrained=False and load a checkpoint")
    from torchvision.models import resnet18

    class Resnet18Features(nn.Module):
        """torchvision resnet18 without avgpool / fc -> [N,512,7,7], with the stem and the four stages as the named
        attributes conv1 / bn1 / layer1..layer4, i.e. the checkpoint keys of the reference's ResNet_features
        (src/models/resnet_features.py:126-214, :237-248)."""

        def __init__(self):
            super().__init__()
            r = resnet18(weights=None)
            self.conv1, self.bn1, self.relu, self.maxpool = r.conv1, r.bn1, r.relu, r.maxpool
            self.layer1, self.layer2, self.layer3, self.layer4 = r.layer1, r.layer2, r.layer3, r.layer4

        def forward(self, x):
            x = self.maxpool(self.relu(self.bn1(self.conv1(x))))
            return self.layer4(self.layer3(self.layer2(self.layer1(x))))

    return Resnet18Features()


def construct_Video_XProtoNet(base_architecture, pretrained=True, img_size=224, prototype_shape=(40, 256, 1, 1, 1),
                              num_classes=4, backbone_last_layer_num=-3):
    backbone = base_architecture if isinstance(base_architecture, nn.Module) else \
        _video_backbone(base_architecture, pretrained, backbone_last_layer_num)
    return Video_XProtoNet(cnn_backbone=backbone, img_size=img_size, prototype_shape=prototype_shape,
                           proto_layer_rf_info=None, num_classes=num_classes, init_weights=True)


def construct_XProtoNet(base_architecture, pretrained=True, img_size=224, prototype_shape=(40, 512, 1, 1),
                        num_classes=4, prototype_activation_function="log", add_on_layers_type="regular"):
    backbone = base_architecture if isinstance(base_architecture, nn.Module) else \
        _image_backbone(base_architecture, pretrained)
    return XProtoNet(features=backbone, img_size=img_size, prototype_shape=prototype_shape, proto_layer_rf_info=None,
                     num_classes=num_classes, init_weights=True,
                     prototype_activation_function=prototype_activation_function, add_on_layers_type=add_on_layers_type)


MODELS = {"XProtoNet": construct_XProtoNet, "Video_XProtoNet": construct_Video_XProtoNet}


def build(model_config: Dict):
    """Same contract as src/models/model_builder.py:14-25 (the ``prototype_shape`` string is parsed, not eval-ed)."""
    import ast

    config = deepcopy(model_config)
    config.pop("checkpoint_path", None)
    if isinstance(config.get("prototype_shape"), str):
        config["prototype_shape"] = tuple(ast.literal_eval(config["prototype_shape"]))
    name = config.pop("name")
    return MODELS[name](**config)
