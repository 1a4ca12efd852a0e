"""Rounding model of the tensor-core forward in bf16 / fp16 mode (TEST INFRASTRUCTURE -- see oracle/__init__.py).

The fused pair (head_sm100*.cu) and the tiled chain (tiled.cu) round at fixed points and accumulate everything else in
fp32.  This module rounds at the same points and accumulates in float64 (torch CPU matmuls), so that its only
disagreement with a kernel is fp32 against float64 accumulation order, plus the rare bf16 rounding flips that order
causes.  Rounding points (round-to-nearest-even throughout):

    quantity              bf16 mode / fp32_fused            fp16 mode                   where
    X                     as given / bf16 on the fly        as given (fp16, exact)      K1 loader; tiled to_tokens_*
    W1, W3                bf16                              fp16                        pack_weights_kernel, tiled_pack_weights
    W4, W5, W2            bf16                              bf16                        same
    b1, b3, b4, b2        bf16, added in fp32               same                        round_bf16 / pack_bias_kernel
    H1, G1, G2            bf16 after bias + ReLU            same                        K1 epilogue E1-E3; tiled (A), (B) OUT_BF16
    O                     bf16 of |W5 G2|                   same (pooling operand)      K1 E4; tiled (C)
    pooled (pool first)   fp32 sum, kept as bf16 hi + lo    same                        K1 E5 -> K2 images; tiled (D) OUT_BF16_HILO
    sum_s O (b2 term)     sum of the bf16 O values          same                        K1 warp 3; psum_rounded / clip_colsum_kernel
    F (W2 first)          bf16 of H1 W2^T + b2              same                        tiled (D') OUT_BF16
    cosine chain          unrounded (fp32 in the kernels)   same                        K2 epilogue; proto_stage.cu

The occurrence map a caller gets back is O in the feature map's dtype, except for fp16 maps of the tiled chain: its
occurrence GEMM stores fp16(|W5 G2|) directly and the pooling reads a bf16 copy.  The fused pair's fp16 map is fp16(O).
Both are returned (``occurrence_map`` = O, ``occurrence_abs`` = |W5 G2| before rounding).
"""
from __future__ import annotations

from typing import Dict, Optional

import numpy as np
import torch

MODES = ("bf16", "fp16", "fp32_fused")
ORDERS = ("pool_first", "w2_first")
_COS_EPS = 1e-8


def head_forward_emulated(x: np.ndarray, sd: Dict[str, np.ndarray], mode: str, order: str, occ: Optional[np.ndarray] = None,
                          dtype: torch.dtype = torch.float64, rounding: bool = True) -> Dict[str, np.ndarray]:
    """Forward of the head as the tensor-core kernels compute it.

    x      feature map [N, C, *spatial] holding the values the kernel reads (bf16 / fp16 values, or fp32 for fp32_fused)
    mode   'bf16', 'fp16' or 'fp32_fused' (PASN_PATH_TCGEN05 on an fp32 map: X rounded to bf16 on the fly)
    order  'pool_first' (fused pair; tiled chain with S >= 2P) or 'w2_first' (tiled chain with S < 2P)
    occ    optional occurrence map [N, P, ...] to run the stages after the map on instead of the emulated one (the kernel's
           own map: in bf16 mode it holds exactly the values the pooling read)
    dtype  accumulation type: float64 is the reference; float32 stands in for the kernel's arithmetic
    rounding  False switches every rounding point off (then this is head_forward_f64 in another summation order)

    Returns numpy arrays: logits [N,K], similarity / distance [N,P], occurrence_map (O) and occurrence_abs [N,P,S],
    features_extracted [N,P,D], and the stage intermediates h1, g1, g2 [N,*,S], osum [N,P], pooled [N,P,D] (pool first)
    or f [N,D,S] (W2 first)."""
    if mode not in MODES:
        raise ValueError(f"mode must be one of {MODES}")
    if order not in ORDERS:
        raise ValueError(f"order must be one of {ORDERS}")
    n, c = x.shape[:2]

    def rnd(t, to):
        return t.to(to).to(dtype) if rounding else t

    def bf(t):
        return rnd(t, torch.bfloat16)

    def param(name, to):
        a = torch.from_numpy(np.ascontiguousarray(sd[name], dtype=np.float32))
        a = a.reshape(a.shape[0], -1) if a.dim() > 1 else a
        return a.to(to).to(dtype) if rounding and to is not None else a.to(dtype)

    l1 = torch.float16 if mode == "fp16" else torch.bfloat16
    w1, w3 = param("add_on_layers.0.weight", l1), param("occurrence_module.0.weight", l1)
    w4, w5 = param("occurrence_module.2.weight", torch.bfloat16), param("occurrence_module.4.weight", torch.bfloat16)
    w2 = param("add_on_layers.2.weight", torch.bfloat16)
    b1, b3 = param("add_on_layers.0.bias", torch.bfloat16), param("occurrence_module.0.bias", torch.bfloat16)
    b4, b2 = param("occurrence_module.2.bias", torch.bfloat16), param("add_on_layers.2.bias", torch.bfloat16)
    protos = param("prototype_vectors", None)
    last = param("last_layer.weight", None)

    xs = torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32)).reshape(n, c, -1).to(dtype)
    if mode == "fp32_fused":
        xs = bf(xs)
    h1 = bf(torch.relu(w1 @ xs + b1[:, None]))
    g1 = bf(torch.relu(w3 @ xs + b3[:, None]))
    g2 = bf(torch.relu(w4 @ g1 + b4[:, None]))
    oabs = (w5 @ g2).abs()
    o = bf(oabs)
    if occ is not None:
        o = torch.from_numpy(np.asarray(occ, dtype=np.float64)).reshape(o.shape).to(dtype)
    osum = o.sum(dim=2)
    out = {}
    if order == "pool_first":
        pooled = o @ h1.transpose(1, 2)
        if rounding:
            hi = bf(pooled)
            pooled = hi + bf(pooled - hi)
        fe = pooled @ w2.t() + osum[:, :, None] * b2
        out["pooled"] = pooled
    else:
        f = bf(w2 @ h1 + b2[:, None])
        fe = o @ f.transpose(1, 2)
        out["f"] = f
    fn = torch.linalg.vector_norm(fe, dim=2, keepdim=True).clamp_min(_COS_EPS)
    vn = torch.linalg.vector_norm(protos, dim=1, keepdim=True).clamp_min(_COS_EPS)
    cos = torch.einsum("npd,pd->np", fe / fn, protos / vn)
    sim = (cos + 1.0) / 2.0
    out.update(logits=sim @ last.t(), similarity=sim, distance=1.0 - sim, occurrence_map=o, occurrence_abs=oabs,
               features_extracted=fe, h1=h1, g1=g1, g2=g2, osum=osum)
    return {k: v.numpy() for k, v in out.items()}


def cosine_chain_f64(feats: np.ndarray, sd: Dict[str, np.ndarray]) -> Dict[str, np.ndarray]:
    """similarity / distance / logits in float64 from given features_extracted [N,P,D] (the kernel's own, to isolate the
    prototype stage)."""
    f = np.asarray(feats, dtype=np.float64)
    pv = sd["prototype_vectors"].astype(np.float64).reshape(sd["prototype_vectors"].shape[0], -1)
    fn = np.maximum(np.linalg.norm(f, axis=2, keepdims=True), _COS_EPS)
    vn = np.maximum(np.linalg.norm(pv, axis=1, keepdims=True), _COS_EPS)
    sim = (np.einsum("npd,pd->np", f / fn, pv / vn) + 1.0) / 2.0
    return {"similarity": sim, "distance": 1.0 - sim, "logits": sim @ sd["last_layer.weight"].astype(np.float64).T}
