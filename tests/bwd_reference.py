"""float64 reference of the head's backward (pasn_head_backward) and the input conditioning its parity tests rely on.

Reference: the gradients of

    loss = sum(logits * wl) + sum(similarity * ws) + sum(occurrence_map * wo)

with respect to the feature map and the eleven head parameters, by float64 autograd through the reference's op sequence
(oracle/head_oracle.py: add-on, occurrence module, pooling, cosine similarity, last layer).  A ``None`` upstream weight
contributes nothing.  The pooling is the same contraction as pooled_features_torch, written as one einsum so that the
large cases do not materialise the [N, P, D, S] product (float64: the summation order does not matter).

Conditioning: the backward decides four signs on pre-activations it recomputes itself -- the ReLU masks of H1, G1, G2
and sign(Opre) under |.| -- and those recomputed values carry fp32-grade error (about 1e-6 of the magnitude sum of their
dot product).  A pre-activation that lies within that error of zero can take the other sub-gradient in the kernel than
in the reference; one such flip moves a feature-map gradient column by percent.  condition_inputs() redraws the
feature vector of every voxel that has such a value, so that fp32-grade agreement can be demanded on any seed.

It also redraws the clips whose pooled feature vector FE[n, p] = sum_s O[p, s] F[:, s] is small against the magnitudes
it is summed from.  The cosine's gradient scales with 1 / |FE|, so such a row dominates every gradient downstream and
carries the relative error of its occurrence values: with one voxel per clip FE = O F, and an O at the 1e-4 margin above
has a relative error of 1e-6 / 1e-4 on the tensor cores.  Such rows moved the feature-map gradient by 7e-4 of its scale
(1.5e-4 with the bound at 1e-3); at 1e-2 they sit with the other rows.
"""
from __future__ import annotations

from typing import Dict, Optional, Tuple

import numpy as np
import torch
import torch.nn.functional as F

from oracle import head_oracle as ho
from protoasnet_b200 import synth

# the eleven tensors of pasn_weights / pasn_grads, in that order
KEYS = ["add_on_layers.0.weight", "add_on_layers.0.bias", "add_on_layers.2.weight", "add_on_layers.2.bias",
        "occurrence_module.0.weight", "occurrence_module.0.bias", "occurrence_module.2.weight",
        "occurrence_module.2.bias", "occurrence_module.4.weight", "prototype_vectors", "last_layer.weight"]
OCC_KEYS = KEYS[4:9]

TAU = 1e-4      # a pre-activation is ambiguous when |value| < TAU * (sum of the magnitudes of its terms)
TAU_FE = 1e-2   # a pooled feature vector is ill-conditioned when its norm < TAU_FE * (its error scale, see below)


def round_to(x: np.ndarray, dtype: str) -> np.ndarray:
    """x (float32) rounded to the values a feature map of ``dtype`` ("fp32", "bf16", "fp16") holds."""
    x = np.ascontiguousarray(x, dtype=np.float32)
    if dtype == "bf16":
        return synth.round_to_bf16(x)
    if dtype == "fp16":
        return x.astype(np.float16).astype(np.float32)
    assert dtype == "fp32", dtype
    return x


def head_forward_f64(xt: torch.Tensor, sdt: Dict[str, torch.Tensor]):
    """(logits, similarity, occurrence_map [N, P, S]) of feature map xt [N, C, *spatial]: oracle/head_oracle.py's op
    sequence (1x1 convolutions as matmuls over the flattened voxels, pooling as one einsum)."""
    n, c = xt.shape[:2]
    x = xt.reshape(n, c, -1)

    def w(k):
        t = sdt[k]
        return t.reshape(t.shape[0], t.shape[1])

    def conv(inp, k, b=None):
        y = torch.einsum("oc,ncs->nos", w(k), inp)
        return y if b is None else y + sdt[b][None, :, None]

    fmap = conv(F.relu(conv(x, "add_on_layers.0.weight", "add_on_layers.0.bias")), "add_on_layers.2.weight",
                "add_on_layers.2.bias")
    g = F.relu(conv(x, "occurrence_module.0.weight", "occurrence_module.0.bias"))
    g = F.relu(conv(g, "occurrence_module.2.weight", "occurrence_module.2.bias"))
    occ = torch.abs(conv(g, "occurrence_module.4.weight"))
    feats = torch.einsum("nps,nds->npd", occ, fmap)
    sim = ho.similarity_torch(feats, sdt["prototype_vectors"])
    logits = F.linear(sim, sdt["last_layer.weight"])
    return logits, sim, occ


def reference_grads(x: np.ndarray, sd: Dict[str, np.ndarray], wl: Optional[np.ndarray], ws: Optional[np.ndarray],
                    wo: Optional[np.ndarray]) -> Tuple[np.ndarray, Dict[str, np.ndarray]]:
    """float64 d(loss)/d(x) as [N, C, S] and d(loss)/d(parameter) for the eleven KEYS (parameter shapes).
    wl [N, K], ws [N, P], wo [N, P, S] (fp32 upstream gradients) or None."""
    sdt = {k: torch.from_numpy(np.ascontiguousarray(sd[k])).double().requires_grad_(True) for k in KEYS}
    xt = torch.from_numpy(np.ascontiguousarray(x)).double().requires_grad_(True)
    logits, sim, occ = head_forward_f64(xt, sdt)
    loss = xt.new_zeros(())
    for out, up in ((logits, wl), (sim, ws), (occ, wo)):
        if up is not None:
            loss = loss + (out * torch.from_numpy(np.asarray(up, np.float32)).double().reshape(out.shape)).sum()
    if not loss.requires_grad:   # no upstream gradient at all
        return np.zeros((x.shape[0], x.shape[1], int(np.prod(x.shape[2:]))), np.float64), \
            {k: np.zeros(sd[k].shape, np.float64) for k in KEYS}
    gx, *gp = torch.autograd.grad(loss, [xt] + [sdt[k] for k in KEYS], allow_unused=True)
    gx = gx.reshape(x.shape[0], x.shape[1], -1).numpy()
    return gx, {k: (np.zeros(sd[k].shape) if g is None else g.numpy()) for k, g in zip(KEYS, gp)}


def _mat(sd, k):
    a = np.asarray(sd[k], np.float64)
    return a.reshape(a.shape[0], -1)


def preactivation_margins(x: np.ndarray, sd: Dict[str, np.ndarray]) -> np.ndarray:
    """[N, S]: per voxel, the smallest |value| / (sum of |terms|) over the pre-activations whose sign the backward decides
    (W1 x + b1, W3 x + b3, W4 G1 + b4, W5 G2), float64.  A value whose terms are all zero (a zeroed weight row and bias:
    an exact zero on both sides) does not count; a voxel without any counted value gets +inf."""
    n, c = x.shape[:2]
    xs = np.asarray(x, np.float64).reshape(n, c, -1)
    ax = np.abs(xs)
    best = np.full((n, xs.shape[2]), np.inf)

    def take(pre, mag):
        with np.errstate(divide="ignore", invalid="ignore"):
            r = np.where(mag > 0, np.abs(pre) / np.where(mag > 0, mag, 1.0), np.inf)
        np.minimum(best, r.min(axis=1), out=best)

    def layer(inp, ainp, wk, bk=None):
        w = _mat(sd, wk)
        pre = np.einsum("oc,ncs->nos", w, inp)
        mag = np.einsum("oc,ncs->nos", np.abs(w), ainp)
        if bk is not None:
            b = np.asarray(sd[bk], np.float64)[None, :, None]
            pre = pre + b
            mag = mag + np.abs(b)
        take(pre, mag)
        return pre

    layer(xs, ax, "add_on_layers.0.weight", "add_on_layers.0.bias")
    g1 = np.maximum(layer(xs, ax, "occurrence_module.0.weight", "occurrence_module.0.bias"), 0)
    g2 = np.maximum(layer(g1, g1, "occurrence_module.2.weight", "occurrence_module.2.bias"), 0)
    layer(g2, g2, "occurrence_module.4.weight")
    return best


def feature_norm_margins(x: np.ndarray, sd: Dict[str, np.ndarray]) -> np.ndarray:
    """[N, P]: |FE[n, p]| / |sqrt(sum_s (M[p, s] F[:, s])^2)|, float64, where M[p, s] = sum_j |W5[p, j]| G2[j, s] is the
    magnitude sum of the occurrence value O[p, s]: the denominator is the size of the error of FE when every O[p, s] is off
    by the same fraction of M[p, s] in independent directions (one voxel per clip: M / O).  +inf where it is zero (a
    zeroed W5 row: FE = 0 exactly on both sides)."""
    n, c = x.shape[:2]
    xs = np.asarray(x, np.float64).reshape(n, c, -1)

    def conv(inp, wk, bk=None):
        y = np.einsum("oc,ncs->nos", _mat(sd, wk), inp)
        return y if bk is None else y + np.asarray(sd[bk], np.float64)[None, :, None]

    f = conv(np.maximum(conv(xs, "add_on_layers.0.weight", "add_on_layers.0.bias"), 0), "add_on_layers.2.weight",
             "add_on_layers.2.bias")
    g2 = np.maximum(conv(np.maximum(conv(xs, "occurrence_module.0.weight", "occurrence_module.0.bias"), 0),
                         "occurrence_module.2.weight", "occurrence_module.2.bias"), 0)
    o = np.abs(conv(g2, "occurrence_module.4.weight"))
    mag = np.einsum("pj,njs->nps", np.abs(_mat(sd, "occurrence_module.4.weight")), g2)
    fe = np.linalg.norm(np.einsum("nps,nds->npd", o, f), axis=2)
    den = np.sqrt(np.einsum("nps,nds->np", mag ** 2, f ** 2))
    with np.errstate(divide="ignore", invalid="ignore"):
        return np.where(den > 0, fe / np.where(den > 0, den, 1.0), np.inf)


def condition_inputs(x: np.ndarray, sd: Dict[str, np.ndarray], dtype: str, tau: float = TAU, seed: int = 0,
                     max_rounds: int = 200, tau_fe: float = TAU_FE) -> Tuple[np.ndarray, float, int]:
    """Redraw (relu(N(0, 1)), rounded to ``dtype``) the feature vector x[n, :, s] of every voxel with a pre-activation
    below ``tau`` of its magnitude sum, and every voxel of a clip with a feature_norm_margins() entry below ``tau_fe``,
    until none is left.  Returns (conditioned x, achieved minimum pre-activation margin, rounds of redrawing).
    x: [N, C, *spatial], already holding ``dtype`` values; it is not modified."""
    shape = x.shape
    n, c = shape[:2]
    xs = np.array(x, np.float32).reshape(n, c, -1)
    rng = np.random.default_rng(10_000 + seed)
    margins = np.empty((n, xs.shape[2]))
    vn, vs = np.nonzero(np.ones(margins.shape, bool))   # round 0: every voxel
    rounds = 0
    while True:
        # margins of this round's voxels only (every layer acts per voxel): the voxels as a batch of one-voxel clips
        margins[vn, vs] = preactivation_margins(xs[vn, :, vs][:, :, None], sd)[:, 0]
        bad = margins < tau
        if not bad.any():
            bad[feature_norm_margins(xs, sd).min(axis=1) < tau_fe] = True   # whole clips
            if not bad.any():
                return xs.reshape(shape), float(margins.min()), rounds
        rounds += 1
        if rounds > max_rounds:
            raise RuntimeError(f"conditioning did not converge: {int(bad.sum())} voxels below tau = {tau}")
        vn, vs = np.nonzero(bad)
        xs[vn, :, vs] = round_to(np.maximum(rng.standard_normal((len(vn), c), dtype=np.float32), 0), dtype)
