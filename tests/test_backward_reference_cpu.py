"""The float64 backward reference and the input conditioning of tests/test_backward_parity_gpu.py, on the CPU: the
conditioning converges on every case of the GPU sweep, the reference agrees with central differences and with autograd
through oracle.head_oracle.push_forward_torch, and it takes the ABI's sub-gradients at exact zeros (relu'(0) = 0,
|x|'(0) = 0, a norm clamped at eps is a constant)."""
import numpy as np
import pytest
import torch

from oracle import head_oracle as ho
from protoasnet_b200 import synth
from tests import test_backward_parity_gpu as sweep
from tests.bwd_reference import (KEYS, TAU, TAU_FE, condition_inputs, feature_norm_margins, head_forward_f64,
                                 preactivation_margins, reference_grads, round_to)

SWEEP_CASES = sorted({c for c, _ in sweep.RUNS} | {sweep.CHUNKED_CASE}, key=sweep.case_id)


@pytest.mark.parametrize("case", SWEEP_CASES, ids=sweep.case_id)
def test_conditioning_meets_its_margin(case):
    path, Cc, D, P, K, spatial, N, kind = case
    dtn = sweep.KINDS[kind][0]
    dims = synth.HeadDims(Cc, D, P, K, spatial)
    sd = sweep.make_params(dims, kind.endswith("degenerate"))
    x0 = round_to(synth.make_features(dims, N, seed=100), dtn)
    x, margin, rounds = condition_inputs(x0, sd, dtn, TAU)
    assert margin >= TAU and rounds < 60
    assert float(preactivation_margins(x, sd).min()) == pytest.approx(margin, rel=1e-9)   # (whole-map einsum order)
    assert float(feature_norm_margins(x, sd).min()) >= TAU_FE
    assert np.array_equal(round_to(x, dtn), x)                      # redrawn voxels hold values of the map's dtype
    changed = np.any(x.reshape(N, Cc, -1) != x0.reshape(N, Cc, -1), axis=1)
    assert changed.mean() < 0.9                                     # only the ambiguous voxels were redrawn


def _tiny(seed=0, n=2):
    dims = synth.HeadDims(6, 4, 4, 2, (2, 3))
    sd = synth.make_head_params(dims, seed=seed + 3, bias_scale=0.1, last_layer_noise=0.3)
    x, margin, _ = condition_inputs(synth.make_features(dims, n, seed=seed), sd, "fp32", TAU)
    rng = np.random.default_rng(seed)
    up = (rng.standard_normal((n, dims.K)), rng.standard_normal((n, dims.P)), rng.standard_normal((n, dims.P, dims.S)))
    return dims, sd, x, [u.astype(np.float32) for u in up]


def test_reference_matches_central_differences():
    dims, sd, x, (wl, ws, wo) = _tiny()
    xt = torch.from_numpy(x).double().requires_grad_(True)
    ps = [torch.from_numpy(np.ascontiguousarray(sd[k])).double().requires_grad_(True) for k in KEYS]
    up = [torch.from_numpy(u).double() for u in (wl, ws, wo)]

    def loss(xv, *pv):
        logits, sim, occ = head_forward_f64(xv, dict(zip(KEYS, pv)))
        return (logits * up[0]).sum() + (sim * up[1]).sum() + (occ * up[2]).sum()

    assert torch.autograd.gradcheck(loss, (xt, *ps), eps=1e-6, atol=1e-7, rtol=1e-5)
    gx, g = reference_grads(x, sd, wl, ws, wo)
    want = torch.autograd.grad(loss(xt, *ps), [xt] + ps)
    assert np.allclose(gx, want[0].reshape(gx.shape).numpy(), rtol=1e-12, atol=1e-14)
    for k, w in zip(KEYS, want[1:]):
        assert np.allclose(g[k], w.numpy(), rtol=1e-12, atol=1e-14), k


def test_reference_matches_push_forward_torch():
    """The einsum pooling of the reference is oracle.head_oracle's broadcast-and-sum pooling: same outputs, same
    gradients in float64."""
    dims = synth.HeadDims(24, 16, 8, 4, (2, 3, 3))
    sd = synth.make_head_params(dims, seed=5, bias_scale=0.1, last_layer_noise=0.2)
    n = 3
    x, _, _ = condition_inputs(synth.make_features(dims, n, seed=2), sd, "fp32", TAU)
    rng = np.random.default_rng(1)
    wl = rng.standard_normal((n, dims.K)).astype(np.float32)
    ws = rng.standard_normal((n, dims.P)).astype(np.float32)
    wo = rng.standard_normal((n, dims.P, dims.S)).astype(np.float32)
    gx, g = reference_grads(x, sd, wl, ws, wo)
    sdt = {k: torch.from_numpy(np.ascontiguousarray(v)).double().requires_grad_(True) for k, v in sd.items()}
    xt = torch.from_numpy(x).double().requires_grad_(True)
    feats, dist, occ, logits = ho.push_forward_torch(xt, sdt)
    ((logits * torch.from_numpy(wl).double()).sum() + ((1 - dist) * torch.from_numpy(ws).double()).sum() +
     (occ.reshape(n, dims.P, -1) * torch.from_numpy(wo).double()).sum()).backward()
    assert np.allclose(gx, xt.grad.reshape(gx.shape).numpy(), rtol=1e-10, atol=1e-13)
    for k in KEYS:
        assert np.allclose(g[k], sdt[k].grad.numpy(), rtol=1e-10, atol=1e-13), k


def test_reference_subgradients_at_exact_zeros():
    """Zero prototype row (its norm clamped), zero W5 row (O and features_extracted of that prototype identically zero),
    zero W1 row and b1 entry (H1 identically zero in that channel): the reference's gradients there, by hand."""
    case = next(c for c in sweep.CASES if c[7] == "fp32_degenerate")
    path, Cc, D, P, K, spatial, N, kind = case
    dims = synth.HeadDims(Cc, D, P, K, spatial)
    sd = sweep.make_params(dims, True)
    x, margin, _ = condition_inputs(round_to(synth.make_features(dims, N, seed=100), "fp32"), sd, "fp32", TAU)
    assert margin >= TAU   # the three zero pre-activation rows (no terms at all) do not count against the margin
    rng = np.random.default_rng(7)
    wl = rng.standard_normal((N, K)).astype(np.float32)
    ws = rng.standard_normal((N, P)).astype(np.float32)
    wo = rng.standard_normal((N, P, dims.S)).astype(np.float32)
    gx, g = reference_grads(x, sd, wl, ws, wo)
    f64 = ho.head_forward_f64(x, sd)
    fe = f64["features_extracted"]
    ll = sd["last_layer.weight"].astype(np.float64)
    gcos = 0.5 * (ws + wl @ ll)                                             # d(loss)/d(cos) [N, P]
    eps = 1e-8
    # prototype 0 is zero: cos = <f, v> / (|f| eps) with eps constant -> d/dv = f / (|f| eps); similarity 1/2
    assert np.all(f64["similarity"][:, 0] == 0.5)
    nf = np.maximum(np.linalg.norm(fe[:, 0], axis=1), eps)
    want = (gcos[:, 0, None] * fe[:, 0] / (nf[:, None] * eps)).sum(0)
    assert np.allclose(g["prototype_vectors"].reshape(P, D)[0], want, rtol=1e-10)
    # W5 row 1 is zero: O[:, 1] = 0 and d|x|/dx(0) = 0 -> no gradient into W5 row 1; features_extracted[:, 1] = 0, its norm
    # clamped -> d(cos)/dv = f / (eps |v|) = 0: no gradient into prototype 1
    assert np.all(f64["occurrence_map"][:, 1] == 0) and np.all(fe[:, 1] == 0)
    assert np.all(g["occurrence_module.4.weight"].reshape(P, -1)[1] == 0)
    assert np.all(g["prototype_vectors"].reshape(P, D)[1] == 0)
    # (W1 row 2, b1[2]) are zero: H1[2] = 0 everywhere and relu'(0) = 0 -> no gradient into either, nor into W2 column 2
    assert np.all(g["add_on_layers.0.weight"].reshape(D, Cc)[2] == 0) and g["add_on_layers.0.bias"][2] == 0
    assert np.all(g["add_on_layers.2.weight"].reshape(D, D)[:, 2] == 0)
    # every other row does get gradient
    assert np.all(np.abs(g["add_on_layers.0.weight"].reshape(D, Cc)[3]) > 0)
    assert np.isfinite(gx).all()
