"""Backward of the prototype head through the library (autograd_mode='kernel', pasn_head_backward) against PyTorch
autograd on the CPU oracle: gradients with respect to the feature map and all eleven parameter tensors."""
import numpy as np
import pytest
import torch

from oracle import head_oracle as ho
from protoasnet_b200 import synth
from tests.util import assert_close, build_model

pytestmark = pytest.mark.gpu

KEYS = ["add_on_layers.0.weight", "add_on_layers.0.bias", "add_on_layers.2.weight", "add_on_layers.2.bias",
        "occurrence_module.0.weight", "occurrence_module.0.bias", "occurrence_module.2.weight",
        "occurrence_module.2.bias", "occurrence_module.4.weight", "prototype_vectors", "last_layer.weight"]


def _oracle_grads(x, sd, wl, ws, wo, dtype=torch.float64):
    """d/d(x, params) of  sum(logits*wl) + sum(sim*ws) + sum(occ*wo)  on the CPU oracle (float64 for a clean reference)."""
    sdt = {k: torch.from_numpy(np.ascontiguousarray(v)).to(dtype).requires_grad_(k != "ones") for k, v in sd.items()}
    xt = torch.from_numpy(x).to(dtype).requires_grad_(True)
    feats, dist, occ, logits = ho.push_forward_torch(xt, sdt)
    sim = 1 - dist
    loss = (logits * torch.from_numpy(wl).to(dtype)).sum() + (sim * torch.from_numpy(ws).to(dtype)).sum() + \
        (occ * torch.from_numpy(wo).to(dtype)).sum()
    loss.backward()
    return float(loss.detach()), xt.grad.numpy(), {k: sdt[k].grad.numpy() for k in KEYS}


@pytest.mark.parametrize("cfg,n,fmt", [("tiny_video", 7, "ncs"), ("tiny_image", 5, "ncs"), ("odd_video", 3, "ncs"),
                                       ("tiny_video", 4, "nsc"), ("tiny_video", 5, "ncs-bf16")])
def test_kernel_backward_matches_autograd(cfg, n, fmt):
    """fmt: the feature map's layout, "-bf16" for a bf16 map (bf16-representable features and parameters; as in the cfg-3
    bf16 case, d(loss)/d(occurrence map) and the feature-map gradient come back in bf16, hence that case's tolerances)."""
    layout, bf = fmt.split("-")[0], fmt.endswith("-bf16")
    dims = synth.CONFIGS[cfg]
    sd = synth.make_head_params(dims, seed=17, bias_scale=0.1, last_layer_noise=0.2, bf16_round=bf)
    x = synth.make_features(dims, n, seed=6, bf16_round=bf)
    rng = np.random.default_rng(3)
    wl = rng.standard_normal((n, dims.K)).astype(np.float32)
    ws = rng.standard_normal((n, dims.P)).astype(np.float32)
    wo = rng.standard_normal((n, dims.P, 1) + dims.spatial).astype(np.float32) * 0.1
    ref_loss, ref_gx, ref_g = _oracle_grads(x, sd, wl, ws, wo)

    m = build_model(dims, sd)
    m.train()
    m.autograd_mode = "kernel"
    xt = torch.from_numpy(x).cuda()
    if layout == "nsc":
        xt = xt.contiguous(memory_format=torch.channels_last_3d if dims.ndim == 3 else torch.channels_last)
    if bf:
        xt = xt.bfloat16()
    xt.requires_grad_(True)
    logits, sim, occ = m(xt)
    loss = (logits * torch.from_numpy(wl).cuda()).sum() + (sim * torch.from_numpy(ws).cuda()).sum() + \
        (occ.float() * torch.from_numpy(wo).cuda()).sum()
    loss.backward()
    rtol, afrac = (1e-2, 4e-3) if bf else (2e-4, 2e-5)
    assert abs(float(loss.detach()) - ref_loss) <= (1e-2 if bf else 1e-4) * max(1.0, abs(ref_loss))
    assert xt.grad.dtype == xt.dtype
    assert_close(xt.grad, ref_gx, rtol, "grad feature map", atol_frac=afrac)
    own = dict(m.named_parameters())
    for k in KEYS:
        assert own[k].grad is not None, k
        assert_close(own[k].grad.reshape(ref_g[k].shape), ref_g[k], rtol, f"grad {k}", atol_frac=afrac)
    assert own["ones"].grad is None


def test_kernel_backward_partial_grads_and_accumulation():
    """Only similarity feeds the loss, the feature map needs no gradient, and two backward passes accumulate."""
    dims = synth.CONFIGS["tiny_video"]
    sd = synth.make_head_params(dims, seed=2, bias_scale=0.1, last_layer_noise=0.2)
    n = 6
    x = synth.make_features(dims, n, seed=1)
    ws = np.random.default_rng(0).standard_normal((n, dims.P)).astype(np.float32)
    _, _, ref_g = _oracle_grads(x, sd, np.zeros((n, dims.K), np.float32), ws, np.zeros((n, dims.P, 1) + dims.spatial, np.float32))
    m = build_model(dims, sd)
    m.autograd_mode = "kernel"
    xt = torch.from_numpy(x).cuda()
    for _ in range(2):
        logits, sim, occ = m(xt)
        (sim * torch.from_numpy(ws).cuda()).sum().backward()
    own = dict(m.named_parameters())
    for k in KEYS:
        if k == "last_layer.weight":
            assert own[k].grad is None or float(own[k].grad.abs().max()) == 0.0
            continue
        assert_close(own[k].grad.reshape(ref_g[k].shape), 2 * ref_g[k], 2e-4, f"accumulated grad {k}", atol_frac=2e-5)


def test_default_mode_still_refuses():
    dims = synth.CONFIGS["tiny_video"]
    m = build_model(dims, synth.make_head_params(dims, seed=2))
    x = torch.from_numpy(synth.make_features(dims, 2, seed=1)).cuda()
    with pytest.raises(NotImplementedError):
        m(x)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_kernel_backward_cfg3_shape(dtype):
    """cfg-3 shape (C=512, D=256, P=40, S=196; every GEMM spans many tiles) against float64 autograd on the CPU oracle.
    bf16 features: the forward runs the fused tcgen05 kernels, the backward is the fp32 gradient on the same
    (bf16-representable) inputs; the feature-map gradient comes back in bf16.  (The PyTorch composite on the GPU is not
    a usable reference here: its TF32 convolutions flip signs of near-zero pre-activations under |.|.)"""
    dims = synth.CONFIGS["cfg3_video_b1024"]
    sd = synth.make_head_params(dims, seed=200, bias_scale=0.02, bf16_round=True)
    n = 5
    x = synth.make_features(dims, n, seed=12, bf16_round=True)
    rng = np.random.default_rng(8)
    wl = rng.standard_normal((n, dims.K)).astype(np.float32)
    ws = rng.standard_normal((n, dims.P)).astype(np.float32)
    wo = rng.standard_normal((n, dims.P, 1) + dims.spatial).astype(np.float32) * 0.05
    _, ref_gx, ref_g = _oracle_grads(x, sd, wl, ws, wo)
    m = build_model(dims, sd)
    m.autograd_mode = "kernel"
    xt = torch.from_numpy(x).cuda().to(dtype).requires_grad_(True)
    logits, sim, occ = m(xt)
    ((logits * torch.from_numpy(wl).cuda()).sum() + (sim * torch.from_numpy(ws).cuda()).sum() +
     (occ.float() * torch.from_numpy(wo).cuda()).sum()).backward()
    own = dict(m.named_parameters())
    # bf16: autograd hands d(loss)/d(occurrence_map) over in the map's dtype, i.e. rounded to bf16 (2^-9 relative), and
    # the feature-map gradient is returned in bf16 -- everything downstream of those carries that rounding
    rtol, afrac = (2e-4, 2e-5) if dtype == torch.float32 else (1e-2, 4e-3)
    for k in KEYS:
        assert_close(own[k].grad.reshape(ref_g[k].shape), ref_g[k], rtol, f"grad {k}", atol_frac=afrac)
    assert xt.grad.dtype == dtype
    assert_close(xt.grad, ref_gx, rtol, "grad feature map", atol_frac=afrac)


@pytest.mark.parametrize("cfg,n,dtype", [("tiny_video", 5, torch.float32), ("cfg3_video_b1024", 4, torch.float32),
                                         ("cfg3_video_b1024", 4, torch.bfloat16), ("cfg2_image", 6, torch.float32),
                                         ("cfg2_image", 6, torch.bfloat16)])
def test_compute_occurence_map_backward(cfg, n, dtype):
    """compute_occurence_map under grad (TransformLoss re-entry, src/loss/loss.py:302) through the library: only the
    occurrence branch is differentiated -- occurrence_module parameters and the feature map get gradients, nothing else."""
    dims = synth.CONFIGS[cfg]
    bf = dtype == torch.bfloat16
    sd = synth.make_head_params(dims, seed=31, bias_scale=0.05, bf16_round=True)
    x = synth.make_features(dims, n, seed=9, bf16_round=True)
    wo = np.random.default_rng(4).standard_normal((n, dims.P, 1) + dims.spatial).astype(np.float32) * 0.1
    _, ref_gx, ref_g = _oracle_grads(x, sd, np.zeros((n, dims.K), np.float32), np.zeros((n, dims.P), np.float32), wo)
    m = build_model(dims, sd)
    m.train()
    m.autograd_mode = "kernel"
    xt = torch.from_numpy(x).cuda().to(dtype).requires_grad_(True)
    occ = m.compute_occurence_map(xt)
    assert occ.shape == (n, dims.P, 1) + dims.spatial and occ.requires_grad
    (occ.float() * torch.from_numpy(wo).cuda()).sum().backward()
    own = dict(m.named_parameters())
    rtol, afrac = (1e-2, 4e-3) if bf else (2e-4, 2e-5)
    for k in KEYS:
        if k.startswith("occurrence_module"):
            assert_close(own[k].grad.reshape(ref_g[k].shape), ref_g[k], rtol, f"grad {k}", atol_frac=afrac)
        else:
            assert own[k].grad is None, k
    assert_close(xt.grad, ref_gx, rtol, "grad feature map", atol_frac=afrac)
