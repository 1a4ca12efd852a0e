"""oracle/emulate.py, the rounding model the tensor-core forward is checked against in bf16 / fp16 mode, checked on the
CPU: against the float64 reference with its rounding switched off, against itself run in float32 (the accumulation
the kernels do), and against the reference golden of the bf16 head."""
import os

import numpy as np
import pytest
import torch

from oracle import head_oracle as ho
from oracle.emulate import cosine_chain_f64, head_forward_emulated
from protoasnet_b200 import synth
from tests.util import (BF16_RTOL, EMU_FEAT_POOL_FIRST, EMU_FEAT_W2_FIRST, EMU_LOGITS_FRAC, EMU_OCC_BITEQ, EMU_SIM_ATOL,
                        assert_close, load_golden, occ_agreement)

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
OUTPUTS = ("logits", "similarity", "distance", "occurrence_map", "features_extracted")


def _inputs(dims, n, mode, seed=23):
    sd = synth.make_head_params(dims, seed=41, bias_scale=0.05, last_layer_noise=0.1)
    x = synth.make_features(dims, n, seed=seed, bf16_round=mode == "bf16")
    if mode == "fp16":
        x = x.astype(np.float16).astype(np.float32)
    return x, sd


def _frac(a, b):
    return float(np.abs(np.asarray(a, np.float64) - b).max() / np.abs(b).max())


@pytest.mark.parametrize("mode", ["bf16", "fp16", "fp32_fused"])
@pytest.mark.parametrize("order", ["pool_first", "w2_first"])
def test_without_rounding_equals_float64_reference(mode, order):
    dims = synth.HeadDims(128, 128, 12, 3, (2, 5, 7))
    x, sd = _inputs(dims, 3, mode)
    emu = head_forward_emulated(x, sd, mode, order, rounding=False)
    ref = ho.head_forward_f64(x, sd)
    for k in OUTPUTS:
        assert _frac(emu[k], ref[k]) <= 1e-12, k


def test_rounding_points_are_applied():
    """Each rounding point leaves values of its type: catches a stage of the model that silently stopped rounding."""
    dims = synth.HeadDims(64, 128, 9, 3, (4, 8))
    x, sd = _inputs(dims, 2, "bf16")
    e = head_forward_emulated(x, sd, "bf16", "w2_first")
    for k in ("h1", "g1", "g2", "occurrence_map", "f"):
        t = torch.from_numpy(e[k])
        assert torch.equal(t, t.bfloat16().double()), k
    assert not torch.equal(torch.from_numpy(e["occurrence_abs"]), torch.from_numpy(e["occurrence_map"]))
    p = head_forward_emulated(x, sd, "bf16", "pool_first")["pooled"]
    assert not np.array_equal(p, torch.from_numpy(p).bfloat16().double().numpy())   # hi + lo, not bf16
    np.testing.assert_array_equal(head_forward_emulated(x, sd, "bf16", "pool_first", occ=e["occurrence_map"])["pooled"], p)


# the shapes of the tensor-core sweeps (C, D, P, K, spatial, n, order): fused cfg 3 / cfg 1 / padding edges, tiled image
# head and small ragged heads
SHAPES = [
    (512, 256, 40, 4, (4, 7, 7), 3, "pool_first"),
    (256, 256, 40, 4, (8, 14, 14), 2, "pool_first"),
    (64, 256, 17, 17, (1, 10, 14), 3, "pool_first"),
    (512, 512, 40, 4, (7, 7), 4, "w2_first"),
    (64, 128, 9, 3, (7, 7), 5, "w2_first"),
    (64, 256, 130, 5, (3, 3, 3), 2, "w2_first"),
]


@pytest.mark.parametrize("mode", ["bf16", "fp16", "fp32_fused"])
@pytest.mark.parametrize("shape", SHAPES, ids=[str(s) for s in SHAPES])
def test_float32_run_stays_within_parity_thresholds(shape, mode):
    """The emulation run in float32 stands in for a kernel that rounds where the model says and accumulates in fp32: it
    must meet the thresholds the GPU parity sweep holds the kernels to, with room to spare (the sweep's maxima on the B200
    are of the same size)."""
    C, D, P, K, spatial, n, order = shape
    if mode == "fp32_fused" and (order != "pool_first" or D != 256):
        pytest.skip("bf16 compute on fp32 maps is a mode of the fused pair only (D = 256, pooling first)")
    dims = synth.HeadDims(C, D, P, K, spatial)
    x, sd = _inputs(dims, n, mode)
    e64 = head_forward_emulated(x, sd, mode, order)
    e32 = head_forward_emulated(x, sd, mode, order, dtype=torch.float32)
    biteq, worst = occ_agreement(e32["occurrence_map"], e64["occurrence_map"])
    assert biteq >= EMU_OCC_BITEQ and worst <= 1.0, (biteq, worst)
    # conditioned on the map of the float32 run, as the GPU sweep does for bf16 maps
    ref = head_forward_emulated(x, sd, mode, order, occ=e32["occurrence_map"]) if mode != "fp16" else e64
    feat_tol = EMU_FEAT_POOL_FIRST if order == "pool_first" else EMU_FEAT_W2_FIRST
    assert _frac(e32["features_extracted"], ref["features_extracted"]) <= feat_tol
    assert np.abs(e32["similarity"] - ref["similarity"]).max() <= EMU_SIM_ATOL
    assert np.abs(e32["distance"] - ref["distance"]).max() <= EMU_SIM_ATOL
    assert _frac(e32["logits"], ref["logits"]) <= EMU_LOGITS_FRAC
    cc = cosine_chain_f64(e32["features_extracted"], sd)
    assert np.abs(cc["similarity"] - e32["similarity"]).max() <= 1e-6


def test_bf16_head_within_budgets_of_reference_golden():
    """The model against the reference itself: on the golden of the bf16 head (cfg 3, bf16 inputs and parameters) it is
    inside the budgets the kernels are held to against that golden."""
    z, r = load_golden(os.path.join(GOLDEN, "head_cfg3_bf16in.npz"))
    dims = synth.CONFIGS[r["config"]]
    sd = synth.make_head_params(dims, **r["params"])
    x = synth.make_features(dims, r["n"], seed=r["feature_seed"], bf16_round=True)
    e = head_forward_emulated(x, sd, "bf16", "pool_first")
    assert_close(e["logits"], z["logits"], BF16_RTOL, "logits")
    assert_close(e["similarity"], z["similarity"], BF16_RTOL, "similarity")
    assert_close(e["features_extracted"], z["features_extracted"], 4e-3, "features_extracted")
    assert_close(e["occurrence_map"], z["occurrence_map"].reshape(e["occurrence_map"].shape), 2e-2, "occurrence_map",
                 atol_frac=1e-2)
