"""GPU parity of the prototype head (through the C ABI) against the reference goldens and the CPU oracle."""
import glob
import os

import numpy as np
import pytest
import torch

from oracle import head_oracle as ho
from protoasnet_b200 import _lib, synth
from tests.util import FP32_TC_FEAT_ATOL, BF16_RTOL, FP32_RTOL, assert_close, build_model, feat_atol, load_golden

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
HEAD = sorted(glob.glob(os.path.join(GOLDEN, "head_*.npz")))


def _run_all(m, x):
    with torch.no_grad():
        logits, sim, occ = m(x)
        feats, dist, occ2, logits2 = m.push_forward(x)
        occ3 = m.compute_occurence_map(x)
    return dict(logits=logits, similarity=sim, occurrence_map=occ, features_extracted=feats, distance=dist,
                occ2=occ2, occ3=occ3, logits2=logits2)


@pytest.mark.parametrize("kernel_path", [_lib.PASN_PATH_AUTO, _lib.PASN_PATH_GENERIC], ids=["auto", "generic"])
@pytest.mark.parametrize("path", HEAD, ids=[os.path.basename(p)[:-4] for p in HEAD])
def test_fp32_matches_reference_golden(path, kernel_path):
    """fp32 feature maps against the goldens produced by the reference classes.  ``auto``: the tiled tensor-core path
    (bf16 hi/lo split) where the shape qualifies (cfg 1 / 2 / 3), CUDA-core FFMA otherwise; ``generic``: FFMA everywhere."""
    z, r = load_golden(path)
    dims = synth.CONFIGS[r["config"]]
    sd = synth.make_head_params(dims, **r["params"])
    x = synth.make_features(dims, r["n"], seed=r["feature_seed"], bf16_round=r["bf16_round"])
    m = build_model(dims, sd, path=kernel_path)
    xg = torch.from_numpy(x).cuda()
    out = _run_all(m, xg)
    fa = feat_atol(m, xg)
    assert tuple(out["occurrence_map"].shape) == z["occurrence_map"].shape
    for k in ("logits", "similarity", "distance"):
        assert_close(out[k], z[k], FP32_RTOL, k)
    for k in ("occurrence_map", "features_extracted"):
        assert_close(out[k], z[k], FP32_RTOL, k, atol_frac=fa)
    assert torch.equal(out["distance"], 1 - out["similarity"])
    assert torch.equal(out["logits"], out["logits2"])
    assert_close(out["occ3"], z["occurrence_map"], FP32_RTOL, "compute_occurence_map", atol_frac=fa)


@pytest.mark.parametrize("case", ["head_cfg3_bf16in"])
def test_bf16_matches_reference_golden(case):
    """bf16 mode: oracle = reference in fp32 on bf16-rounded inputs and weights (SURVEY.md section 7)."""
    z, r = load_golden(os.path.join(GOLDEN, case + ".npz"))
    dims = synth.CONFIGS[r["config"]]
    sd = synth.make_head_params(dims, **r["params"])
    x = synth.make_features(dims, r["n"], seed=r["feature_seed"], bf16_round=True)
    m = build_model(dims, sd)
    out = _run_all(m, torch.from_numpy(x).cuda().bfloat16())
    assert out["occurrence_map"].dtype == torch.bfloat16
    assert_close(out["logits"], z["logits"], BF16_RTOL, "logits")
    assert_close(out["similarity"], z["similarity"], BF16_RTOL, "similarity")
    assert_close(out["features_extracted"], z["features_extracted"], 4e-3, "features_extracted")
    # the map itself is stored in bf16 and computed from bf16 hidden activations: entries are judged against the
    # map's scale (|.| of a near-zero pre-activation has no meaningful relative error)
    assert_close(out["occurrence_map"], z["occurrence_map"], 2e-2, "occurrence_map (bf16)", atol_frac=1e-2)
    # compute_occurence_map (Video_XProtoNet.py:100-109) and push_forward's copy of the map, bf16 output
    assert out["occ3"].dtype == torch.bfloat16 and out["occ3"].shape == out["occurrence_map"].shape
    assert_close(out["occ3"], z["occurrence_map"], 2e-2, "compute_occurence_map (bf16)", atol_frac=1e-2)
    assert_close(out["occ2"], z["occurrence_map"], 2e-2, "push_forward occurrence_map (bf16)", atol_frac=1e-2)


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
def test_cfg5_scaled_sweep_matches_oracle(dtype):
    """BASELINE config 5 (P=4096, D=512, C=512, 16x14x14 feature maps) at N=2 against the CPU oracle (the reference's ops
    with the broadcast product reduced 16 prototypes at a time -- the full product would need 26 GB per clip)."""
    dims = synth.CONFIGS["cfg5_scaled"]
    bf = dtype == torch.bfloat16
    sd = synth.make_head_params(dims, seed=200, bias_scale=0.02, bf16_round=bf)
    x = synth.make_features(dims, 2, seed=3, bf16_round=bf)
    torch.set_num_threads(os.cpu_count() or 1)
    with torch.no_grad():
        rf, rd, ro, rl = ho.push_forward_torch_pchunk(torch.from_numpy(x), ho.to_torch_sd(sd), p_chunk=16)
    m = build_model(dims, sd)
    out = _run_all(m, torch.from_numpy(x).cuda().to(dtype))
    tol = BF16_RTOL if bf else FP32_RTOL
    assert_close(out["logits"], rl.numpy(), tol, "logits")
    assert_close(out["similarity"], (1 - rd).numpy(), tol, "similarity")
    assert_close(out["distance"], rd.numpy(), tol, "distance", atol_frac=tol)
    if bf:
        assert_close(out["features_extracted"], rf.numpy(), 4e-3, "features_extracted")
        assert_close(out["occurrence_map"], ro.numpy(), 2e-2, "occurrence_map (bf16)", atol_frac=1e-2)
        assert_close(out["occ3"], ro.numpy(), 2e-2, "compute_occurence_map (bf16)", atol_frac=1e-2)
    else:
        fa = feat_atol(m, torch.from_numpy(x).cuda())
        assert_close(out["features_extracted"], rf.numpy(), FP32_RTOL, "features_extracted", atol_frac=fa)
        assert_close(out["occurrence_map"], ro.numpy(), FP32_RTOL, "occurrence_map", atol_frac=fa)
        assert_close(out["occ3"], ro.numpy(), FP32_RTOL, "compute_occurence_map", atol_frac=fa)
    # forward() at P >= 1024 takes its cosine from row statistics left by the pooling GEMM (the 8 MB of pooled features per
    # clip are never stored), push_forward() from the stored features: same fp32 formula, different summation order
    assert float((out["distance"] - (1 - out["similarity"])).abs().max()) < 2e-6


def test_cfg2_image_bf16_matches_oracle():
    """BASELINE config 2 (image head, D=512, 7x7) in bf16 at the push-loader batch of 150 (as_dataloader.py:49-50)."""
    dims = synth.CONFIGS["cfg2_image"]
    sd = synth.make_head_params(dims, seed=200, bias_scale=0.02, bf16_round=True)
    x = synth.make_features(dims, 150, seed=5, bf16_round=True)
    with torch.no_grad():
        rf, rd, ro, rl = ho.push_forward_torch(torch.from_numpy(x), ho.to_torch_sd(sd))
    m = build_model(dims, sd)
    out = _run_all(m, torch.from_numpy(x).cuda().bfloat16())
    assert_close(out["logits"], rl.numpy(), BF16_RTOL, "logits")
    assert_close(out["similarity"], (1 - rd).numpy(), BF16_RTOL, "similarity")
    # pooled features: bf16 hidden activations (H1, O: 2^-9 relative each) summed over only S = 49 voxels -- entries are
    # judged against the tensor's scale at 1e-3 (measured 7e-4); north_star's 1e-3 bound is on logits / similarities
    assert_close(out["features_extracted"], rf.numpy(), 4e-3, "features_extracted", atol_frac=1e-3)
    assert_close(out["occurrence_map"], ro.numpy(), 2e-2, "occurrence_map (bf16)", atol_frac=1e-2)
    assert_close(out["occ3"], ro.numpy(), 2e-2, "compute_occurence_map (bf16)", atol_frac=1e-2)


SHAPES = [
    # C, D, P, K, spatial, n
    (7, 6, 4, 2, (1, 1, 1), 3),      # S = 1
    (33, 18, 9, 3, (3, 3, 3), 2),    # nothing a multiple of 8/16
    (64, 32, 8, 4, (5, 7), 5),       # image head
    (130, 66, 6, 2, (2, 9, 5), 1),   # dims just over a tile edge
    (16, 8, 128, 4, (2, 2, 2), 2),   # many prototypes
]


@pytest.mark.parametrize("shape", SHAPES, ids=[str(s) for s in SHAPES])
@pytest.mark.parametrize("layout", ["ncs", "nsc"])
def test_ragged_shapes_and_layouts_vs_oracle(shape, layout):
    C, D, P, K, spatial, n = shape
    dims = synth.HeadDims(C, D, P, K, spatial)
    sd = synth.make_head_params(dims, seed=31, bias_scale=0.1, last_layer_noise=0.2)
    x = synth.make_features(dims, n, seed=17)
    tsd = ho.to_torch_sd(sd)
    with torch.no_grad():
        rf, rd, ro, rl = ho.push_forward_torch(torch.from_numpy(x), tsd)
        _, rs, _ = ho.head_forward_torch(torch.from_numpy(x), tsd)
    m = build_model(dims, sd)
    xg = torch.from_numpy(x).cuda()
    if layout == "nsc":
        xg = xg.contiguous(memory_format=torch.channels_last_3d if len(spatial) == 3 else torch.channels_last)
    out = _run_all(m, xg)
    assert_close(out["logits"], rl.numpy(), FP32_RTOL, "logits")
    assert_close(out["similarity"], rs.numpy(), FP32_RTOL, "similarity")
    assert_close(out["occurrence_map"], ro.numpy(), FP32_RTOL, "occ")
    assert_close(out["features_extracted"], rf.numpy(), FP32_RTOL, "feats")
    assert_close(out["distance"], rd.numpy(), FP32_RTOL, "dist")


def test_empty_batch_and_errors():
    dims = synth.CONFIGS["tiny_video"]
    m = build_model(dims, synth.make_head_params(dims, seed=1))
    with torch.no_grad():
        logits, sim, occ = m(torch.zeros((0, dims.C) + dims.spatial, device="cuda"))
    assert logits.shape == (0, dims.K) and sim.shape == (0, dims.P) and occ.shape[0] == 0
    with torch.no_grad(), pytest.raises(_lib.PasnError):
        m(torch.zeros((2, dims.C + 1) + dims.spatial, device="cuda"))          # wrong channel count
    with torch.no_grad(), pytest.raises(_lib.PasnError):
        m(torch.zeros((2, dims.C) + dims.spatial, device="cuda", dtype=torch.float16))


def test_zero_features_hit_cosine_eps_clamp():
    """All-zero clip: pooled features are exactly 0 -> the 1e-8 norm clamp path; similarity must be exactly 0.5."""
    dims = synth.CONFIGS["tiny_video"]
    m = build_model(dims, synth.make_head_params(dims, seed=3))   # zero biases (reference init)
    with torch.no_grad():
        logits, sim, occ = m(torch.zeros((2, dims.C) + dims.spatial, device="cuda"))
    assert torch.all(sim == 0.5) and torch.all(occ == 0)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_full_size_properties_cfg3(dtype):
    """BASELINE config 3 at full size (N=1024): size-independent properties + a spot check against the oracle."""
    dims = synth.CONFIGS["cfg3_video_b1024"]
    bf = dtype == torch.bfloat16
    sd = synth.make_head_params(dims, seed=200, bias_scale=0.02, bf16_round=bf)
    m = build_model(dims, sd)
    g = torch.Generator(device="cuda").manual_seed(0)
    x = torch.relu(torch.randn((1024, dims.C) + dims.spatial, device="cuda", generator=g)).to(dtype)
    with torch.no_grad():
        f, d, occ, logits = m.push_forward(x)
        logits_a, sim_a, _ = m(x)
        perm = torch.randperm(1024, device="cuda", generator=g)
        f_p, d_p, occ_p, logits_p = m.push_forward(x[perm])
        parts = [m.push_forward(x[i:i + 200]) for i in range(0, 1024, 200)]
    # distance is exactly 1 - similarity; similarity in [0, 1]
    assert torch.equal(d, 1 - sim_a) and float(sim_a.min()) >= 0 and float(sim_a.max()) <= 1.0 + 1e-6
    assert torch.equal(logits, logits_a)
    # clips are independent: permuting / re-chunking the batch permutes / concatenates the outputs
    tol = FP32_RTOL if not bf else BF16_RTOL
    assert_close(d_p, d[perm].cpu().numpy(), tol, "perm dist")
    assert_close(torch.cat([p[1] for p in parts]), d.cpu().numpy(), tol, "chunk dist")
    assert_close(torch.cat([p[3] for p in parts]), logits.cpu().numpy(), tol, "chunk logits")
    # logits are the last layer applied to the similarities (linearity check of the epilogue)
    assert_close(logits, (sim_a.double() @ m.last_layer.weight.detach().double().t()).cpu().numpy(), 1e-6, "logits=W sim")
    # occurrence map is non-negative (abs) and pooled features reproduce from it: spot check 3 clips vs oracle
    assert float(occ.float().min()) >= 0
    idx = [0, 517, 1023]
    xs = x[idx].float().cpu()
    with torch.no_grad():
        rf, rd, ro, rl = ho.push_forward_torch(xs, ho.to_torch_sd(sd))
    assert_close(d[idx], rd.numpy(), tol, "dist vs oracle")
    assert_close(logits[idx], rl.numpy(), tol, "logits vs oracle")
    assert_close(f[idx], rf.numpy(), tol if not bf else 4e-3, "feats vs oracle", atol_frac=feat_atol(m, x))


# ------------------------------------------------------------------------------------------------
# fused tcgen05 path: shape sweep (every template instantiation, ragged tails, CTA / tile boundaries)
# ------------------------------------------------------------------------------------------------
TC_SHAPES = [
    # C, P, K, spatial (S % 4 == 0, S >= 128), n
    (64, 8, 4, (2, 8, 8), 3),        # smallest channel count, PP=16 instantiation, S = 128 (tile == clip)
    (128, 12, 3, (1, 10, 14), 5),    # S = 140: every tile straddles clips; P not a multiple of 8
    (256, 24, 4, (8, 14, 14), 2),    # cfg-1 feature map, PP=32
    (512, 40, 4, (4, 7, 7), 9),      # cfg-3, PP=40
    (512, 48, 4, (4, 7, 7), 4),      # PP=48
    (1024, 40, 8, (3, 8, 8), 2),     # 16 channel chunks; S = 192
    (512, 40, 4, (4, 7, 7), 149),    # one more clip than SMs: uneven clip ranges per CTA
    (512, 40, 4, (4, 7, 7), 301),    # 3 clips per CTA with a short last CTA
]


@pytest.mark.parametrize("shape", TC_SHAPES, ids=[str(s) for s in TC_SHAPES])
def test_tcgen05_path_shape_sweep(shape):
    C, P, K, spatial, n = shape
    dims = synth.HeadDims(C, 256, P, K, spatial)
    sd = synth.make_head_params(dims, seed=41, bias_scale=0.05, last_layer_noise=0.1, bf16_round=True)
    x = synth.make_features(dims, n, seed=23, bf16_round=True)
    m = build_model(dims, sd, path=_lib.PASN_PATH_TCGEN05)      # errors out if the fused path cannot take the shape
    mg = build_model(dims, sd, path=_lib.PASN_PATH_GENERIC)
    xg = torch.from_numpy(x).cuda().bfloat16()
    out = _run_all(m, xg)
    ref = _run_all(mg, xg)                                      # generic CUDA path: fp32 math on the same bf16 inputs
    nref = min(n, 4)
    with torch.no_grad():
        rf, rd, ro, rl = ho.push_forward_torch(torch.from_numpy(x[:nref]), ho.to_torch_sd(sd))
    assert_close(out["similarity"][:nref], (1 - rd).numpy(), BF16_RTOL, "similarity vs oracle")
    assert_close(out["logits"][:nref], rl.numpy(), BF16_RTOL, "logits vs oracle")
    assert_close(out["similarity"], ref["similarity"].cpu().numpy(), BF16_RTOL, "similarity vs generic")
    assert_close(out["logits"], ref["logits"].cpu().numpy(), BF16_RTOL, "logits vs generic")
    assert_close(out["features_extracted"], ref["features_extracted"].cpu().numpy(), 4e-3, "features vs generic")
    assert_close(out["occurrence_map"], ref["occurrence_map"].float().cpu().numpy(), 2e-2, "occ vs generic", atol_frac=1e-2)
    assert torch.equal(out["distance"], 1 - out["similarity"])


TILED_SHAPES = [
    # C, D, P, K, spatial, n       (C a multiple of 64, D of 128: what the tiled GEMM chain takes)
    (64, 128, 9, 3, (7,  7), 5),          # odd P and S: unaligned map rows -> plain stores; W2 before the pooling
    (128, 128, 33, 3, (1, 5, 10), 3),     # P just over a 32-column group, S = 50 (16-byte aligned rows)
    (64, 256, 130, 5, (3, 3, 3), 2),      # P over one 128-row tile, S = 27
    (192, 128, 8, 2, (2, 10, 12), 7),     # S = 240 > 2P: W2 after the pooling (row sums, rank-1 bias term)
    (512, 512, 40, 4, (7, 7), 11),        # the image head
    (64, 128, 72, 4, (4, 16, 16), 2),     # P > 64: occurrence GEMM per clip, S = 1024 (aligned: no transposition in bf16)
    (128, 256, 40, 4, (1, 2, 4), 1),      # a single clip of 8 voxels: every GEMM is one ragged tile
]


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32], ids=["bf16", "fp32"])
@pytest.mark.parametrize("layout", ["ncs", "nsc"])
@pytest.mark.parametrize("shape", TILED_SHAPES, ids=[str(s) for s in TILED_SHAPES])
def test_tiled_path_shape_sweep(shape, layout, dtype):
    """The tiled tensor-core chain (explicitly requested) on ragged shapes, both layouts and dtypes, against the CPU oracle."""
    C, D, P, K, spatial, n = shape
    dims = synth.HeadDims(C, D, P, K, spatial)
    bf = dtype == torch.bfloat16
    sd = synth.make_head_params(dims, seed=43, bias_scale=0.05, last_layer_noise=0.1, bf16_round=bf)
    x = synth.make_features(dims, n, seed=29, bf16_round=bf)
    m = build_model(dims, sd, path=_lib.PASN_PATH_TILED)        # errors out if the tiled path cannot take the shape
    xg = torch.from_numpy(x).cuda().to(dtype)
    if layout == "nsc":
        xg = xg.contiguous(memory_format=torch.channels_last_3d if dims.ndim == 3 else torch.channels_last)
    out = _run_all(m, xg)
    with torch.no_grad():
        rf, rd, ro, rl = ho.push_forward_torch(torch.from_numpy(x), ho.to_torch_sd(sd))
    tol = BF16_RTOL if bf else FP32_RTOL
    assert_close(out["similarity"], (1 - rd).numpy(), tol, "similarity")
    assert_close(out["logits"], rl.numpy(), tol, "logits")
    # forward() may take its cosine from row statistics folded into the pooling GEMM (few prototypes, W2 before the pooling),
    # push_forward() from the stored features: the same fp32 formula in another summation order
    assert float((out["distance"] - (1 - out["similarity"])).abs().max()) < 2e-6
    assert_close(out["logits"], out["logits2"].cpu().numpy(), 1e-5, "forward vs push_forward logits", atol_frac=2e-6)
    if bf:
        # bf16 hidden activations (2^-9 relative each) are averaged over the S voxels of a clip: the fewer voxels, the
        # more of that rounding is left in the pooled features (north_star's 1e-3 bound is on similarities / logits, above)
        assert_close(out["features_extracted"], rf.numpy(), 4e-3, "features_extracted", atol_frac=max(1e-3, 6e-3 / dims.S ** 0.5))
        for k in ("occurrence_map", "occ2", "occ3"):
            assert_close(out[k], ro.numpy(), 2e-2, k, atol_frac=1e-2)
    else:
        for k in ("occurrence_map", "occ2", "occ3"):
            assert_close(out[k], ro.numpy(), FP32_RTOL, k, atol_frac=FP32_TC_FEAT_ATOL)
        assert_close(out["features_extracted"], rf.numpy(), FP32_RTOL, "features_extracted", atol_frac=FP32_TC_FEAT_ATOL)


def test_tcgen05_path_refuses_unsupported_shapes():
    dims = synth.CONFIGS["cfg2_image"]                            # D = 512, S = 49: generic path only (DESIGN.md section 7)
    m = build_model(dims, synth.make_head_params(dims, seed=1, bf16_round=True), path=_lib.PASN_PATH_TCGEN05)
    x = torch.zeros((2, dims.C) + dims.spatial, device="cuda", dtype=torch.bfloat16)
    with torch.no_grad(), pytest.raises(_lib.PasnError):
        m(x)
    m.kernel_path = _lib.PASN_PATH_AUTO                           # AUTO silently picks the generic CUDA path
    with torch.no_grad():
        logits, sim, occ = m(x)
    assert logits.shape == (2, dims.K)


def test_cfg2_image_bf16_generic_matches_oracle():
    dims = synth.CONFIGS["cfg2_image"]
    sd = synth.make_head_params(dims, seed=200, bias_scale=0.02, bf16_round=True)
    x = synth.make_features(dims, 5, seed=0, bf16_round=True)
    m = build_model(dims, sd, path=_lib.PASN_PATH_GENERIC)   # AUTO serves this shape on the tiled tensor-core path
    out = _run_all(m, torch.from_numpy(x).cuda().bfloat16())
    with torch.no_grad():
        rf, rd, ro, rl = ho.push_forward_torch(torch.from_numpy(x), ho.to_torch_sd(sd))
    assert_close(out["similarity"], (1 - rd).numpy(), BF16_RTOL, "similarity")
    assert_close(out["logits"], rl.numpy(), BF16_RTOL, "logits")
    assert_close(out["features_extracted"], rf.numpy(), BF16_RTOL, "features (fp32 math on bf16 inputs)")


def test_tcgen05_bf16_compute_on_fp32_features():
    """Opt-in fused path for fp32 feature maps (the reference's native dtype): inputs are rounded to bf16 on the fly."""
    dims = synth.CONFIGS["cfg3_video_b1024"]
    sd = synth.make_head_params(dims, seed=200, bias_scale=0.02, bf16_round=True)
    m = build_model(dims, sd, path=_lib.PASN_PATH_TCGEN05)
    # (a) bf16-representable fp32 inputs must reproduce the bf16-input run exactly (same kernel arithmetic)
    x = synth.make_features(dims, 9, seed=3, bf16_round=True)
    xg = torch.from_numpy(x).cuda()
    o32 = _run_all(m, xg)
    o16 = _run_all(m, xg.bfloat16())
    assert o32["occurrence_map"].dtype == torch.float32
    assert torch.equal(o32["similarity"], o16["similarity"]) and torch.equal(o32["logits"], o16["logits"])
    assert torch.equal(o32["features_extracted"], o16["features_extracted"])
    assert torch.equal(o32["occurrence_map"], o16["occurrence_map"].float())
    # (b) arbitrary fp32 inputs: within the bf16 budget of the fp32 reference on the unrounded inputs
    x2 = synth.make_features(dims, 4, seed=5, bf16_round=False)
    with torch.no_grad():
        rf, rd, ro, rl = ho.push_forward_torch(torch.from_numpy(x2), ho.to_torch_sd(sd))
    o = _run_all(m, torch.from_numpy(x2).cuda())
    assert_close(o["similarity"], (1 - rd).numpy(), BF16_RTOL, "similarity")
    assert_close(o["logits"], rl.numpy(), BF16_RTOL, "logits")
    # AUTO takes fp32 inputs through the hi/lo-split tiled path: fp32 parity on the similarities
    m.kernel_path = _lib.PASN_PATH_AUTO
    oa = _run_all(m, torch.from_numpy(x2).cuda())
    assert_close(oa["similarity"], (1 - rd).numpy(), FP32_RTOL, "similarity (fp32 path)")


# tiles that straddle clips; P = 40 / 24 / 12 (padded to 40 / 24 / 16 rows); C = 512 / 256 / 128
FUSED_SHAPES = [(512, 40, 4, (4, 7, 7), 37), (256, 24, 4, (8, 14, 14), 2), (128, 12, 3, (1, 10, 14), 5)]


@pytest.mark.parametrize("shape", FUSED_SHAPES, ids=[str(s) for s in FUSED_SHAPES])
def test_token_kernel_matches_generic_path(shape):
    """The fused token kernel stays inside the bf16 budget against the generic CUDA path."""
    C, P, K, spatial, n = shape
    dims = synth.HeadDims(C, 256, P, K, spatial)
    sd = synth.make_head_params(dims, seed=77, bias_scale=0.05, last_layer_noise=0.1, bf16_round=True)
    xg = torch.from_numpy(synth.make_features(dims, n, seed=29, bf16_round=True)).cuda().bfloat16()
    out = _run_all(build_model(dims, sd, path=_lib.PASN_PATH_TCGEN05), xg)
    ref = _run_all(build_model(dims, sd, path=_lib.PASN_PATH_GENERIC), xg)
    assert_close(out["similarity"], ref["similarity"].cpu().numpy(), BF16_RTOL, "similarity")
    assert_close(out["logits"], ref["logits"].cpu().numpy(), BF16_RTOL, "logits")


@pytest.mark.parametrize("shape", [(512, 40, 4, (4, 7, 7), 37), (256, 24, 4, (8, 14, 14), 2), (64, 8, 4, (2, 8, 8), 3),
                                   (1024, 40, 8, (3, 8, 8), 2)], ids=str)
def test_tcgen05_channels_last_matches_ncdhw(shape):
    """A channels_last_3d bf16 feature map ([N,S,C] in memory) takes the fused path directly (K-major X tile, 16-byte
    cp.async gather) and gives the same results as the NCDHW gather: same MMAs in the same order."""
    C, P, K, spatial, n = shape
    dims = synth.HeadDims(C, 256, P, K, spatial)
    sd = synth.make_head_params(dims, seed=5, bias_scale=0.05, last_layer_noise=0.1, bf16_round=True)
    x = torch.from_numpy(synth.make_features(dims, n, seed=31, bf16_round=True)).cuda().bfloat16()
    xcl = x.contiguous(memory_format=torch.channels_last_3d)
    assert not xcl.is_contiguous() and xcl.is_contiguous(memory_format=torch.channels_last_3d)
    m = build_model(dims, sd, path=_lib.PASN_PATH_TCGEN05)
    ref = _run_all(m, x)
    out = _run_all(m, xcl)
    for k in ("logits", "similarity", "features_extracted", "distance"):
        assert_close(out[k], ref[k].cpu().numpy(), 1e-5, f"{k}, channels_last")
    assert out["occurrence_map"].shape == ref["occurrence_map"].shape
    assert torch.equal(out["occurrence_map"], ref["occurrence_map"])


def test_host_pipeline_matches_direct_forward():
    """HostPipeline (chunked H2D copy overlapped with the kernels, pinned host results) == forward on the device tensor."""
    import protoasnet_b200 as pasn
    dims = synth.CONFIGS["cfg3_video_b1024"]
    sd = synth.make_head_params(dims, seed=200, bias_scale=0.02, bf16_round=True)
    m = build_model(dims, sd)
    x = torch.from_numpy(synth.make_features(dims, 37, seed=2, bf16_round=True)).bfloat16()
    xh = x.pin_memory()
    with torch.no_grad():
        logits, sim, occ = m(x.cuda())
    pipe = pasn.HostPipeline(m, chunks=4, want_occ=True)
    for _ in range(2):      # second call reuses the staging buffers
        lg, sm, oc = pipe(xh)
        torch.cuda.synchronize()
        assert lg.is_pinned() and not lg.is_cuda
        # per-chunk launches tile the clips differently (clips per CTA), so pooled sums may differ in the last bits
        assert_close(lg, logits.cpu().numpy(), 1e-5, "logits")
        assert_close(sm, sim.cpu().numpy(), 1e-5, "similarity")
        assert torch.equal(oc, occ.cpu())
    lg1, sm1 = pasn.HostPipeline(m, chunks=1)(xh)
    torch.cuda.synchronize()
    assert torch.equal(lg1, logits.cpu()) and torch.equal(sm1, sim.cpu())


def test_forward_is_cuda_graph_capturable():
    """The C ABI neither allocates nor synchronises, so a forward call can be captured in a CUDA graph and replayed
    (serving loops): same results as the eager call, on new input data copied into the captured buffer."""
    dims = synth.CONFIGS["cfg3_video_b1024"]
    sd = synth.make_head_params(dims, seed=200, bias_scale=0.02, bf16_round=True)
    m = build_model(dims, sd)
    x1 = torch.from_numpy(synth.make_features(dims, 33, seed=7, bf16_round=True)).cuda().bfloat16()
    x2 = torch.from_numpy(synth.make_features(dims, 33, seed=8, bf16_round=True)).cuda().bfloat16()
    static_x = x1.clone()
    with torch.no_grad():
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            for _ in range(2):      # warm-up: function attributes, packed weights, workspace
                m(static_x)
        torch.cuda.current_stream().wait_stream(s)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            logits, sim, occ = m(static_x)
        for x in (x1, x2):
            static_x.copy_(x)
            g.replay()
            torch.cuda.synchronize()
            el, es, eo = m(x)
            assert torch.equal(logits, el) and torch.equal(sim, es) and torch.equal(occ, eo)


def test_small_batch_voxel_group_split_matches_unsplit():
    """Batches that cannot fill the SMs (cfg 1: 8 clips of 1568 voxels) are processed as G voxel groups per clip whose
    pooled features are summed after K2.  Same results as the unsplit computation (the generic fp32-math path on the
    same bf16 inputs: the fused path always splits a batch this small) and the fixed-size outputs agree with a larger
    batch that is not split."""
    dims = synth.CONFIGS["cfg1_video_yml"]
    sd = synth.make_head_params(dims, seed=200, bias_scale=0.02, bf16_round=True)
    m = build_model(dims, sd, path=_lib.PASN_PATH_TCGEN05)
    mg = build_model(dims, sd, path=_lib.PASN_PATH_GENERIC)
    x = torch.from_numpy(synth.make_features(dims, 80, seed=3, bf16_round=True)).cuda().bfloat16()
    big = _run_all(m, x)                                  # 80 clips: no split
    for n in (1, 5, 8):
        small = _run_all(m, x[:n])                        # split into voxel groups
        ref = _run_all(mg, x[:n])
        assert_close(small["similarity"], ref["similarity"].cpu().numpy(), BF16_RTOL, f"similarity n={n}")
        assert_close(small["logits"], ref["logits"].cpu().numpy(), BF16_RTOL, f"logits n={n}")
        assert torch.equal(small["distance"], 1 - small["similarity"])
        assert torch.equal(small["occurrence_map"], big["occurrence_map"][:n])      # per-voxel results do not depend on the split
        assert_close(small["similarity"], big["similarity"][:n].cpu().numpy(), 1e-4, f"split vs unsplit n={n}")
        assert_close(small["features_extracted"], big["features_extracted"][:n].cpu().numpy(), 1e-4, f"features n={n}")


def test_sticky_fault_word_is_surfaced_without_debug_sync():
    """A kernel that gives up on a bounded wait writes a code into the host-mapped fault word; every later compute call
    must then fail loudly (PASN_ERR_FAULT) instead of returning garbage with status 0 -- no PASN_DEBUG_SYNC needed."""
    dims = synth.CONFIGS["tiny_video"]
    m = build_model(dims, synth.make_head_params(dims, seed=1))
    x = torch.zeros((2, dims.C) + dims.spatial, device="cuda")
    lib = _lib.load()
    with torch.no_grad():
        m(x)
    assert lib.pasn_debug_fault() == 0
    try:
        assert lib.pasn_debug_set_fault(612) == 0
        with torch.no_grad(), pytest.raises(_lib.PasnError, match="fault"):
            m(x)
        with torch.no_grad(), pytest.raises(_lib.PasnError, match="fault"):
            m.compute_occurence_map(x)
    finally:
        lib.pasn_debug_set_fault(0)
    with torch.no_grad():
        m(x)
