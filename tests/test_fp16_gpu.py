"""fp16 feature maps (torch.autocast's default dtype, PASN_F16) on the two tensor-core families: forward, push_forward,
compute_occurence_map, push, backward, the loss consumers and the host pipeline, against the CPU oracle in fp32 / float64
on the same fp16 input.  Numerics of fp16 mode: the map is read exactly, the first-layer weights are rounded to fp16,
everything after the first layer is bf16 mode's arithmetic -- so bf16 mode's tolerances apply."""
import ctypes as C

import numpy as np
import pytest
import torch

import protoasnet_b200 as pasn
from oracle import head_oracle as ho
from oracle import push_oracle as po
from protoasnet_b200 import _lib, synth
from protoasnet_b200 import push as pushmod
from tests.test_backward_gpu import KEYS, _oracle_grads
from tests.test_fp16_cpu import Gemm, Output, OUT_F16
from tests.util import BF16_RTOL, assert_close, build_model

pytestmark = pytest.mark.gpu


def _f16_input(dims, n, seed):
    """fp16 feature map on the GPU and the same values as fp32 numpy for the oracle."""
    x16 = torch.from_numpy(synth.make_features(dims, n, seed=seed)).half()
    return x16.cuda(), x16.float().numpy()


def _check_head(m, xg, x_ref, sd, pchunk=False):
    with torch.no_grad():
        logits, sim, occ = m(xg)
        feats, dist, occ2, logits2 = m.push_forward(xg)
        occ3 = m.compute_occurence_map(xg)
        if pchunk:
            rf, rd, ro, rl = ho.push_forward_torch_pchunk(torch.from_numpy(x_ref), ho.to_torch_sd(sd), p_chunk=16)
        else:
            rf, rd, ro, rl = ho.push_forward_torch(torch.from_numpy(x_ref), ho.to_torch_sd(sd))
    for o in (occ, occ2, occ3):
        assert o.dtype == torch.float16 and tuple(o.shape) == tuple(ro.shape)
    assert logits.dtype == sim.dtype == feats.dtype == torch.float32
    assert_close(logits, rl.numpy(), BF16_RTOL, "logits")
    assert_close(sim, (1 - rd).numpy(), BF16_RTOL, "similarity")
    assert_close(dist, rd.numpy(), BF16_RTOL, "distance", atol_frac=BF16_RTOL)
    assert_close(feats, rf.numpy(), 4e-3, "features_extracted", atol_frac=1e-3)
    for name, o in (("occurrence_map", occ), ("push_forward map", occ2), ("compute_occurence_map", occ3)):
        assert_close(o, ro.numpy(), 2e-2, name, atol_frac=1e-2)
    assert torch.equal(occ, occ2) and torch.equal(occ, occ3)
    # (forward() may take its cosine from row statistics of the pooling GEMM, push_forward() from the stored features: same
    # fp32 formula, another summation order)
    assert float((logits - logits2).abs().max()) <= 2e-6 * float(logits.abs().max())


@pytest.mark.parametrize("cfg,n,layout", [("cfg3_video_b1024", 37, "ncs"), ("cfg3_video_b1024", 37, "nsc"),
                                          ("cfg1_video_yml", 8, "ncs")])
def test_fused_path_matches_oracle(cfg, n, layout):
    """Fused token kernel pair: N = 37 makes 128-voxel tiles straddle clips; cfg 1 at N = 8 takes the voxel-group split."""
    dims = synth.CONFIGS[cfg]
    sd = synth.make_head_params(dims, seed=200, bias_scale=0.05, bf16_round=True)
    xg, x_ref = _f16_input(dims, n, seed=4)
    if layout == "nsc":
        xg = xg.contiguous(memory_format=torch.channels_last_3d)
    m = build_model(dims, sd)
    lib = _lib.load()
    dims_c = m._rt.make_dims(xg, m.kernel_path)[0]
    assert dims_c.dtype == _lib.PASN_F16 and dims_c.layout == (_lib.PASN_LAYOUT_NSC if layout == "nsc" else _lib.PASN_LAYOUT_NCS)
    def launches(x):
        with torch.no_grad():
            m(x)   # packs the weights
            torch.cuda.synchronize()
            c0 = lib.pasn_debug_launch_count()
            m(x)
            torch.cuda.synchronize()
        return lib.pasn_debug_launch_count() - c0
    # the fused pair (token kernel + prototype kernel; the voxel-group split of cfg 1 adds its sum and prototype stage), the
    # same launches as bf16 mode on this shape
    launched = launches(xg)
    assert launched == launches(xg.bfloat16()), launched
    if cfg == "cfg3_video_b1024":
        assert launched == 2, launched
    _check_head(m, xg, x_ref, sd)


def test_feature_map_is_not_rounded_to_bf16():
    """Two channels carry 257 and 256 (exact in fp16; bf16 rounds 257 to 256).  One-hot rows of W3 form their difference,
    identity-like W4 / W5 carry it to the occurrence map: fp16 mode gives 1 where a bf16 rounding of the input gives 0."""
    dims = synth.CONFIGS["cfg3_video_b1024"]
    sd = synth.make_head_params(dims, seed=1, bias_scale=0.0, bf16_round=True)
    D, C, P = dims.D, dims.C, dims.P
    w3 = np.zeros((D, C), np.float32); w3[0, 0], w3[0, 1] = 1.0, -1.0          # G1[0] = relu(x0 - x1)
    w4 = np.zeros((D // 2, D), np.float32); w4[0, 0] = 1.0                     # G2[0] = G1[0]
    w5 = np.zeros((P, D // 2), np.float32); w5[:, 0] = 1.0                     # O[p] = |G2[0]|
    sd["occurrence_module.0.weight"] = w3.reshape(sd["occurrence_module.0.weight"].shape)
    sd["occurrence_module.2.weight"] = w4.reshape(sd["occurrence_module.2.weight"].shape)
    sd["occurrence_module.4.weight"] = w5.reshape(sd["occurrence_module.4.weight"].shape)
    for k in ("occurrence_module.0.bias", "occurrence_module.2.bias"):
        sd[k] = np.zeros_like(sd[k])
    x = np.zeros((2, C) + dims.spatial, np.float32)
    x[:, 0], x[:, 1] = 257.0, 256.0
    m = build_model(dims, sd)
    with torch.no_grad():
        occ16 = m.compute_occurence_map(torch.from_numpy(x).cuda().half())
        occ_bf = m.compute_occurence_map(torch.from_numpy(x).cuda().bfloat16())
    assert float(occ16.float().min()) == 1.0 and float(occ16.float().max()) == 1.0
    assert float(occ_bf.float().abs().max()) == 0.0


@pytest.mark.parametrize("cfg,n", [("cfg2_image", 150), ("cfg5_scaled", 2)])
def test_tiled_path_matches_oracle(cfg, n):
    dims = synth.CONFIGS[cfg]
    sd = synth.make_head_params(dims, seed=200, bias_scale=0.02, bf16_round=True)
    xg, x_ref = _f16_input(dims, n, seed=5)
    m = build_model(dims, sd)
    lib = _lib.load()
    d = m._rt.make_dims(xg, m.kernel_path)[0]
    d.path = _lib.PASN_PATH_TCGEN05
    assert not lib.pasn_tcgen05_supported(C.byref(d))                    # not a fused shape: the tiled chain serves it
    assert lib.pasn_head_workspace_bytes(C.byref(m._rt.make_dims(xg, m.kernel_path)[0])) > 0
    if cfg == "cfg5_scaled":
        import os
        torch.set_num_threads(os.cpu_count() or 1)
    _check_head(m, xg, x_ref, sd, pchunk=cfg == "cfg5_scaled")


def _run_gemm(g):
    lib = _lib.load()
    _lib.check(lib.pasn_debug_tc_gemm(C.byref(g), C.sizeof(Gemm), torch.cuda.current_stream().cuda_stream), "tc_gemm")
    torch.cuda.synchronize()
    assert lib.pasn_debug_fault() == 0


def _eleven_bits(shape, seed):
    """values with 11 significant bits (exact in fp16, not in bf16)"""
    gen = torch.Generator(device="cuda").manual_seed(seed)
    return torch.randn(shape, device="cuda", generator=gen).half()


@pytest.mark.parametrize("pair", [0, 1])
def test_tc_gemm_fp16_operands_reach_fp32_accumulation(pair):
    """ab_f16: both operands fp16, one pass, fp32 output; against float64.  A bf16 pass would miss by ~4e-3 of scale."""
    M, N, K = 640, 256, 512
    A, B = _eleven_bits((M, K), 1), _eleven_bits((N, K), 2)
    o32 = torch.zeros((M, N), device="cuda")
    g = Gemm()
    g.A, g.lda, g.ka = A.data_ptr(), K, K
    g.B, g.ldb, g.kb = B.data_ptr(), K, K
    g.M, g.N, g.K, g.batch, g.npass, g.bn, g.pair, g.ab_f16 = M, N, K, 1, 1, 256, pair, 1
    g.out[0] = Output(o32.data_ptr(), 3, N, 0, 0, 0, 0, 0)
    _run_gemm(g)
    ref = A.double() @ B.double().T
    err = float((o32.double() - ref).abs().max()) / float(ref.abs().max())
    assert err <= 2e-6, err
    bf = (A.bfloat16().double() @ B.bfloat16().double().T)
    assert float((bf - ref).abs().max()) / float(ref.abs().max()) > 1e-3   # (the case separates the two types)


@pytest.mark.parametrize("aligned", [True, False], ids=["tma", "plain"])
def test_tc_gemm_fp16_output_stores(aligned):
    """OUT_F16 through TMA stores (16-byte pitch) and plain stores (odd pitch), |.| epilogue; bf16 operands."""
    M, N, K = 300, 136 if aligned else 131, 128
    gen = torch.Generator(device="cuda").manual_seed(3)
    A = torch.randn((M, K), device="cuda", generator=gen).bfloat16()
    B = torch.randn((N, K), device="cuda", generator=gen).bfloat16()
    out = torch.full((M, N), 7.0, device="cuda", dtype=torch.float16)
    g = Gemm()
    g.A, g.lda, g.ka = A.data_ptr(), K, K
    g.B, g.ldb, g.kb = B.data_ptr(), K, K
    g.M, g.N, g.K, g.batch, g.npass, g.bn, g.act = M, N, K, 1, 1, 256, 2
    g.out[0] = Output(out.data_ptr(), OUT_F16, N, 0, 0, 0, 0, 0)
    _run_gemm(g)
    ref = (A.double() @ B.double().T).abs()
    assert torch.equal(out, ref.float().half()) or float((out.double() - ref).abs().max()) <= 1e-3 * float(ref.max())


def test_tc_gemm_refuses_fp16_with_several_passes():
    A = torch.zeros((128, 128), device="cuda", dtype=torch.float16)
    g = Gemm()
    g.A, g.lda, g.ka, g.B, g.ldb, g.kb = A.data_ptr(), 128, 128, A.data_ptr(), 128, 128
    g.M, g.N, g.K, g.batch, g.npass, g.bn, g.ab_f16 = 128, 128, 64, 1, 2, 128, 1
    g.out[0] = Output(A.data_ptr(), OUT_F16, 128, 0, 0, 0, 0, 0)
    assert _lib.load().pasn_debug_tc_gemm(C.byref(g), C.sizeof(Gemm), torch.cuda.current_stream().cuda_stream) == -1


@pytest.mark.parametrize("cfg,n,chunk", [("cfg3_video_b1024", 2048, 512), ("cfg2_image", 120, 50)])
def test_push_on_fp16_maps_matches_oracle(cfg, n, chunk):
    dims = synth.CONFIGS[cfg]
    sd = synth.make_head_params(dims, seed=77, bias_scale=0.05, bf16_round=True)
    xg, x_ref = _f16_input(dims, n, seed=13)
    labels = synth.push_labels(n, dims.K - 1, seed=3)
    m = build_model(dims, sd)
    res = pushmod.push_resident(m, xg, torch.from_numpy(labels).cuda(), chunk=chunk)
    new, ref_idx, ref_d = po.push_prototypes_oracle(x_ref, labels, sd, dims.K, batch=chunk, tie_rule="lowest")
    idx = res["index"].cpu().numpy()
    # margin between the winner and the runner-up of every prototype (class-restricted), next to the exact-index check
    with torch.no_grad():
        m2 = build_model(dims, sd)
        d_all = torch.cat([m2.push_forward(xg[i:i + chunk])[1] for i in range(0, n, chunk)]).cpu().numpy()
    pc = pushmod.proto_class_restriction(m2).numpy()
    keep = np.where((pc[None, :] < 0) | (labels[:, None] == pc[None, :]), d_all, np.inf)
    two = np.sort(keep, axis=0)[:2]
    print(f"fp16 push {cfg} n={n}: min top-2 margin {float((two[1] - two[0]).min()):.3e}, max |d - d_oracle| "
          f"{float(np.abs(res['distance'].cpu().numpy() - ref_d).max()):.3e}")
    assert np.array_equal(idx, ref_idx), np.nonzero(idx != ref_idx)
    assert_close(res["distance"], ref_d, BF16_RTOL, "winner distances", atol_frac=BF16_RTOL)
    assert_close(m.prototype_vectors.data, new, 4e-3, "pushed prototype_vectors", atol_frac=1e-3)


@pytest.mark.parametrize("layout", ["ncs", "nsc"])
def test_backward_with_fp16_features(layout):
    dims = synth.CONFIGS["cfg3_video_b1024"]
    n = 6
    sd = synth.make_head_params(dims, seed=17, bias_scale=0.1, last_layer_noise=0.2)
    xg, x_ref = _f16_input(dims, n, seed=6)
    if layout == "nsc":
        xg = xg.contiguous(memory_format=torch.channels_last_3d)
    rng = np.random.default_rng(3)
    wl = rng.standard_normal((n, dims.K)).astype(np.float32)
    ws = rng.standard_normal((n, dims.P)).astype(np.float32)
    # (the map is fp16, so its upstream gradient arrives rounded to fp16: the oracle gets the same values)
    wo = (rng.standard_normal((n, dims.P, 1) + dims.spatial) * 0.1).astype(np.float16).astype(np.float32)
    ref_loss, ref_gx, ref_g = _oracle_grads(x_ref, sd, wl, ws, wo)
    m = build_model(dims, sd)
    m.autograd_mode = "kernel"
    xt = xg.clone().requires_grad_(True)
    logits, sim, occ = m(xt)
    assert occ.dtype == torch.float16
    # the loss is formed in fp32 from the head's outputs (the fp16 map is bf16-grade, its gradient input is fp32)
    loss = (logits * torch.from_numpy(wl).cuda()).sum() + (sim * torch.from_numpy(ws).cuda()).sum() + \
        (occ.float() * torch.from_numpy(wo).cuda()).sum()
    loss.backward()
    assert xt.grad.dtype == torch.float16
    assert_close(xt.grad, ref_gx, 1e-3, "grad feature map", atol_frac=1e-4)
    own = dict(m.named_parameters())
    for k in KEYS:
        assert_close(own[k].grad.reshape(ref_g[k].shape), ref_g[k], 1e-3, f"grad {k}", atol_frac=1e-4)
    # compute_occurence_map backward alone
    for p in m.parameters():
        p.grad = None
    xo = xg.clone().requires_grad_(True)
    o = m.compute_occurence_map(xo)
    (o.float() * torch.from_numpy(wo).cuda()).sum().backward()
    _, ref_gx2, ref_g2 = _oracle_grads(x_ref, sd, np.zeros_like(wl), np.zeros_like(ws), wo)
    assert xo.grad.dtype == torch.float16
    assert_close(xo.grad, ref_gx2, 1e-3, "occ-only grad feature map", atol_frac=1e-4)
    for k in KEYS[4:9]:
        assert_close(own[k].grad.reshape(ref_g2[k].shape), ref_g2[k], 1e-3, f"occ-only grad {k}", atol_frac=1e-4)


class _Stub(torch.nn.Module):
    """Conv3d + ReLU backbone stub with C = 512 output channels."""

    def __init__(self):
        super().__init__()
        self.conv = torch.nn.Conv3d(8, 512, kernel_size=1)
        self.out_channels = 512

    def forward(self, x):
        self.last = torch.relu(self.conv(x))   # kept for the oracle
        return self.last


def test_end_to_end_under_autocast():
    torch.manual_seed(0)
    dims = synth.CONFIGS["cfg3_video_b1024"]
    sd = synth.make_head_params(dims, seed=9, bias_scale=0.05, last_layer_noise=0.2, bf16_round=True)
    m = pasn.construct_Video_XProtoNet(_Stub(), pretrained=False, prototype_shape=dims.prototype_shape, num_classes=dims.K)
    m.load_state_dict({**{k: torch.from_numpy(v) for k, v in sd.items()},
                       **{"cnn_backbone." + k: v for k, v in m.cnn_backbone.state_dict().items()}})
    m = m.cuda()
    inp = torch.randn((4, 8) + dims.spatial, device="cuda")
    with torch.no_grad(), torch.autocast("cuda", dtype=torch.float16):
        logits, sim, occ = m(inp)
        feat = m.cnn_backbone.last
    assert feat.dtype == torch.float16 and occ.dtype == torch.float16
    with torch.no_grad():
        rf, rd, ro, rl = ho.push_forward_torch(feat.float().cpu(), ho.to_torch_sd(sd))
    assert_close(logits, rl.numpy(), BF16_RTOL, "logits")
    assert_close(sim, (1 - rd).numpy(), BF16_RTOL, "similarity")
    assert_close(occ, ro.numpy(), 2e-2, "occurrence_map", atol_frac=1e-2)
    # one training step with a GradScaler, head gradients through the library
    m.train()
    m.autograd_mode = "kernel"
    scaler = torch.amp.GradScaler("cuda")
    with torch.autocast("cuda", dtype=torch.float16):
        logits, sim, occ = m(inp)
        feat = m.cnn_backbone.last
        loss = logits.float().logsumexp(1).sum() + sim.float().sum() * 0.1
    scaler.scale(loss).backward()
    scale = float(scaler.get_scale())
    grads = {k: p.grad.detach().double() / scale for k, p in m.named_parameters() if not k.startswith("cnn_backbone") and p.grad is not None}
    for g in grads.values():
        assert torch.isfinite(g).all()
    x_ref = feat.detach().float().cpu()
    sdt = {k: torch.from_numpy(np.ascontiguousarray(v)).double().requires_grad_(k != "ones") for k, v in sd.items()}
    _, dist, _, lg = ho.push_forward_torch(x_ref.double(), sdt)
    (lg.logsumexp(1).sum() + (1 - dist).sum() * 0.1).backward()
    for k in ("add_on_layers.0.weight", "occurrence_module.0.weight", "prototype_vectors", "last_layer.weight"):
        assert_close(grads[k].reshape(sdt[k].shape).float().cpu(), sdt[k].grad.numpy(), 1e-3, f"grad {k}", atol_frac=1e-4)


def test_lnorm_and_host_pipeline_on_fp16():
    from protoasnet_b200.metrics import L_norm
    dims = synth.CONFIGS["cfg3_video_b1024"]
    sd = synth.make_head_params(dims, seed=3, bias_scale=0.05, bf16_round=True)
    xg, _ = _f16_input(dims, 24, seed=8)
    m = build_model(dims, sd)
    with torch.no_grad():
        logits, sim, occ = m(xg)
    o64 = occ.double().reshape(occ.shape[0], occ.shape[1], -1)
    for p in (1, 2):
        got = float(L_norm(p=p, loss_weight=1.0).compute(occ, dim=(3, 4, 5)))
        ref = float(o64.abs().sum(-1).sum()) if p == 1 else float(o64.pow(2).sum(-1).sqrt().sum())
        assert abs(got - ref) <= 1e-5 * ref, (p, got, ref)
    host = xg.cpu().pin_memory()
    pipe = pasn.HostPipeline(m, chunks=3, want_occ=True)
    hl, hs, ho_ = pipe(host)
    assert torch.equal(hl, logits.cpu()) and torch.equal(hs, sim.cpu()) and torch.equal(ho_, occ.cpu())
