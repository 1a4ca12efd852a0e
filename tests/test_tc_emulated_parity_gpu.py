"""Tensor-core forward in bf16 / fp16 mode against oracle/emulate.py, a float64 model that rounds where the kernels round,
over the shape branches of the fused token / prototype kernel pair (head_sm100*.cu) and of the tiled GEMM chain
(tiled.cu).  The reference oracle rounds nowhere, so the tests against it need budgets (1e-3 on similarities) that a
kernel bug of the usual size fits inside; against the emulation only fp32 accumulation order is left, and the
thresholds (tests/util.py) are 10 to 100 times tighter.

Parameters are drawn without bf16 rounding, so the packing kernels' round-to-nearest is part of what is checked; the
kernel path is set explicitly, so a shape that silently fell back to another path fails."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

from oracle.emulate import cosine_chain_f64, head_forward_emulated
from protoasnet_b200 import _lib, synth
from tests.util import (EMU_COSINE_FWD, EMU_COSINE_PUSH, EMU_FEAT_POOL_FIRST, EMU_FEAT_W2_FIRST, EMU_LOGITS_FRAC,
                        EMU_OCC_BITEQ, EMU_OCC_BITEQ_F16, EMU_SIM_ATOL, build_model, occ_agreement)

pytestmark = pytest.mark.gpu

FUSED, TILED = _lib.PASN_PATH_TCGEN05, _lib.PASN_PATH_TILED
NUM_SMS = 148
# input kinds: dtype and memory layout of the feature map
KINDS = {"bf16": (torch.bfloat16, False), "bf16_cl": (torch.bfloat16, True), "fp16": (torch.float16, False),
         "fp16_cl": (torch.float16, True), "fp32_fused": (torch.float32, False)}

# (path, C, D, P, K, spatial, N, kind)
CASES = [
    # ---- fused K1 / K2 pair
    (FUSED, 64, 256, 1, 1, (2, 8, 8), 3, "bf16"),             # P = 1 -> PP = 16, K = 1, S = 128: tile == clip
    (FUSED, 128, 256, 16, 4, (3, 4, 11), 9, "bf16"),          # P = 16 (PP = 16, 8 clips per K2 tile), S = 132 straddles
    (FUSED, 64, 256, 17, 17, (1, 10, 14), 10, "bf16_cl"),     # P = 17 -> PP = 32, K = P, S = 140, channels_last
    (FUSED, 256, 256, 32, 4, (4, 7, 7), 12, "fp16"),          # P = 32 (PP = 32, 4 clips per K2 tile), fp16 NCDHW
    (FUSED, 128, 256, 33, 3, (1, 10, 14), 7, "fp16_cl"),      # P = 33 -> PP = 40, fp16 channels_last
    (FUSED, 512, 256, 40, 4, (4, 7, 7), 37, "bf16"),          # cfg 3 at PP = 40 (3 clips per K2 tile)
    (FUSED, 64, 256, 41, 41, (2, 8, 8), 11, "bf16"),          # P = 41 -> PP = 48, K = P
    (FUSED, 1024, 256, 48, 4, (3, 8, 8), 9, "bf16"),          # C = 1024 (16 channel chunks), P = 48, 2 clips per K2 tile
    (FUSED, 512, 256, 40, 4, (4, 7, 7), 148, "bf16"),         # one clip per CTA
    (FUSED, 512, 256, 40, 4, (4, 7, 7), 149, "fp16"),         # 2 clips per CTA, 75 CTAs
    (FUSED, 512, 256, 40, 4, (4, 7, 7), 296, "bf16_cl"),      # 2 clips per CTA, every CTA full
    (FUSED, 512, 256, 40, 4, (4, 7, 7), 297, "bf16"),         # 3 clips per CTA with a short last CTA
    (FUSED, 256, 256, 40, 4, (8, 14, 14), 1, "bf16"),         # cfg 1, voxel-group split G = 8
    (FUSED, 256, 256, 40, 4, (8, 14, 14), 5, "fp16"),         # split G = 8
    (FUSED, 256, 256, 40, 4, (8, 14, 14), 8, "bf16_cl"),      # split G = 8, channels_last
    (FUSED, 256, 256, 40, 4, (8, 14, 14), 74, "bf16"),        # last N that splits: G = 2
    (FUSED, 256, 256, 40, 4, (8, 14, 14), 75, "fp16"),        # first N that does not split
    (FUSED, 256, 256, 24, 4, (8, 8, 8), 37, "bf16"),          # S = 512: G = 4
    (FUSED, 256, 256, 24, 4, (8, 8, 8), 74, "fp16_cl"),       # S = 512: G = 2
    (FUSED, 256, 256, 24, 4, (4, 8, 8), 6, "fp32_fused"),     # fp32 map rounded on the fly, split G = 2
    (FUSED, 512, 256, 40, 4, (4, 7, 7), 149, "fp32_fused"),   # fp32 map, several clips per CTA
    (FUSED, 512, 256, 40, 4, (4, 7, 7), 9, "bf16_rounded"),   # bf16-exact parameters, as the older sweeps use them
    # ---- tiled GEMM chain
    (TILED, 64, 128, 9, 3, (7, 7), 5, "bf16"),                # P % 8 != 0, S = 49 >= 2P: pooling first; small-clip transposition
    (TILED, 192, 128, 8, 2, (2, 10, 12), 7, "bf16"),          # pooling first, O over all tokens + column sums; direct operand
    (TILED, 64, 128, 72, 4, (4, 16, 16), 2, "bf16"),          # pooling first, O per clip (P > 64) with rounded row sums
    (TILED, 64, 128, 72, 4, (4, 16, 16), 2, "fp16"),          # same in fp16: the map in fp16, the pooling on a bf16 copy
    (TILED, 128, 128, 20, 4, (2, 5, 13), 3, "bf16"),          # S = 130: unaligned rows, transposition kernel
    (TILED, 128, 128, 20, 4, (2, 5, 13), 3, "fp16"),          # fp16 transposition
    (TILED, 64, 256, 12, 4, (4, 6, 6), 4, "fp16_cl"),         # pooling first, fp16 channels_last
    (TILED, 512, 512, 40, 4, (7, 7), 5, "bf16_cl"),           # image head, W2 first, row statistics, no block diagonal (N < 2G)
    (TILED, 512, 512, 40, 4, (7, 7), 6, "bf16"),              # image head: three clips per 128-row tile, block-diagonally
    (TILED, 512, 512, 40, 4, (7, 7), 7, "fp16"),              # block-diagonal with a ragged last group
    (TILED, 128, 128, 33, 3, (1, 5, 10), 3, "bf16_cl"),       # W2 first, P just over 32, S = 50
    (TILED, 64, 256, 130, 5, (3, 3, 3), 2, "bf16"),           # P = 130: O per clip, no row statistics, S = 27
    (TILED, 64, 128, 100, 4, (8, 8), 3, "fp16"),              # W2 first, O per clip, fp16
    (TILED, 64, 128, 4096, 4, (4, 8, 8), 1, "bf16"),          # P = 4096 at N = 1: O per clip, row statistics
    (TILED, 128, 256, 40, 4, (1, 2, 4), 1, "bf16"),           # one clip of 8 voxels: every GEMM a single ragged tile
]


def _ids(c):
    return f"{'fused' if c[0] == FUSED else 'tiled'}-C{c[1]}-D{c[2]}-P{c[3]}-K{c[4]}-S{math.prod(c[5])}-N{c[6]}-{c[7]}"


def split_groups(N, S):
    """Voxel groups per clip of the fused pair (head_sm100.cu: split_groups)."""
    if N > 74:
        return 1
    best = 1
    for g in range(2, S // 128 + 1):
        if S % g or S // g < 128 or (S // g) % 4:
            continue
        if N * g > NUM_SMS:
            break
        best = g
    return best


def k2_ppad(P):
    p8 = (P + 7) // 8 * 8
    return 16 if p8 <= 16 else 32 if p8 <= 32 else 40 if p8 <= 40 else 48


def fused_clips(N, S, P):
    """Clips to emulate on a fused case with many clips: the first and the last, both sides of a K1 CTA range boundary
    and of a K2 tile boundary, and two clips that share a 128-voxel tile (head_sm100.cu: clips_per_cta, cpt)."""
    G = split_groups(N, S)
    Nv, Sv = N * G, S // G
    cpc = -(-Nv // NUM_SMS)
    cpt = 128 // k2_ppad(P)
    sel = {0, N - 1}
    if cpc < Nv:
        sel |= {(cpc - 1) // G, cpc // G}
    if cpt < Nv:
        b = (Nv // cpt // 2) * cpt or cpt
        sel |= {(b - 1) // G, b // G}
    for v in range(min(cpc, Nv) - 1):                   # virtual clips v, v + 1 of the first CTA share a tile
        if ((v + 1) * Sv) % 128:
            sel |= {v // G, (v + 1) // G}
            break
    return sorted(sel)


def _inputs(case):
    path, Cc, D, P, K, spatial, N, kind = case
    dims = synth.HeadDims(Cc, D, P, K, spatial)
    rounded = kind == "bf16_rounded"
    sd = synth.make_head_params(dims, seed=41, bias_scale=0.05, last_layer_noise=0.1, bf16_round=rounded)
    dtype, cl = KINDS["bf16" if rounded else kind]
    x = torch.from_numpy(synth.make_features(dims, N, seed=23)).to(dtype)
    xg = x.cuda()
    if cl:
        xg = xg.contiguous(memory_format=torch.channels_last_3d if dims.ndim == 3 else torch.channels_last)
    return dims, sd, x.float().numpy(), xg


def run_case(case):
    """Runs one case, asserts the branch and the output types, returns the measured deviations from the emulation."""
    path, Cc, D, P, K, spatial, N, kind = case
    dims, sd, x, xg = _inputs(case)
    S = dims.S
    m = build_model(dims, sd, path=path)
    lib = _lib.load()
    cd = m._rt.make_dims(xg, path)[0]
    assert lib.pasn_tcgen05_supported(C.byref(cd))
    with torch.no_grad():
        logits, sim, occ = m(xg)
        torch.cuda.synchronize()
        c0 = lib.pasn_debug_launch_count()
        logits, sim, occ = m(xg)
        torch.cuda.synchronize()
        launched = lib.pasn_debug_launch_count() - c0
        feats, dist, occ2, logits2 = m.push_forward(xg)
        occ3 = m.compute_occurence_map(xg)
    if path == FUSED:
        order = "pool_first"
        G = split_groups(N, S)
        assert (launched == 2) == (G == 1), (launched, G)   # the pair alone, or the split's sum and prototype stage after it
    else:
        order = "w2_first" if S < 2 * P else "pool_first"
    sel = fused_clips(N, S, P) if path == FUSED and N > 8 else list(range(N))
    mode = "fp32_fused" if kind == "fp32_fused" else "fp16" if xg.dtype == torch.float16 else "bf16"
    for o in (occ, occ2, occ3):
        assert o.dtype == xg.dtype and tuple(o.shape) == (N, P, 1) + tuple(spatial)
    assert logits.dtype == sim.dtype == feats.dtype == dist.dtype == torch.float32
    got = {k: v.float().cpu().numpy()[sel] for k, v in dict(logits=logits, similarity=sim, distance=dist, feats=feats,
                                                             logits2=logits2).items()}
    maps = [o.float().cpu().numpy()[sel].reshape(len(sel), P, S) for o in (occ, occ2, occ3)]
    xs = x[sel]
    emu = head_forward_emulated(xs, sd, mode, order)
    if mode == "fp16":
        want = emu["occurrence_abs"] if path == TILED else emu["occurrence_map"]   # tiled: fp16(|.|); fused: fp16(bf16)
        want_map = torch.from_numpy(want).half().double().numpy()
        ref = emu   # the fp16 map is not the pooling operand
    else:
        want_map = emu["occurrence_map"]
        ref = head_forward_emulated(xs, sd, mode, order, occ=maps[1])
    r = {"order": order, "biteq_min": EMU_OCC_BITEQ_F16 if mode == "fp16" and path == TILED else EMU_OCC_BITEQ}
    agree = [occ_agreement(mp, want_map) for mp in maps]
    r["occ_biteq_min"] = min(a[0] for a in agree)
    r["occ_worst"] = max(a[1] for a in agree)
    fe_ref = ref["features_extracted"]
    r["feat"] = float(np.abs(got["feats"] - fe_ref).max() / np.abs(fe_ref).max())
    r["sim"] = float(max(np.abs(got["similarity"] - ref["similarity"]).max(), np.abs(got["distance"] - ref["distance"]).max()))
    r["logits"] = float(np.abs(got["logits2"] - ref["logits"]).max() / np.abs(ref["logits"]).max())
    cc = cosine_chain_f64(got["feats"], sd)
    lscale = np.abs(cc["logits"]).max()
    r["cos_push"] = float(max(np.abs(got["distance"] - cc["distance"]).max(), np.abs(got["logits2"] - cc["logits"]).max() / lscale))
    r["cos_fwd"] = float(max(np.abs(got["similarity"] - cc["similarity"]).max(), np.abs(got["logits"] - cc["logits"]).max() / lscale))
    return r


def check(r):
    feat_tol = EMU_FEAT_POOL_FIRST if r["order"] == "pool_first" else EMU_FEAT_W2_FIRST
    assert r["occ_biteq_min"] >= r["biteq_min"] and r["occ_worst"] <= 1.0, r
    assert r["feat"] <= feat_tol, r
    assert r["sim"] <= EMU_SIM_ATOL, r
    assert r["logits"] <= EMU_LOGITS_FRAC, r
    assert r["cos_push"] <= EMU_COSINE_PUSH, r
    assert r["cos_fwd"] <= EMU_COSINE_FWD, r


@pytest.mark.parametrize("case", CASES, ids=[_ids(c) for c in CASES])
def test_forward_matches_emulation(case):
    check(run_case(case))
