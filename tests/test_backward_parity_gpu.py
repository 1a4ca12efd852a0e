"""pasn_head_backward, called through the C ABI, against float64 autograd (tests/bwd_reference.py) over the shape
branches of both backward families: the tiled tensor-core chain (tiled.cu, three-pass bf16 hi|lo GEMMs) and the generic
CUDA-core kernels (generic.cu).

test_backward_gpu.py goes through autograd, which hands d(occurrence map) over rounded to the map's dtype and returns
the feature-map gradient in it; here the upstream gradients are exact fp32, the feature-map gradient comes back in fp32
for every map dtype, and NULL upstream pointers are reachable.  The inputs are conditioned (no pre-activation whose sign
the backward decides lies within 1e-4 of its magnitude sum of zero), so every gradient can be held to fp32-grade
agreement on any seed (PASN_BWD_PARITY_SEED selects the draw); clips whose pooled features are tiny against the
magnitudes they are summed from (the cosine's gradient scales with their inverse norm) are redrawn as well.

Every call also checks the ABI contract of include/pasn.h: the workspace is filled with 0xFF bytes (NaN) before the call,
the gradient buffers hold seeded values R that the gradients must be ADDED to, the buffers of the parameters outside the
occurrence branch stay bit-identical in occurrence-only mode, and grad_feat is channel-major whatever the map's layout."""
import ctypes as C
import functools
import json
import math
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import head_oracle as ho
from protoasnet_b200 import _lib, synth
from protoasnet_b200._lib import PasnDims, PasnGrads, PasnWeights
from tests.bwd_reference import (KEYS, OCC_KEYS, TAU, TAU_FE, condition_inputs, feature_norm_margins, reference_grads,
                                 round_to)
from tests.util import BWD_GENERIC_MAX, BWD_TILED_MAX, FP32_RTOL, assert_close, build_model

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

TILED, GENERIC = _lib.PASN_PATH_TILED, _lib.PASN_PATH_GENERIC
SEED = int(os.environ.get("PASN_BWD_PARITY_SEED", "0"))
# feature map kinds: (dtype name, channels_last)
KINDS = {"bf16": ("bf16", False), "bf16_cl": ("bf16", True), "fp16": ("fp16", False), "fp16_cl": ("fp16", True),
         "fp32": ("fp32", False), "fp32_cl": ("fp32", True), "fp32_degenerate": ("fp32", False)}
TORCH_DT = {"fp32": torch.float32, "bf16": torch.bfloat16, "fp16": torch.float16}

# (path, C, D, P, K, spatial, N, kind)
CASES = [
    # ---- tiled tensor-core backward
    (TILED, 64, 128, 9, 3, (7, 7), 5, "bf16"),            # P % 8 != 0 (Pp = 16), small-clip token kernel, D/2 = 64, one part
    (TILED, 192, 128, 8, 2, (2, 10, 12), 7, "fp32"),      # fp32 hi|lo transposition, C = 192
    (TILED, 128, 128, 20, 4, (2, 5, 13), 3, "fp16"),      # fp16 split, S = 130 (unaligned rows)
    (TILED, 64, 256, 12, 4, (4, 6, 6), 4, "fp16_cl"),     # NSC split kernel; grad_feat channel-major from channels_last
    (TILED, 512, 256, 40, 4, (4, 7, 7), 5, "bf16_cl"),    # cfg 3, channels_last read in place
    (TILED, 512, 512, 40, 4, (7, 7), 70, "bf16"),         # nb >= 64: 16 clip slices with atomics in proto_bwd_reduce
    (TILED, 64, 128, 130, 5, (3, 3, 3), 2, "bf16"),       # P > 128: ragged 256-wide tile, Pp = 136
    (TILED, 64, 128, 4096, 4, (2, 2, 2), 5, "fp32"),      # N*P = 20480 > 148*16*8 rows: grid-stride proto_bwd_rows
    (TILED, 64, 128, 2304, 4, (4, 4, 4), 72, "bf16"),     # part-buffer cap of wgrad (gW5 is the largest), T = 4608
    (TILED, 64, 128, 1, 1, (1, 2, 4), 1, "bf16"),         # P = K = N = 1: every GEMM one ragged tile
    (TILED, 64, 128, 16, 300, (4, 4), 3, "bf16"),         # K > 256: last-layer rows beyond one block of threads
    (TILED, 64, 128, 12, 3, (5, 5), 4, "fp32_degenerate"),  # zero prototype, zero W5 row, zero (W1 row, b1 entry)
    (TILED, 64, 128, 8, 2, (1, 1), 70000, "bf16"),        # more than 65535 clips per chunk
    # ---- generic CUDA-core backward
    (GENERIC, 40, 24, 12, 3, (3, 5, 2), 3, "fp32"),       # ragged 64 x 64 x 16 FFMA tiles
    (GENERIC, 40, 24, 12, 3, (3, 5, 2), 3, "bf16_cl"),    # bf16 B operand with channels_last strides
    (GENERIC, 64, 128, 9, 3, (7, 7), 5, "bf16"),          # the first tiled case's inputs: the two families agree
    (GENERIC, 64, 128, 2048, 300, (4, 7, 7), 55, "fp32"),  # two chunks of the backward (52 + 3 clips), K > 256
    (GENERIC, 20, 12, 8, 4, (1, 1), 70000, "fp32"),       # more than 65535 clips per chunk (launch_gemm's z)
]

# upstream gradients handed over: (logits, similarity, occurrence map, feature-map gradient wanted)
COMBOS = {"all": (1, 1, 1, 1), "logits": (1, 0, 0, 1), "sim": (0, 1, 0, 1), "no_occ": (1, 1, 0, 1),
          "occ_only": (0, 0, 1, 1), "none": (0, 0, 0, 1), "no_gx": (1, 1, 1, 0)}
COMBO_CASES = [(TILED, 128, 128, 20, 4, (2, 5, 13), 3, "fp32"), (GENERIC, 40, 24, 12, 3, (3, 5, 2), 3, "fp32")]
# (case, combo) pairs of the sweep: every case with all three gradients, the combinations on one shape per family, and
# occurrence-only on the > 65535-clip shapes
RUNS = [(c, "all") for c in CASES] + [(c, k) for c in COMBO_CASES for k in COMBOS if k != "all"] + \
    [(c, "occ_only") for c in CASES if c[6] == 70000]
# backward chunks: PASN_TILED_CHUNK = 3 splits 7 clips into 3 + 3 + 1 (the variable is read once per process)
CHUNKED_CASE = (TILED, 128, 128, 20, 4, (7, 7), 7, "fp32")


def case_id(c, combo="all"):
    fam = "tiled" if c[0] == TILED else "generic"
    return f"{fam}-C{c[1]}-D{c[2]}-P{c[3]}-K{c[4]}-S{math.prod(c[5])}-N{c[6]}-{c[7]}-{combo}"


def make_params(dims: synth.HeadDims, degenerate: bool):
    """Head parameters (fp32, not bf16-rounded: the backward uses the weights unrounded); the last layer is drawn for any
    K.  degenerate: prototype 0 is zero, W5 row 1 is zero (O[1] = 0, features_extracted[:, 1] = 0: both cosine norms
    clamped somewhere) and (W1 row 2, b1[2]) are zero (H1[2] = 0 everywhere)."""
    sd = synth.make_head_params(synth.HeadDims(dims.C, dims.D, dims.P, 1, dims.spatial), seed=41, bias_scale=0.05)
    rng = np.random.default_rng(42)
    sd["last_layer.weight"] = (rng.standard_normal((dims.K, dims.P)) * 0.5).astype(np.float32)
    if degenerate:
        sd["prototype_vectors"][0] = 0
        sd["occurrence_module.4.weight"][1] = 0
        sd["add_on_layers.0.weight"][2] = 0
        sd["add_on_layers.0.bias"][2] = 0
    return sd


@functools.lru_cache(maxsize=4)
def prepare(case, combo="all", seed=SEED):
    """CPU side of a run: conditioned inputs, upstream gradients, the float64 reference and the seeded buffer contents R."""
    path, Cc, D, P, K, spatial, N, kind = case
    dtn, _ = KINDS[kind]
    dims = synth.HeadDims(Cc, D, P, K, spatial)
    S = dims.S
    sd = make_params(dims, kind.endswith("degenerate"))
    x = round_to(synth.make_features(dims, N, seed=100 + seed), dtn)
    x, margin, rounds = condition_inputs(x, sd, dtn, TAU, seed=seed)
    fe_margin = float(feature_norm_margins(x, sd).min())
    use_l, use_s, use_o, want_gx = COMBOS[combo]
    rng = np.random.default_rng(1000 + seed)
    wl = rng.standard_normal((N, K)).astype(np.float32) if use_l else None
    ws = rng.standard_normal((N, P)).astype(np.float32) if use_s else None
    wo = (rng.standard_normal((N, P, S)) * 0.1).astype(np.float32) if use_o else None
    gx_ref, g_ref = reference_grads(x, sd, wl, ws, wo)
    R = {}
    for k in KEYS:   # at the scale of each row of the gradient (a zero prototype's row is 1e7 times the others)
        g = g_ref[k].reshape(g_ref[k].shape[0], -1)
        scale = np.abs(g).max(axis=1, keepdims=True)
        scale = np.where(scale > 0, scale, float(np.abs(g).max()) or 1.0)
        R[k] = (rng.uniform(-1.0, 1.0, g.shape) * scale).astype(np.float32).reshape(g_ref[k].shape)
    return dict(dims=dims, sd=sd, x=x, margin=margin, fe_margin=fe_margin, rounds=rounds, wl=wl, ws=ws, wo=wo, want_gx=bool(want_gx),
                gx_ref=gx_ref, g_ref=g_ref, R=R)


def call_backward(case, prep):
    """pasn_head_backward on the device: returns (grad_feat [N, C, S] fp32 or None, {key: gradient buffer after the call})."""
    path, Cc, D, P, K, spatial, N, kind = case
    dtn, cl = KINDS[kind]
    dims, S = prep["dims"], prep["dims"].S
    lib = _lib.load()
    x = torch.from_numpy(prep["x"]).to(TORCH_DT[dtn]).cuda()
    if cl:
        x = x.contiguous(memory_format=torch.channels_last_3d if dims.ndim == 3 else torch.channels_last)
    d = PasnDims(N, Cc, D, P, K, S, _lib.DTYPES[x.dtype], _lib.PASN_LAYOUT_NSC if cl else _lib.PASN_LAYOUT_NCS,
                 _lib.PASN_OCC_ABS, path)
    # the family is the one asked for: a shape that fell back to the other one fails here
    assert lib.pasn_tcgen05_supported(C.byref(d)) == (1 if path == TILED else 0), case
    params = [torch.from_numpy(np.ascontiguousarray(prep["sd"][k])).cuda() for k in KEYS]
    grads = [torch.from_numpy(prep["R"][k]).cuda() for k in KEYS]
    w, gw = PasnWeights(*[t.data_ptr() for t in params]), PasnGrads(*[t.data_ptr() for t in grads])
    up = [None if prep[k] is None else torch.from_numpy(prep[k]).cuda() for k in ("wl", "ws", "wo")]
    gx = torch.full((N, Cc, S), float("nan"), device="cuda") if prep["want_gx"] else None
    need = int(lib.pasn_head_backward_workspace_bytes(C.byref(d)))
    assert need > 0
    ws = torch.full((need,), 0xFF, dtype=torch.uint8, device="cuda")   # NaN in fp32 and bf16: unwritten scratch shows
    ptr = lambda t: None if t is None else t.data_ptr()                  # noqa: E731
    stream = torch.cuda.current_stream().cuda_stream
    st = lib.pasn_head_backward(x.data_ptr(), C.byref(w), C.byref(d), ptr(up[0]), ptr(up[1]), ptr(up[2]), C.byref(gw),
                                ptr(gx), ws.data_ptr(), ws.numel(), stream)
    _lib.check(st, "pasn_head_backward")
    torch.cuda.synchronize()
    return (None if gx is None else gx.cpu().numpy()), {k: g.cpu().numpy() for k, g in zip(KEYS, grads)}


def deviation(got, ref):
    """(max |got - ref| / max |ref|, ||got - ref|| / ||ref||), float64; an all-zero reference wants an exact zero."""
    diff = np.asarray(got, np.float64) - ref
    scale = float(np.abs(ref).max())
    if scale == 0.0:
        return (0.0, 0.0) if not diff.any() else (math.inf, math.inf)
    return float(np.abs(diff).max() / scale), float(np.linalg.norm(diff) / np.linalg.norm(ref))


def run_case(case, combo="all", seed=SEED):
    """One backward call against the reference: the deviation of every gradient (what the sweep asserts and
    tools/bwd_parity_report.py prints), the conditioning margin, and the bit-identity of the untouched buffers."""
    prep = prepare(case, combo, seed)
    gx, got = call_backward(case, prep)
    r = {"margin": prep["margin"], "fe_margin": prep["fe_margin"], "rounds": prep["rounds"], "dev": {}, "norm": {}, "untouched": []}
    occ_only = combo in ("occ_only", "none")
    for k in KEYS:
        R = prep["R"][k]
        if occ_only and k not in OCC_KEYS or combo == "none":
            # the contract: these buffers are not written at all
            if not np.array_equal(got[k].view(np.uint32), R.view(np.uint32)):
                r["untouched"].append(k)
            continue
        r["dev"][k], r["norm"][k] = deviation(got[k].astype(np.float64) - R.astype(np.float64), prep["g_ref"][k])
    if gx is not None:
        r["dev"]["grad_feat"], r["norm"]["grad_feat"] = deviation(gx, prep["gx_ref"])
    return r


def threshold(case):
    return BWD_TILED_MAX if case[0] == TILED else BWD_GENERIC_MAX


def check(case, r):
    assert r["margin"] >= TAU and r["fe_margin"] >= TAU_FE, (r["margin"], r["fe_margin"])
    assert not r["untouched"], f"buffers written that the call must leave alone: {r['untouched']}"
    bad = {k: v for k, v in r["dev"].items() if not v <= threshold(case)}
    assert not bad, f"deviation from float64 above {threshold(case):g} of scale: {bad}"


@pytest.mark.parametrize("case,combo", RUNS, ids=[case_id(c, k) for c, k in RUNS])
def test_backward_matches_float64(case, combo):
    r = run_case(case, combo)
    check(case, r)
    if combo == "none":
        assert r["dev"]["grad_feat"] == 0.0   # no upstream gradient: grad_feat comes back as zeros


@pytest.mark.parametrize("case", [c for c in CASES if c[6] == 70000], ids=lambda c: case_id(c, "forward"))
def test_forward_past_65535_clips(case):
    """forward() and compute_occurence_map() at the shapes whose chunk would hold more than 65535 clips: bit-identical to
    two calls on the halves of the batch (every clip is computed on its own), and the generic fp32 path against the
    float64 oracle as well.  (The bf16 chain's own parity is test_tc_emulated_parity_gpu.py's; over 560 000 similarities
    its rare bf16 rounding flips exceed that file's per-case budgets.)"""
    path, Cc, D, P, K, spatial, N, kind = case
    dtn, _ = KINDS[kind]
    dims = synth.HeadDims(Cc, D, P, K, spatial)
    sd = make_params(dims, False)
    x = round_to(synth.make_features(dims, N, seed=5), dtn)
    m = build_model(dims, sd, path=path)
    xg = torch.from_numpy(x).to(TORCH_DT[dtn]).cuda()
    with torch.no_grad():
        whole = [t.float().cpu().numpy() for t in m(xg)] + [m.compute_occurence_map(xg).float().cpu().numpy()]
        halves = [[t.float().cpu().numpy() for t in m(h)] + [m.compute_occurence_map(h).float().cpu().numpy()]
                  for h in (xg[:N // 2], xg[N // 2:])]
    for name, w, h0, h1 in zip(("logits", "similarity", "occurrence_map", "compute_occurence_map"), whole, *halves):
        assert np.array_equal(w, np.concatenate([h0, h1])), name
    if dtn == "fp32":
        ref = ho.head_forward_f64(x, sd)
        assert_close(whole[0], ref["logits"], FP32_RTOL, "logits")
        assert_close(whole[1], ref["similarity"], FP32_RTOL, "similarity")
        for mp in whole[2:]:
            assert_close(mp.reshape(N, P, -1), ref["occurrence_map"], FP32_RTOL, "occurrence map")


CHUNK_SCRIPT = r"""
import json, sys
sys.path.insert(0, %r)
from protoasnet_b200 import _lib
_lib.LIB_PATH = %r
from tests import test_backward_parity_gpu as t
print(json.dumps({k: t.run_case(t.CHUNKED_CASE, k, %d) for k in ("all", "occ_only")}))
"""


def run_chunked(seed=SEED):
    """run_case of CHUNKED_CASE, full and occurrence-only, in a process with PASN_TILED_CHUNK = 3 (the same library
    build as this process): {combo: result}."""
    env = dict(os.environ, PASN_TILED_CHUNK="3")
    out = subprocess.run([sys.executable, "-c", CHUNK_SCRIPT % (ROOT, _lib.LIB_PATH, seed)], check=True, env=env, cwd=ROOT, timeout=600,
                         capture_output=True, text=True).stdout
    return json.loads(out.strip().splitlines()[-1])


def test_backward_chunks_match_float64():
    """Three backward chunks with a ragged last (PASN_TILED_CHUNK = 3), full and occurrence-only: gradients accumulate
    across chunks into the same buffers and must still meet the float64 reference."""
    for combo, r in run_chunked().items():
        check(CHUNKED_CASE, r)
