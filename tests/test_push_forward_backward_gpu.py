"""Training through push_forward and get_occurence_map_absolute_val on the library.

pasn_head_backward_ex takes the upstream gradient of every head output, d(features_extracted) and d(distance) included.
It is called through the C ABI on both backward families and checked against float64 autograd through push_forward's op
sequence (oracle/head_oracle.py). The checks are those of test_backward_parity_gpu.py: conditioned inputs, exact fp32
upstream gradients, a NaN-filled workspace, gradients added to seeded buffers and a channel-major fp32 grad_feat.
pasn_head_backward must equal the new call with distance and features NULL, bit for bit. A distance gradient g must equal
a similarity gradient -g. At module level, push_forward and get_occurence_map_absolute_val under
autograd_mode='kernel' must be served by the library."""
import ctypes as C
import functools
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import head_oracle as ho
from protoasnet_b200 import _lib, synth
from protoasnet_b200._lib import PasnDims, PasnGrads, PasnUpstream, PasnWeights
from tests.bwd_reference import KEYS, TAU, condition_inputs, round_to
from tests.test_backward_parity_gpu import GENERIC, KINDS, TILED, TORCH_DT, case_id, deviation, make_params
from tests.util import BWD_GENERIC_MAX, BWD_TILED_MAX, assert_close, build_model

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SEED = int(os.environ.get("PASN_BWD_PARITY_SEED", "0"))

# head outputs in pasn_upstream's field order
OUTPUTS = ("logits", "similarity", "distance", "occurrence_map", "features_extracted")
FIELDS = dict(zip(OUTPUTS, (f for f, _ in PasnUpstream._fields_)))

# (path, C, D, P, K, spatial, N, kind): a subset of test_backward_parity_gpu.CASES
CASES = [
    (TILED, 64, 128, 9, 3, (7, 7), 5, "bf16"),            # P % 8 != 0; T = 245 tokens: one colsum block, no atomics race
    (TILED, 192, 128, 8, 2, (2, 10, 12), 7, "fp32"),      # fp32 hi|lo
    (TILED, 64, 256, 12, 4, (4, 6, 6), 4, "fp16_cl"),     # fp16 map, channels_last
    (TILED, 64, 128, 130, 5, (3, 3, 3), 2, "bf16"),       # P > 128: ragged 256-wide tile
    (TILED, 64, 128, 16, 300, (4, 4), 3, "bf16"),         # K > 256
    (GENERIC, 40, 24, 12, 3, (3, 5, 2), 3, "fp32"),
    (GENERIC, 40, 24, 12, 3, (3, 5, 2), 3, "bf16_cl"),
    (GENERIC, 20, 12, 8, 4, (1, 1), 70000, "fp32"),       # two chunks of the generic backward (65535 + 4465 clips)
]
# upstream gradients handed over per combination
COMBOS = {"all": OUTPUTS, "features": ("features_extracted",), "distance": ("distance",),
          # no logits / similarity gradient, yet the full chain must run (occurrence-only mode would drop the features')
          "features_occ": ("features_extracted", "occurrence_map")}
COMBO_CASES = [CASES[0], CASES[5]]
RUNS = [(c, "all") for c in CASES] + [(c, k) for c in COMBO_CASES for k in COMBOS if k != "all"]
# deterministic shapes (no atomics whose order could differ between two calls): bit-identity checks
EXACT_CASES = [CASES[0], CASES[5]]
# backward chunks: PASN_TILED_CHUNK = 3 splits 7 clips into 3 + 3 + 1
CHUNKED_CASE = (TILED, 128, 128, 20, 4, (7, 7), 7, "fp32")


def push_reference_grads(x, sd, up):
    """float64 d(loss)/d(x) as [N, C, S] and d(loss)/d(parameter) for the eleven KEYS, where
    loss = sum over the outputs named in ``up`` of (output * up[name]), the outputs being those of
    oracle.head_oracle.push_forward_torch (similarity = 1 - distance)."""
    sdt = {k: torch.from_numpy(np.ascontiguousarray(sd[k])).double().requires_grad_(True) for k in KEYS}
    xt = torch.from_numpy(np.ascontiguousarray(x)).double().requires_grad_(True)
    feats, dist, occ, logits = ho.push_forward_torch(xt, sdt)
    outs = {"logits": logits, "similarity": 1 - dist, "distance": dist, "occurrence_map": occ, "features_extracted": feats}
    loss = sum((outs[k] * torch.from_numpy(w).double().reshape(outs[k].shape)).sum() for k, w in up.items())
    gx, *gp = torch.autograd.grad(loss, [xt] + [sdt[k] for k in KEYS], allow_unused=True)
    gx = gx.reshape(x.shape[0], x.shape[1], -1).numpy()
    return gx, {k: (np.zeros(sd[k].shape) if g is None else g.numpy()) for k, g in zip(KEYS, gp)}


@functools.lru_cache(maxsize=4)
def prepare(case, combo="all", seed=SEED):
    """CPU side of a run: conditioned inputs, upstream gradients, the float64 reference and the seeded buffer contents R."""
    path, Cc, D, P, K, spatial, N, kind = case
    dtn, _ = KINDS[kind]
    dims = synth.HeadDims(Cc, D, P, K, spatial)
    S = dims.S
    sd = make_params(dims, False)
    x = round_to(synth.make_features(dims, N, seed=100 + seed), dtn)
    x, margin, _ = condition_inputs(x, sd, dtn, TAU, seed=seed)
    fe = np.linalg.norm(ho.head_forward_f64(x, sd)["features_extracted"], axis=2)
    rng = np.random.default_rng(2000 + seed)
    draw = {"logits": lambda: rng.standard_normal((N, K)), "similarity": lambda: rng.standard_normal((N, P)),
            "distance": lambda: rng.standard_normal((N, P)), "occurrence_map": lambda: rng.standard_normal((N, P, S)) * 0.1,
            # at the scale of the cosine's own gradient of the pooled features (1 / |FE|): neither term hides the other
            "features_extracted": lambda: rng.standard_normal((N, P, D)) / np.where(fe > 0, fe, 1.0)[:, :, None]}
    up = {k: draw[k]().astype(np.float32) for k in COMBOS[combo]}
    gx_ref, g_ref = push_reference_grads(x, sd, up)
    R = {}
    for k in KEYS:   # at the scale of each row of the gradient
        g = g_ref[k].reshape(g_ref[k].shape[0], -1)
        scale = np.abs(g).max(axis=1, keepdims=True)
        scale = np.where(scale > 0, scale, float(np.abs(g).max()) or 1.0)
        R[k] = (rng.uniform(-1.0, 1.0, g.shape) * scale).astype(np.float32).reshape(g_ref[k].shape)
    return dict(dims=dims, sd=sd, x=x, margin=margin, up=up, gx_ref=gx_ref, g_ref=g_ref, R=R)


def call_backward(case, prep, up, legacy=False):
    """pasn_head_backward_ex (legacy: pasn_head_backward, which has no distance / features gradient) with the upstream
    gradients ``up`` {output name: fp32 array}: returns (grad_feat [N, C, S] fp32, {key: gradient buffer after the call})."""
    path, Cc, D, P, K, spatial, N, kind = case
    dtn, cl = KINDS[kind]
    dims, S = prep["dims"], prep["dims"].S
    lib = _lib.load()
    x = torch.from_numpy(prep["x"]).to(TORCH_DT[dtn]).cuda()
    if cl:
        x = x.contiguous(memory_format=torch.channels_last_3d if dims.ndim == 3 else torch.channels_last)
    d = PasnDims(N, Cc, D, P, K, S, _lib.DTYPES[x.dtype], _lib.PASN_LAYOUT_NSC if cl else _lib.PASN_LAYOUT_NCS,
                 _lib.PASN_OCC_ABS, path)
    assert lib.pasn_tcgen05_supported(C.byref(d)) == (1 if path == TILED else 0), case
    params = [torch.from_numpy(np.ascontiguousarray(prep["sd"][k])).cuda() for k in KEYS]
    grads = [torch.from_numpy(prep["R"][k]).cuda() for k in KEYS]
    w, gw = PasnWeights(*[t.data_ptr() for t in params]), PasnGrads(*[t.data_ptr() for t in grads])
    ups = {k: torch.from_numpy(v).cuda() for k, v in up.items()}
    gx = torch.full((N, Cc, S), float("nan"), device="cuda")
    need = int(lib.pasn_head_backward_workspace_bytes(C.byref(d)))
    assert need > 0
    ws = torch.full((need,), 0xFF, dtype=torch.uint8, device="cuda")   # NaN in fp32 and bf16: unwritten scratch shows
    ptr = lambda name: ups[name].data_ptr() if name in ups else None    # noqa: E731
    stream = torch.cuda.current_stream().cuda_stream
    if legacy:
        assert not {"distance", "features_extracted"} & set(up)
        st = lib.pasn_head_backward(x.data_ptr(), C.byref(w), C.byref(d), ptr("logits"), ptr("similarity"),
                                    ptr("occurrence_map"), C.byref(gw), gx.data_ptr(), ws.data_ptr(), ws.numel(), stream)
    else:
        u = PasnUpstream(**{FIELDS[k]: ptr(k) for k in OUTPUTS})
        st = lib.pasn_head_backward_ex(x.data_ptr(), C.byref(w), C.byref(d), C.byref(u), C.byref(gw), gx.data_ptr(),
                                       ws.data_ptr(), ws.numel(), stream)
    _lib.check(st, "pasn_head_backward_ex")
    torch.cuda.synchronize()
    return gx.cpu().numpy(), {k: g.cpu().numpy() for k, g in zip(KEYS, grads)}


def run_case(case, combo="all", seed=SEED):
    """One pasn_head_backward_ex call against the float64 reference: the deviation of every gradient."""
    prep = prepare(case, combo, seed)
    gx, got = call_backward(case, prep, prep["up"])
    dev = {k: deviation(got[k].astype(np.float64) - prep["R"][k].astype(np.float64), prep["g_ref"][k])[0] for k in KEYS}
    dev["grad_feat"] = deviation(gx, prep["gx_ref"])[0]
    return {"margin": prep["margin"], "dev": dev}


def check(case, r):
    assert r["margin"] >= TAU, r["margin"]
    limit = BWD_TILED_MAX if case[0] == TILED else BWD_GENERIC_MAX
    bad = {k: v for k, v in r["dev"].items() if not v <= limit}
    assert not bad, f"deviation from float64 above {limit:g} of scale: {bad}"


@pytest.mark.parametrize("case,combo", RUNS, ids=[case_id(c, k) for c, k in RUNS])
def test_backward_ex_matches_float64(case, combo):
    check(case, run_case(case, combo))


CHUNK_SCRIPT = r"""
import json, sys
sys.path.insert(0, %r)
from protoasnet_b200 import _lib
_lib.LIB_PATH = %r
from tests import test_push_forward_backward_gpu as t
print(json.dumps({k: t.run_case(t.CHUNKED_CASE, k, %d) for k in ("all", "features_occ")}))
"""


def test_backward_ex_chunks_match_float64():
    """Three tiled backward chunks with a ragged last (PASN_TILED_CHUNK = 3, read once per process, hence the subprocess):
    the distance and feature gradients are offset by each chunk's first clip."""
    env = dict(os.environ, PASN_TILED_CHUNK="3")
    out = subprocess.run([sys.executable, "-c", CHUNK_SCRIPT % (ROOT, _lib.LIB_PATH, SEED)], check=True, env=env, cwd=ROOT,
                         timeout=600, capture_output=True, text=True).stdout
    for combo, r in json.loads(out.strip().splitlines()[-1]).items():
        check(CHUNKED_CASE, r)


def _bit_equal(a, b):
    return np.array_equal(np.asarray(a).view(np.uint32), np.asarray(b).view(np.uint32))


@pytest.mark.parametrize("case", EXACT_CASES, ids=[case_id(c, "wrapper") for c in EXACT_CASES])
def test_legacy_entry_is_the_new_one_with_distance_and_features_null(case):
    prep = prepare(case, "all")
    up = {k: prep["up"][k] for k in ("logits", "similarity", "occurrence_map")}
    gx0, g0 = call_backward(case, prep, up, legacy=True)
    gx1, g1 = call_backward(case, prep, up)
    assert _bit_equal(gx0, gx1)
    for k in KEYS:
        assert _bit_equal(g0[k], g1[k]), k


@pytest.mark.parametrize("case", EXACT_CASES, ids=[case_id(c, "fold") for c in EXACT_CASES])
def test_distance_gradient_is_minus_the_similarity_gradient(case):
    """distance = 1 - similarity: grad_distance = g alone and grad_similarity = -g alone give the same gradients (up to
    the sign of a zero, which np.array_equal ignores)."""
    prep = prepare(case, "all")
    g = prep["up"]["distance"]
    gx0, g0 = call_backward(case, prep, {"distance": g})
    gx1, g1 = call_backward(case, prep, {"similarity": -g})
    assert np.array_equal(gx0, gx1)
    for k in KEYS:
        assert np.array_equal(g0[k], g1[k]), k


# ---- module level --------------------------------------------------------------------------------------------------
# (config, clips, feature-map format, parameter / feature seeds): the inputs of test_backward_gpu.py's cases at these shapes
MODULE_CASES = [("tiny_video", 7, "ncs", (17, 6)), ("tiny_video", 4, "nsc", (17, 6)),
                ("cfg3_video_b1024", 5, "ncs", (200, 12)), ("cfg3_video_b1024", 5, "nsc", (200, 12)),
                ("cfg3_video_b1024", 5, "ncs-bf16", (200, 12))]


def _module_inputs(cfg, n, fmt, seeds):
    dims = synth.CONFIGS[cfg]
    bf = fmt.endswith("-bf16")
    if cfg == "tiny_video":
        sd = synth.make_head_params(dims, seed=seeds[0], bias_scale=0.1, last_layer_noise=0.2, bf16_round=bf)
    else:
        sd = synth.make_head_params(dims, seed=seeds[0], bias_scale=0.02, bf16_round=True)
    x = synth.make_features(dims, n, seed=seeds[1], bf16_round=bf or cfg != "tiny_video")
    m = build_model(dims, sd)
    m.train()
    xt = torch.from_numpy(x).cuda()
    if fmt.startswith("nsc"):
        xt = xt.contiguous(memory_format=torch.channels_last_3d if dims.ndim == 3 else torch.channels_last)
    if bf:
        xt = xt.bfloat16()
    return dims, sd, x, m, xt.requires_grad_(True)


@pytest.mark.parametrize("cfg,n,fmt,seeds", MODULE_CASES, ids=[f"{c[0]}-{c[2]}" for c in MODULE_CASES])
def test_push_forward_trains_through_the_library(cfg, n, fmt, seeds, monkeypatch):
    dims, sd, x, m, xt = _module_inputs(cfg, n, fmt, seeds)
    rng = np.random.default_rng(5)
    fe = np.linalg.norm(ho.head_forward_f64(x, sd)["features_extracted"], axis=2)
    up = {"features_extracted": rng.standard_normal((n, dims.P, dims.D)) / np.where(fe > 0, fe, 1.0)[:, :, None],
          "distance": rng.standard_normal((n, dims.P)), "occurrence_map": rng.standard_normal((n, dims.P, dims.S)) * 0.1,
          "logits": rng.standard_normal((n, dims.K))}
    up = {k: v.astype(np.float32) for k, v in up.items()}
    ref_gx, ref_g = push_reference_grads(x, sd, up)

    def refuse(*a, **k):
        raise AssertionError("push_forward fell back to the PyTorch composite")

    monkeypatch.setattr(m, "_composite", refuse)
    m.autograd_mode = "kernel"
    feats, dist, occ, logits = m.push_forward(xt)
    assert feats.shape == (n, dims.P, dims.D) and dist.shape == (n, dims.P) and logits.shape == (n, dims.K)
    assert occ.shape == (n, dims.P, 1) + dims.spatial and all(t.requires_grad for t in (feats, dist, occ, logits))
    g = {k: torch.from_numpy(v).cuda() for k, v in up.items()}
    ((feats * g["features_extracted"]).sum() + (dist * g["distance"]).sum() +
     (occ.float() * g["occurrence_map"].reshape(occ.shape)).sum() + (logits * g["logits"]).sum()).backward()
    # bf16: autograd hands d(occurrence map) over rounded to bf16, and the feature-map gradient comes back in bf16
    rtol, afrac = (1e-2, 4e-3) if fmt.endswith("-bf16") else (2e-4, 2e-5)
    own = dict(m.named_parameters())
    for k in KEYS:
        assert_close(own[k].grad.reshape(ref_g[k].shape), ref_g[k], rtol, f"grad {k}", atol_frac=afrac)
    assert own["ones"].grad is None
    assert xt.grad.dtype == xt.dtype
    assert_close(xt.grad.reshape(ref_gx.shape), ref_gx, rtol, "grad feature map", atol_frac=afrac)


@pytest.mark.parametrize("cfg,n", [("tiny_video", 5), ("cfg3_video_b1024", 2)])
def test_get_occurence_map_absolute_val_trains_like_compute_occurence_map(cfg, n):
    dims, sd, x, m, xt = _module_inputs(cfg, n, "ncs", (31, 9))
    m.autograd_mode = "kernel"
    wo = torch.from_numpy(np.random.default_rng(4).standard_normal((n, dims.P, 1) + dims.spatial).astype(np.float32)).cuda()
    runs = []
    for method in (m.compute_occurence_map, m.get_occurence_map_absolute_val):
        m.zero_grad(set_to_none=True)
        xt.grad = None
        occ = method(xt)
        assert occ.grad_fn is not None and "_OccFunction" in type(occ.grad_fn).__name__
        (occ * wo).sum().backward()
        runs.append([xt.grad.clone()] + [p.grad.clone() for p in m.occurrence_module.parameters()])
        assert m.prototype_vectors.grad is None and m.add_on_layers[0].weight.grad is None
    for a, b in zip(*runs):
        assert _bit_equal(a.cpu().numpy(), b.cpu().numpy())


def test_other_autograd_modes_are_unchanged():
    dims, sd, x, m, xt = _module_inputs("tiny_video", 3, "ncs", (17, 6))
    m.autograd_mode = "error"
    for call in (m.push_forward, m.get_occurence_map_absolute_val):
        with pytest.raises(NotImplementedError):
            call(xt)
    m.autograd_mode = "composite"
    composite = m._composite(xt)
    m._composite = lambda x: composite
    feats, dist, occ, logits = m.push_forward(xt)
    assert feats is composite[0] and occ is composite[2] and logits is composite[3]
    assert torch.equal(dist, 1 - composite[1]) and dist.grad_fn is not None
    occ = m.get_occurence_map_absolute_val(xt)
    assert occ.grad_fn is not None and "_OccFunction" not in type(occ.grad_fn).__name__
    torch.testing.assert_close(occ, torch.abs(m.occurrence_module(xt)).unsqueeze(2))
