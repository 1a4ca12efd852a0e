"""The backward computes only the gradients that are wanted.

pasn_head_backward_ex is called through the C ABI with NULL for every gradient that is not wanted, on the shapes of
test_push_forward_backward_gpu.py and for the requires_grad patterns of ProtoPNet-style training stages.  Each requested
gradient must agree with float64 autograd (push_forward's op sequence) as in the full call, and on the deterministic shapes
be bit-identical to the full call's buffer; a pruned call never launches more kernels than a call that wants more.
pasn_last_layer_backward, the one-kernel backward of a last-layer-only stage, is checked against float64 gLᵀ·sim.  At
module level every stage pattern trains through the library (the PyTorch composite is patched to raise) and gives its
trainable parameters the joint run's gradients, while frozen ones get none."""
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
from tests.test_push_forward_backward_gpu import (CASES, CHUNKED_CASE, EXACT_CASES, FIELDS, OUTPUTS, _module_inputs,
                                                  push_reference_grads)
from tests.util import BWD_GENERIC_MAX, BWD_TILED_MAX

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SEED = int(os.environ.get("PASN_BWD_PARITY_SEED", "0"))
GX = "grad_feat"

# wanted outputs of the backward: parameter keys (tests.bwd_reference.KEYS) and GX for the feature-map gradient
ADDON, OCC, PROTO, LAST = KEYS[:4], KEYS[4:9], KEYS[9], KEYS[10]
SUBSETS = {
    "full": KEYS + [GX], "warm": KEYS, "conv": ADDON + OCC, "addon": ADDON, "occ": OCC, "proto_last": [PROTO, LAST],
    "last": [LAST], "feat": [GX], "nothing": [],
}
SINGLES = {f"only:{k}": [k] for k in KEYS}
OCC_SUBSETS = {"full": KEYS + [GX], "occ": OCC, "w3": [KEYS[8]], "w4_b4": KEYS[6:8], "w3_b3": KEYS[4:6],
               "occ_feat": OCC + [GX], "feat": [GX], "proto_last": [PROTO, LAST], "nothing": []}
# upstream gradients handed over (outputs) and the subsets tried with them
UPSTREAMS = {"all": OUTPUTS, "occ": ("occurrence_map",), "features": ("features_extracted",)}
RUNS = [(c, "all", SUBSETS) for c in CASES] + \
    [(c, "all", dict(SINGLES, full=SUBSETS["full"])) for c in EXACT_CASES] + \
    [(c, "occ", OCC_SUBSETS) for c in EXACT_CASES] + \
    [(c, "features", {"full": SUBSETS["full"], "proto_last": [PROTO, LAST], "nothing": []}) for c in EXACT_CASES]


@functools.lru_cache(maxsize=2)
def prepare(case, upstream="all", seed=SEED):
    """Conditioned inputs, upstream gradients of the outputs UPSTREAMS[upstream], the float64 reference and seeded buffer
    contents R (the recipe of test_push_forward_backward_gpu.prepare)."""
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
            "features_extracted": lambda: rng.standard_normal((N, P, D)) / np.where(fe > 0, fe, 1.0)[:, :, None]}
    up = {k: draw[k]().astype(np.float32) for k in UPSTREAMS[upstream]}
    gx_ref, g_ref = push_reference_grads(x, sd, up)
    R = {}
    for k in KEYS:
        g = g_ref[k].reshape(g_ref[k].shape[0], -1)
        scale = np.abs(g).max(axis=1, keepdims=True)
        scale = np.where(scale > 0, scale, float(np.abs(g).max()) or 1.0)
        R[k] = (rng.uniform(-1.0, 1.0, g.shape) * scale).astype(np.float32).reshape(g_ref[k].shape)
    return dict(dims=dims, sd=sd, x=x, margin=margin, up=up, gx_ref=gx_ref, g_ref=g_ref, R=R)


def call_subset(case, prep, wanted):
    """pasn_head_backward_ex with NULL for every gradient outside ``wanted``: returns (grad_feat or None, {key: buffer
    after the call} for the wanted keys, kernels launched)."""
    path, Cc, D, P, K, spatial, N, kind = case
    dtn, cl = KINDS[kind]
    dims, S = prep["dims"], prep["dims"].S
    lib = _lib.load()
    x = torch.from_numpy(prep["x"]).to(TORCH_DT[dtn]).cuda()
    if cl:
        x = x.contiguous(memory_format=torch.channels_last_3d if dims.ndim == 3 else torch.channels_last)
    d = PasnDims(N, Cc, D, P, K, S, _lib.DTYPES[x.dtype], _lib.PASN_LAYOUT_NSC if cl else _lib.PASN_LAYOUT_NCS,
                 _lib.PASN_OCC_ABS, path)
    params = [torch.from_numpy(np.ascontiguousarray(prep["sd"][k])).cuda() for k in KEYS]
    grads = {k: torch.from_numpy(prep["R"][k]).cuda() for k in KEYS if k in wanted}
    w = PasnWeights(*[t.data_ptr() for t in params])
    gw = PasnGrads(*[grads[k].data_ptr() if k in grads else None for k in KEYS])
    ups = {k: torch.from_numpy(v).cuda() for k, v in prep["up"].items()}
    u = PasnUpstream(**{FIELDS[k]: ups[k].data_ptr() if k in ups else None for k in OUTPUTS})
    gx = torch.full((N, Cc, S), float("nan"), device="cuda") if GX in wanted else None
    need = int(lib.pasn_head_backward_workspace_bytes(C.byref(d)))
    ws = torch.full((need,), 0xFF, dtype=torch.uint8, device="cuda")   # NaN in fp32 and bf16: unwritten scratch shows
    torch.cuda.synchronize()
    before = lib.pasn_debug_launch_count()
    st = lib.pasn_head_backward_ex(x.data_ptr(), C.byref(w), C.byref(d), C.byref(u), C.byref(gw),
                                   None if gx is None else gx.data_ptr(), ws.data_ptr(), ws.numel(),
                                   torch.cuda.current_stream().cuda_stream)
    launches = lib.pasn_debug_launch_count() - before
    _lib.check(st, "pasn_head_backward_ex")
    torch.cuda.synchronize()
    return (None if gx is None else gx.cpu().numpy()), {k: g.cpu().numpy() for k, g in grads.items()}, launches


def run_subsets(case, upstream, subsets, seed=SEED):
    """Every subset once: deviation of each wanted gradient from float64, bit-identity with the "full" call, launches."""
    prep = prepare(case, upstream, seed)
    out = {n: call_subset(case, prep, set(s)) for n, s in subsets.items()}
    gx_full, g_full, _ = out["full"]
    res = {"margin": prep["margin"], "dev": {}, "same": {}, "launches": {}}
    for n, (gx, got, launches) in out.items():
        dev = {k: deviation(got[k].astype(np.float64) - prep["R"][k].astype(np.float64), prep["g_ref"][k])[0] for k in got}
        same = {k: bool(np.array_equal(got[k].view(np.uint32), g_full[k].view(np.uint32))) for k in got}
        if gx is not None:
            dev[GX] = deviation(gx, prep["gx_ref"])[0]
            same[GX] = bool(np.array_equal(gx.view(np.uint32), gx_full.view(np.uint32)))
        res["dev"][n], res["same"][n], res["launches"][n] = dev, same, launches
    return res


def check(case, subsets, r, exact):
    assert r["margin"] >= TAU, r["margin"]
    limit = BWD_TILED_MAX if case[0] == TILED else BWD_GENERIC_MAX
    for n, dev in r["dev"].items():
        assert set(dev) == set(subsets[n]), n
        bad = {k: v for k, v in dev.items() if not v <= limit}
        assert not bad, f"{n}: deviation from float64 above {limit:g} of scale: {bad}"
        if exact:
            assert all(r["same"][n].values()), f"{n}: not bit-identical to the full call: {r['same'][n]}"
    launches = r["launches"]
    if "nothing" in launches:
        assert launches["nothing"] == 0, launches
    for a, sa in subsets.items():
        for b, sb in subsets.items():
            if set(sa) < set(sb):
                assert launches[a] <= launches[b], (a, b, launches)


@pytest.mark.parametrize("case,upstream,subsets", RUNS,
                         ids=[case_id(c, u) + ("-singles" if "only:" + KEYS[0] in s else "") for c, u, s in RUNS])
def test_subsets_match_float64_and_the_full_call(case, upstream, subsets):
    r = run_subsets(case, upstream, subsets)
    check(case, subsets, r, case in EXACT_CASES)
    if "warm" in subsets:
        launches = r["launches"]
        assert launches["proto_last"] < launches["warm"] and launches["last"] < launches["warm"], launches


CHUNK_SUBSETS = {"full": SUBSETS["full"], "conv": SUBSETS["conv"], "w3_feat": [KEYS[4], GX]}
CHUNK_SCRIPT = r"""
import json, sys
sys.path.insert(0, %r)
from protoasnet_b200 import _lib
_lib.LIB_PATH = %r
from tests import test_backward_subsets_gpu as t
print(json.dumps(t.run_subsets(t.CHUNKED_CASE, "all", t.CHUNK_SUBSETS, %d)))
"""


def test_pruned_subsets_in_chunks_match_float64():
    """Three tiled backward chunks with a ragged last (PASN_TILED_CHUNK = 3, read once per process, hence the subprocess),
    pruned to the convolution parameters, and to one half of the first layer's stacked weight gradient."""
    env = dict(os.environ, PASN_TILED_CHUNK="3")
    out = subprocess.run([sys.executable, "-c", CHUNK_SCRIPT % (ROOT, _lib.LIB_PATH, SEED)], check=True, env=env, cwd=ROOT,
                         timeout=600, capture_output=True, text=True).stdout
    check(CHUNKED_CASE, CHUNK_SUBSETS, json.loads(out.strip().splitlines()[-1]), False)


# ---- pasn_last_layer_backward ---------------------------------------------------------------------------------------
def _last_layer(gl, sim, g):
    lib = _lib.load()
    N, K = gl.shape
    P = sim.shape[1]
    _lib.check(lib.pasn_last_layer_backward(gl.data_ptr(), sim.data_ptr(), N, P, K, g.data_ptr(),
                                            torch.cuda.current_stream().cuda_stream), "pasn_last_layer_backward")


@pytest.mark.parametrize("N,P,K", [(256, 40, 4), (5, 9, 3), (70000, 40, 4), (64, 4096, 300)])
def test_last_layer_backward_matches_float64(N, P, K):
    rng = np.random.default_rng(N + P + K)
    gl = rng.standard_normal((N, K)).astype(np.float32)
    sim = rng.uniform(0.0, 1.0, (N, P)).astype(np.float32)
    ref = gl.astype(np.float64).T @ sim.astype(np.float64)
    R = (rng.uniform(-1.0, 1.0, (K, P)) * np.abs(ref).max()).astype(np.float32)
    glt, simt = torch.from_numpy(gl).cuda(), torch.from_numpy(sim).cuda()
    outs = []
    for _ in range(2):
        g = torch.from_numpy(R).cuda()
        lib = _lib.load()
        before = lib.pasn_debug_launch_count()
        _last_layer(glt, simt, g)
        assert lib.pasn_debug_launch_count() - before == 1
        outs.append(g.cpu().numpy())
    assert np.array_equal(outs[0].view(np.uint32), outs[1].view(np.uint32))
    # fp32 sums over 70 000 clips: the budget of such sums in the backward sweeps
    limit = 1e-6 if N <= 4096 else BWD_GENERIC_MAX
    dev = deviation(outs[0].astype(np.float64) - R.astype(np.float64), ref)[0]
    assert dev <= limit, dev


def test_last_layer_backward_without_clips_is_a_no_op():
    g = torch.full((3, 5), 7.0, device="cuda")
    e = torch.empty((0, 3), device="cuda")
    lib = _lib.load()
    before = lib.pasn_debug_launch_count()
    assert lib.pasn_last_layer_backward(e.data_ptr(), e.data_ptr(), 0, 5, 3, g.data_ptr(), None) == 0
    assert lib.pasn_debug_launch_count() == before
    assert torch.equal(g, torch.full((3, 5), 7.0, device="cuda"))


# ---- module level ---------------------------------------------------------------------------------------------------
# requires_grad patterns of training stages: (feature map, the eleven head parameters in KEYS order)
STAGES = {"joint": (True, [True] * 11), "warm": (False, [True] * 11), "conv": (False, [True] * 9 + [False] * 2),
          "proto_last": (False, [False] * 9 + [True] * 2), "last": (False, [False] * 10 + [True])}
# (config, clips, feature-map format, parameter / feature seeds): tiny_video runs the generic CUDA-core backward
# (deterministic: bit-identical gradients), cfg 3 the tiled chain
STAGE_CASES = [("tiny_video", 7, "ncs", (17, 6)), ("cfg3_video_b1024", 5, "ncs", (200, 12)),
               ("cfg3_video_b1024", 5, "ncs-bf16", (200, 12))]


def _train_step(m, xt, method, stage, up):
    """One forward + backward of ``method`` with the requires_grad pattern of ``stage``; returns (feature-map gradient,
    {key: parameter gradient or None}, the similarity the forward produced (forward) or 1 - distance (push_forward),
    library kernels launched by the backward)."""
    want_x, flags = STAGES[stage]
    own = dict(m.named_parameters())
    for k, f in zip(KEYS, flags):
        own[k].requires_grad_(f)
        own[k].grad = None
    x = xt.detach().clone().requires_grad_(want_x)
    if method == "forward":
        logits, sim, occ = m(x)
        loss = (logits * up["logits"]).sum() + (sim * up["similarity"]).sum()
    else:
        feats, dist, occ, logits = m.push_forward(x)
        sim = 1 - dist
        loss = (logits * up["logits"]).sum() + (dist * up["similarity"]).sum() + (feats * up["features"]).sum()
    loss = loss + (occ.float() * up["occurrence_map"].reshape(occ.shape)).sum()
    lib = _lib.load()
    torch.cuda.synchronize()
    before = lib.pasn_debug_launch_count()
    loss.backward()
    torch.cuda.synchronize()
    launches = lib.pasn_debug_launch_count() - before
    return x.grad, {k: (None if own[k].grad is None else own[k].grad.clone()) for k in KEYS}, sim.detach(), launches


def _dev(a, b):
    return deviation(a.double().cpu().numpy(), b.double().cpu().numpy())[0]


@pytest.mark.parametrize("method", ["forward", "push_forward"])
@pytest.mark.parametrize("cfg,n,fmt,seeds", STAGE_CASES, ids=[f"{c[0]}-{c[2]}" for c in STAGE_CASES])
def test_stages_train_their_parameters_like_the_joint_run(cfg, n, fmt, seeds, method, monkeypatch):
    dims, sd, x, m, xt = _module_inputs(cfg, n, fmt, seeds)

    def refuse(*a, **k):
        raise AssertionError("the head fell back to the PyTorch composite")

    monkeypatch.setattr(m, "_composite", refuse)
    m.autograd_mode = "kernel"
    rng = np.random.default_rng(7)
    up = {"logits": (n, dims.K), "similarity": (n, dims.P), "features": (n, dims.P, dims.D),
          "occurrence_map": (n, dims.P, dims.S)}
    up = {k: torch.from_numpy((rng.standard_normal(s) * (0.1 if k != "logits" else 1.0)).astype(np.float32)).cuda()
          for k, s in up.items()}
    runs = {s: _train_step(m, xt, method, s, up) for s in STAGES}
    gx_j, g_j, _, _ = runs["joint"]
    exact = cfg == "tiny_video"   # generic CUDA-core backward: every reduction in a fixed order
    for stage, (gx, g, sim, launches) in runs.items():
        want_x, flags = STAGES[stage]
        assert (gx is not None) == want_x, stage
        for k, f in zip(KEYS, flags):
            assert (g[k] is not None) == f, (stage, k)
            if not f or (stage == "last" and k == LAST):
                continue
            if exact:
                assert torch.equal(g[k], g_j[k]), (stage, k)
            else:
                assert _dev(g[k], g_j[k]) <= BWD_TILED_MAX, (stage, k, _dev(g[k], g_j[k]))
    # last layer alone: one kernel, gLᵀ·sim from the forward's own similarity
    _, g, sim, launches = runs["last"]
    assert launches == 1, launches
    ref = up["logits"].double().t() @ sim.double()
    assert _dev(g[LAST], ref) <= 1e-6, _dev(g[LAST], ref)
    # the joint run's gradient comes from the backward's fp32 recompute; a bf16 map's forward similarity is bf16 mode's
    assert _dev(g[LAST], g_j[LAST]) <= (1e-3 if fmt.endswith("-bf16") else BWD_TILED_MAX), _dev(g[LAST], g_j[LAST])


@pytest.mark.parametrize("cfg,n", [("tiny_video", 5), ("cfg3_video_b1024", 2)])
def test_compute_occurence_map_with_a_frozen_part_of_the_occurrence_module(cfg, n, monkeypatch):
    dims, sd, x, m, xt = _module_inputs(cfg, n, "ncs", (31, 9))
    m.autograd_mode = "kernel"
    monkeypatch.setattr(m, "_composite", lambda *a, **k: pytest.fail("fell back to the PyTorch composite"))
    wo = torch.from_numpy(np.random.default_rng(4).standard_normal((n, dims.P, 1) + dims.spatial).astype(np.float32)).cuda()
    occ_params = list(m.occurrence_module.parameters())   # W3, b3, W4, b4, W5
    runs = []
    for frozen in ((), (0, 1), (0, 1, 2, 3)):
        m.zero_grad(set_to_none=True)
        for i, p in enumerate(occ_params):
            p.requires_grad_(i not in frozen)
        xi = xt.detach().clone().requires_grad_(not frozen)
        occ = m.compute_occurence_map(xi)
        assert "_OccFunction" in type(occ.grad_fn).__name__
        (occ * wo).sum().backward()
        assert (xi.grad is not None) == (not frozen)
        assert m.prototype_vectors.grad is None and m.add_on_layers[0].weight.grad is None
        for i, p in enumerate(occ_params):
            assert (p.grad is None) == (i in frozen), (frozen, i)
        runs.append([None if p.grad is None else p.grad.clone() for p in occ_params])
    for run in runs[1:]:
        for a, b in zip(runs[0], run):
            if b is None:
                continue
            if cfg == "tiny_video":
                assert torch.equal(a, b)
            else:
                assert _dev(b, a) <= BWD_TILED_MAX, _dev(b, a)
