"""Shared helpers for the GPU parity tests (they call the CUDA path through the C ABI via protoasnet_b200)."""
import json

import numpy as np
import torch

import protoasnet_b200 as pasn
from protoasnet_b200 import synth

FP32_RTOL = 1e-5   # north_star: logits and similarities within 1e-5 relative in fp32
BF16_RTOL = 1e-3   # ... and 1e-3 relative in bf16
# fp32 feature maps on the tensor cores (tiled path: bf16 hi/lo split, 16 significant bits per operand, fp32 accumulation):
# logits / similarities / distances keep north_star's 1e-5; the big intermediate tensors that are also outputs
# (features_extracted, occurrence_map, pushed prototype_vectors) are judged against their scale at this fraction.
# kernel_path = PASN_PATH_GENERIC (CUDA-core FFMA) is the path that meets 1e-6 of scale on those as well.
FP32_TC_FEAT_ATOL = 3e-5

# bf16 / fp16 mode on the tensor cores against oracle/emulate.py (the same rounding points, float64 accumulation): what is
# left is fp32 accumulation order and the rare rounding flips it causes.  Comments: the worst value measured over the
# cases of tests/test_tc_emulated_parity_gpu.py on one B200 at a 1000 W power limit (tools/emu_parity_report.py).
EMU_OCC_BITEQ = 0.98          # fraction of occurrence-map entries bit-equal to the emulation, at least        (0.994)
EMU_OCC_BITEQ_F16 = 0.9       # ... for fp16 maps stored straight from fp32 (tiled chain): a grid 8x finer    (0.958)
EMU_OCC_ULPS = 32             # every other entry within this many bf16 ulps of the emulated value ...        (12)
EMU_OCC_ATOL_FRAC = 4e-3      # ... or within this fraction of the map's scale (near-zero entries)          (9.3e-4)
EMU_FEAT_POOL_FIRST = 4e-4    # features_extracted, fraction of their scale: pooling before W2             (9.5e-5)
EMU_FEAT_W2_FIRST = 1e-3      # ... W2 before the pooling (F is rounded to bf16 per voxel: flips reach the features) (3.4e-4)
EMU_SIM_ATOL = 5e-5           # similarity and distance, absolute                                          (1.4e-5)
EMU_LOGITS_FRAC = 1e-5        # logits, fraction of their scale                                            (2.4e-6)
EMU_COSINE_PUSH = 2e-6        # float64 cosine chain on the kernel's own features vs push_forward: similarity and
                              # distance absolute, logits as a fraction of their scale                    (4.7e-7)
EMU_COSINE_FWD = 2e-6         # ... vs forward() (which may take its cosine from row statistics of the pooling GEMM) (4.7e-7)

# pasn_head_backward against float64 autograd on conditioned inputs (tests/test_backward_parity_gpu.py): max |got - ref|
# over max |ref| of the feature-map gradient and of each of the eleven parameter gradients, per backward family.  Comments:
# the worst value over the sweep at two seeds on one B200 at a 1000 W power limit (tools/bwd_parity_report.py).
BWD_TILED_MAX = 1e-4          # tiled tensor-core chain (three-pass bf16 hi|lo GEMMs, fp32 accumulation)        (3.5e-5)
BWD_GENERIC_MAX = 5e-5        # generic CUDA-core FFMA kernels: prototype / last-layer gradients summed in fp32
                              # over 70 000 clips (2.1e-5); every shape with fewer than 100 clips stays at 1e-6  (9.7e-7)

def occ_agreement(got, ref):
    """(fraction of entries bit-equal, worst entry in units of its allowance) of an occurrence map against the emulated
    one, both given as the values of the map's dtype.  An entry is allowed EMU_OCC_ULPS bf16 ulps of the reference value
    or EMU_OCC_ATOL_FRAC of the map's scale, whichever is larger; the map agrees when the second number is <= 1."""
    got = np.asarray(got, dtype=np.float64)
    ref = np.asarray(ref, dtype=np.float64)
    if got.size == 0:
        return 1.0, 0.0
    diff = np.abs(got - ref)
    mag = np.maximum(np.abs(ref), np.finfo(np.float32).tiny)
    ulp = np.exp2(np.floor(np.log2(mag)) - 7)    # bf16: 8 significant bits
    allow = np.maximum(EMU_OCC_ULPS * ulp, EMU_OCC_ATOL_FRAC * float(np.abs(ref).max()))
    return float(np.mean(diff == 0)), float((diff / allow).max())


def feat_atol(model, x):
    """atol_frac for features_extracted / occurrence_map of ``model`` fed ``x``: None (default, rtol/10) unless an fp32 input
    is served by a tensor-core path."""
    import ctypes as C
    from protoasnet_b200 import _lib
    if x.dtype != torch.float32:
        return None
    dims = model._rt.make_dims(x, model.kernel_path)[0]
    return FP32_TC_FEAT_ATOL if _lib.load().pasn_tcgen05_supported(C.byref(dims)) else None


def build_model(dims: synth.HeadDims, sd_np, device="cuda", path=None):
    if dims.ndim == 3:
        m = pasn.construct_Video_XProtoNet(pasn.FeatureInput(dims.C), pretrained=False,
                                           prototype_shape=dims.prototype_shape, num_classes=dims.K)
    else:
        m = pasn.construct_XProtoNet(pasn.FeatureInput(dims.C), pretrained=False,
                                     prototype_shape=dims.prototype_shape, num_classes=dims.K)
    own = m.state_dict()
    assert set(own.keys()) == set(sd_np.keys())
    m.load_state_dict({k: torch.from_numpy(np.ascontiguousarray(v)) for k, v in sd_np.items()})
    m = m.to(device).eval()
    if path is not None:
        m.kernel_path = path
    return m


def assert_close(got, ref, rtol, name="", atol_frac=None):
    """|got - ref| <= atol + rtol*|ref| with atol = atol_frac * max|ref| (default rtol/10: near-zero entries of a
    tensor are judged against the tensor's scale, everything else relatively)."""
    got = got.detach().float().cpu().numpy() if isinstance(got, torch.Tensor) else np.asarray(got)
    ref = np.asarray(ref, dtype=np.float64)
    scale = float(np.abs(ref).max()) if ref.size else 1.0
    frac = rtol * 0.1 if atol_frac is None else atol_frac
    np.testing.assert_allclose(got, ref, rtol=rtol, atol=frac * scale + 1e-30, err_msg=name)


def load_golden(path):
    z = np.load(path)
    return z, json.loads(str(z["recipe"]))
