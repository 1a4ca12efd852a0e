"""Small fused-path run for compute-sanitizer (memcheck): ragged shapes."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from protoasnet_b200 import _lib, synth
from tests.util import build_model
for (C, P, K, spatial, n) in [(128, 12, 3, (1, 10, 14), 5), (512, 40, 4, (4, 7, 7), 9)]:
    dims = synth.HeadDims(C, 256, P, K, spatial)
    sd = synth.make_head_params(dims, seed=41, bias_scale=0.05, bf16_round=True)
    m = build_model(dims, sd, path=_lib.PASN_PATH_TCGEN05)
    x = torch.from_numpy(synth.make_features(dims, n, seed=23, bf16_round=True)).cuda().bfloat16()
    with torch.no_grad():
        out = m.push_forward(x)
    torch.cuda.synchronize()
    print(C, P, n, "ok", float(out[1].sum()))
# tiled chain: statistics folded into the pooling GEMM (few prototypes: cached slices; many: direct reads), plain forward
for (C, D, P, K, spatial, n, dt) in [(64, 128, 9, 3, (2, 2), 5, torch.bfloat16), (128, 256, 40, 4, (7, 7), 6, torch.bfloat16),
                                     (64, 128, 1024, 4, (4, 4), 2, torch.bfloat16), (64, 128, 33, 3, (1, 5, 10), 3, torch.float32)]:
    dims = synth.HeadDims(C, D, P, K, spatial)
    bf = dt == torch.bfloat16
    sd = synth.make_head_params(dims, seed=43, bias_scale=0.05, bf16_round=bf)
    m = build_model(dims, sd, path=_lib.PASN_PATH_TILED)
    x = torch.from_numpy(synth.make_features(dims, n, seed=29, bf16_round=bf)).cuda().to(dt)
    with torch.no_grad():
        logits, sim, occ = m(x)
        out = m.push_forward(x)
    torch.cuda.synchronize()
    print("tiled", C, D, P, n, str(dt)[6:], "ok", float(sim.sum()), float((out[1] - (1 - sim)).abs().max()))
