"""Fused vs generic path over awkward batch sizes (CTA / tile boundary cases) for both layouts."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from protoasnet_b200 import _lib, synth
from tests.util import build_model
dims = synth.CONFIGS["cfg3_video_b1024"]
sd = synth.make_head_params(dims, seed=200, bias_scale=0.02, bf16_round=True)
m = build_model(dims, sd, path=_lib.PASN_PATH_TCGEN05)
mg = build_model(dims, sd, path=_lib.PASN_PATH_GENERIC)
worst = 0.0
for n in (1, 2, 147, 148, 150, 295, 444, 1023, 2050, 4099):
    x = torch.relu(torch.randn((n, dims.C) + dims.spatial, device="cuda", generator=torch.Generator(device="cuda").manual_seed(n))).bfloat16()
    with torch.no_grad():
        ref = mg.push_forward(x)
        for xx, name in ((x, "ncdhw"), (x.contiguous(memory_format=torch.channels_last_3d), "cl")):
            out = m.push_forward(xx)
            torch.cuda.synchronize()
            e_sim = float((out[1] - ref[1]).abs().max())
            e_log = float((out[3] - ref[3]).abs().max() / ref[3].abs().max())
            e_occ = float((out[2].float() - ref[2].float()).abs().max() / ref[2].float().abs().max())
            worst = max(worst, e_sim, e_log)
            flag = "" if (e_sim < 1e-3 and e_log < 1e-3 and e_occ < 2e-2 and not torch.isnan(out[3]).any()) else "  <-- FAIL"
            print(f"n={n:5d} {name:6s} sim {e_sim:.2e} logits {e_log:.2e} occ {e_occ:.2e}{flag}")
print("worst", worst)
