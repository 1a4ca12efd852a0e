"""Phase trace (see trace_k1.py) for a channels_last feature map."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from protoasnet_b200 import _lib, synth
from tests.util import build_model
dims = synth.CONFIGS["cfg3_video_b1024"]
sd = synth.make_head_params(dims, seed=200, bias_scale=0.02, bf16_round=True)
m = build_model(dims, sd, path=_lib.PASN_PATH_TCGEN05)
x = torch.relu(torch.randn((1024, dims.C) + dims.spatial, device="cuda")).bfloat16().contiguous(memory_format=torch.channels_last_3d)
lib = _lib.load()
buf = torch.zeros(1024, dtype=torch.int64, device="cuda")
with torch.no_grad():
    for _ in range(3): m(x)
    lib.pasn_debug_set_trace(buf.data_ptr()); m(x); torch.cuda.synchronize(); lib.pasn_debug_set_trace(None)
t = buf.cpu()[:768].view(3, 16, 16); t0 = int(t[0, 0, 0])
names_m = ["start", "gbfree", "Gissued", "abfree", "G2issued", "Oissued", "Aissued", "pool0", "pool1", "g1ready_seen", "w4a_seen"]
names_e = ["E-start", "gdone", "E1done", "g2done", "E3done", "odone", "E4done", "adone", "E2done", "fedone", "E5done"]
for tile in range(3, 7):
    print(f"tile {tile}")
    print("  MMA: " + " ".join(f"{n}={int(t[0, tile, i]) - t0}" for i, n in enumerate(names_m)))
    print(f"  blocked x {int(t[0, tile, 11])} w {int(t[0, tile, 12])}")
    print("  chunks (G + A blocks):", [int(v) for v in t[2, tile, :8]])
    print("  EPI: " + " ".join(f"{n}={int(t[1, tile, i]) - t0}" for i, n in enumerate(names_e)))
