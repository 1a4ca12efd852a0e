"""Wall-clock (globaltimer, ns) timeline of CTA 0 of the prototype kernel K2 next to the token kernel K1 of the same call."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from protoasnet_b200 import _lib, synth
from tests.util import build_model

dims = synth.CONFIGS["cfg3_video_b1024"]
sd = synth.make_head_params(dims, seed=200, bias_scale=0.02, bf16_round=True)
m = build_model(dims, sd, path=_lib.PASN_PATH_TCGEN05)
x = torch.relu(torch.randn((1024, dims.C) + dims.spatial, device="cuda")).bfloat16()
lib = _lib.load()
buf = torch.zeros(1024, dtype=torch.int64, device="cuda")
with torch.no_grad():
    for _ in range(3):
        m(x)
    lib.pasn_debug_set_trace(buf.data_ptr())
    m(x)
    torch.cuda.synchronize()
    lib.pasn_debug_set_trace(None)
t = buf.cpu()[768:].tolist()
k1s, k1e = t[0], t[1]
g = t[16:]
print(f"K1 CTA0: start 0, end {k1e - k1s} ns")
rel = lambda v: (v - k1s) if v else None
print(f"K2 CTA0: start {rel(g[0])}, prologue done {rel(g[1])}, griddep_wait passed {rel(g[2])}, end {rel(g[3])}")
for it in range(20):
    b = g[16 + it * 8: 16 + it * 8 + 8]
    if not b[0]:
        break
    print(f"  it {it} tile {t[200 + it]}: tile taken {rel(b[7])}, stage full seen {[rel(v) for v in b[:4]]}, MMAs committed {rel(b[4])}, epilogue start {rel(b[5])}, end {rel(b[6])}")
