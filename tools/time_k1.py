"""Time the fused head (K1 main-kernel events + whole step) at N=1024."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from protoasnet_b200 import _lib, synth
from tests.util import build_model
dims = synth.CONFIGS[sys.argv[1] if len(sys.argv) > 1 else "cfg3_video_b1024"]
n = int(sys.argv[2]) if len(sys.argv) > 2 else 1024
sd = synth.make_head_params(dims, seed=200, bias_scale=0.02, bf16_round=True)
m = build_model(dims, sd, path=_lib.PASN_PATH_TCGEN05)
x = torch.relu(torch.randn((n, dims.C) + dims.spatial, device="cuda")).bfloat16()
lib = _lib.load()
with torch.no_grad():
    for _ in range(3): m(x)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(10): m(x)
    e1.record(); torch.cuda.synchronize()
    lib.pasn_debug_time_main_kernel(1)
    ks = []
    for _ in range(10):
        m(x); ks.append(lib.pasn_debug_last_main_kernel_ms())
print(f"{sys.argv[1:]} step {e0.elapsed_time(e1)/10*1e3:.1f} us, K1 {np.mean(ks)*1e3:.1f} us")
