"""Soak: many back-to-back fused forwards (both layouts, several batch sizes) must be bit-identical to the first one and never trip a bounded wait (PASN_DEBUG_SYNC=1 makes every call check the kernel's error word)."""
import os, sys, time
os.environ["PASN_DEBUG_SYNC"] = "1"
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from protoasnet_b200 import _lib, synth
from tests.util import build_model
t0 = time.time()
bad = 0
for cfg, ns in (("cfg3_video_b1024", (1024, 333, 75, 8)), ("cfg1_video_yml", (8, 40, 150))):
    dims = synth.CONFIGS[cfg]
    sd = synth.make_head_params(dims, seed=200, bias_scale=0.02, bf16_round=True)
    m = build_model(dims, sd, path=_lib.PASN_PATH_TCGEN05)
    for n in ns:
        x = torch.relu(torch.randn((n, dims.C) + dims.spatial, device="cuda")).bfloat16()
        for xx, name in ((x, "ncdhw"), (x.contiguous(memory_format=torch.channels_last_3d), "cl")):
            with torch.no_grad():
                ref = m.push_forward(xx)
                reps = int(os.environ.get("SOAK_SCALE", "1")) * (150 if n >= 300 else 60)
                for i in range(reps):
                    out = m.push_forward(xx)
                    if not all(torch.equal(a, b) for a, b in zip(out, ref)):
                        bad += 1
                        print("MISMATCH", cfg, n, name, i)
                        break
            print(cfg, n, name, "ok", f"{time.time() - t0:.0f}s", flush=True)
print("soak done, mismatches:", bad)
