"""fp16 against bf16 feature maps on the same head, alternating in one process: CUDA-event step times (and the token
kernel's own time where the fused path runs) for config 3 (NCDHW and channels_last, N = 1024), config 2 (N = 1024),
config 5 (N = 32) and forward + backward at config 3, N = 256.  Prints the card and its power limit first.

    python tools/time_fp16.py [--reps 5] [--iters 20]
"""
import argparse
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from protoasnet_b200 import _lib, synth  # noqa: E402
from tests.util import build_model  # noqa: E402


def _time(fn, iters):
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record()
    for _ in range(iters):
        fn()
    ev[1].record()
    torch.cuda.synchronize()
    return ev[0].elapsed_time(ev[1]) / iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--iters", type=int, default=20)
    a = ap.parse_args()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip()
    print(f"card: {q or torch.cuda.get_device_name()}")
    lib = _lib.load()
    cases = [("cfg3 N=1024 ncdhw", "cfg3_video_b1024", 1024, False, False),
             ("cfg3 N=1024 channels_last", "cfg3_video_b1024", 1024, True, False),
             ("cfg2 N=1024", "cfg2_image", 1024, False, False),
             ("cfg5 N=32", "cfg5_scaled", 32, False, False),
             ("cfg3 N=256 fwd+bwd", "cfg3_video_b1024", 256, False, True)]
    for name, cfg, n, cl, bwd in cases:
        dims = synth.CONFIGS[cfg]
        sd = synth.make_head_params(dims, seed=200, bias_scale=0.05, bf16_round=True)
        m = build_model(dims, sd)
        x32 = torch.from_numpy(synth.make_features(dims, n, seed=1)).cuda()
        xs = {}
        for dt in (torch.float16, torch.bfloat16):
            x = x32.to(dt)
            if cl:
                x = x.contiguous(memory_format=torch.channels_last_3d if dims.ndim == 3 else torch.channels_last)
            xs[dt] = x
        del x32
        if bwd:
            m.autograd_mode = "kernel"
            for dt in xs:
                xs[dt].requires_grad_(True)

            def step(x):
                lg, sm, oc = m(x)
                (lg.sum() + sm.sum() + oc.float().sum() * 1e-3).backward()
        else:
            def step(x):
                with torch.no_grad():
                    m(x)
        res = {dt: [] for dt in xs}
        k1 = {dt: [] for dt in xs}
        for dt in xs:   # warm-up of both shapes (packing, module loads)
            for _ in range(3):
                step(xs[dt])
        torch.cuda.synchronize()
        for _ in range(a.reps):
            for dt in xs:
                res[dt].append(_time(lambda: step(xs[dt]), a.iters))
                if not bwd:
                    lib.pasn_debug_time_main_kernel(1)
                    step(xs[dt])
                    k1[dt].append(lib.pasn_debug_last_main_kernel_ms())
                    lib.pasn_debug_time_main_kernel(0)
        line = [name]
        for dt, tag in ((torch.float16, "fp16"), (torch.bfloat16, "bf16")):
            r = sorted(res[dt])
            s = f"{tag} step {r[len(r) // 2]:.4f} ms (min {r[0]:.4f}, max {r[-1]:.4f})"
            if k1[dt]:
                kk = sorted(k1[dt])
                s += f", main kernel {kk[len(kk) // 2]:.4f} ms"
            line.append(s)
        f16, b16 = sorted(res[torch.float16])[a.reps // 2], sorted(res[torch.bfloat16])[a.reps // 2]
        line.append(f"fp16/bf16 {f16 / b16:.3f}")
        print(" | ".join(line), flush=True)
        del m, xs
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
