"""Forward + backward of the head at the cfg-3 shape (fp32 feature map), through the library (autograd_mode='kernel')
against the PyTorch composite, for forward() and push_forward(); the two modes alternate within one process.  Prints
the card and its power limit first, then per (N, method, mode) the median step time over the repetitions.

--stages times forward() instead under the requires_grad patterns of training stages (STAGES: which of the feature map
and the head's parameters are trained), and prints the library kernels one backward launches in each.

    python tools/time_backward.py [--n 64 256] [--reps 5] [--iters 20] [--stages]
"""
import argparse
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from protoasnet_b200 import _lib, synth  # noqa: E402
from protoasnet_b200.head import _head_params  # noqa: E402
from tests.util import build_model  # noqa: E402


def _time(fn, iters):
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record()
    for _ in range(iters):
        fn()
    ev[1].record()
    torch.cuda.synchronize()
    return ev[0].elapsed_time(ev[1]) / iters


def _loss(method, m, x):
    """A loss on every output the method returns."""
    if method == "forward":
        logits, sim, occ = m(x)
        return logits.sum() + sim.sum() + occ.float().abs().sum() * 1e-4
    feats, dist, occ, logits = m.push_forward(x)
    return feats.sum() * 1e-4 + dist.sum() + occ.float().abs().sum() * 1e-4 + logits.sum()


# stage -> (feature map trained, head parameters trained, by index into _head_params' order)
STAGES = {"joint": (True, range(11)), "warm": (False, range(11)), "conv-only": (False, range(9)),
          "prototypes+last": (False, (9, 10)), "last-layer": (False, (10,))}


def _set_stage(m, stage):
    trained = set(STAGES[stage][1])
    for i, p in enumerate(_head_params(m)):
        p.requires_grad_(i in trained)


def _stages(a, models, dims):
    lib = _lib.load()
    for n in a.n:
        x0 = torch.relu(torch.randn((n, dims.C) + dims.spatial, device="cuda"))
        for stage, (want_x, _) in STAGES.items():
            x = x0.detach().requires_grad_(want_x)

            def step(m):
                for p in m.parameters():
                    p.grad = None
                x.grad = None
                _loss("forward", m, x).backward()

            for m in models.values():
                _set_stage(m, stage)
                for _ in range(3):
                    step(m)
            loss = _loss("forward", models["kernel"], x)
            torch.cuda.synchronize()
            before = lib.pasn_debug_launch_count()
            loss.backward()
            launches = lib.pasn_debug_launch_count() - before
            torch.cuda.synchronize()
            res = {mode: [] for mode in models}
            for _ in range(a.reps):
                for mode, m in models.items():
                    res[mode].append(_time(lambda: step(m), a.iters))
            med = {mode: sorted(r)[len(r) // 2] for mode, r in res.items()}
            print(f"N={n} {stage}: fwd+bwd " + ", ".join(
                f"{mode} {med[mode]:.3f} ms (min {min(res[mode]):.3f}, max {max(res[mode]):.3f})" for mode in models) +
                f" | kernel/composite {med['kernel'] / med['composite']:.3f} | library launches per backward {launches}",
                flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, nargs="+", default=[64, 256])
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--stages", action="store_true", help="time forward() per training stage (STAGES)")
    a = ap.parse_args()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip()
    print(f"card: {q or torch.cuda.get_device_name()}")
    dims = synth.CONFIGS["cfg3_video_b1024"]
    sd = synth.make_head_params(dims, seed=200, bias_scale=0.02, bf16_round=True)
    models = {mode: build_model(dims, sd) for mode in ("kernel", "composite")}
    for mode, m in models.items():
        m.autograd_mode = mode
    if a.stages:
        return _stages(a, models, dims)
    for n in a.n:
        x = torch.relu(torch.randn((n, dims.C) + dims.spatial, device="cuda"))
        for method in ("forward", "push_forward"):
            def step(m):
                for p in m.parameters():
                    p.grad = None
                _loss(method, m, x).backward()

            for m in models.values():   # warm-up (weight packing, module loads, cuDNN algorithm choice)
                for _ in range(3):
                    step(m)
            torch.cuda.synchronize()
            res = {mode: [] for mode in models}
            for _ in range(a.reps):
                for mode, m in models.items():
                    res[mode].append(_time(lambda: step(m), a.iters))
            med = {mode: sorted(r)[len(r) // 2] for mode, r in res.items()}
            print(f"N={n} {method}: fwd+bwd " + ", ".join(
                f"{mode} {med[mode]:.3f} ms (min {min(res[mode]):.3f}, max {max(res[mode]):.3f})" for mode in models) +
                f" | kernel/composite {med['kernel'] / med['composite']:.3f}", flush=True)


if __name__ == "__main__":
    main()
