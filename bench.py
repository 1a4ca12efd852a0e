#!/usr/bin/env python
"""Benchmark of the ProtoASNet prototype-head hot path on B200 (contract: see DESIGN.md 'Measurement').

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

One "step" = one prototype-head forward (BASELINE config 3: feature map 512x4x7x7 bf16, D=256, P=40, K=4) over a
batch of 1024 synthetic clips per GPU.  ``value`` = clips/s with the feature maps resident in HBM; ``e2e`` = the same
through the public module API with pinned HOST buffers (H2D of the batch + D2H of logits/similarity inside the timed
region); ``push`` = seconds for one push / prototype projection over 50 000 clips sharded across the N ranks
(fused similarity+argmin, one NCCL all-reduce(MIN) of packed keys + one all-reduce(SUM) of winner rows).
``--impl reference`` times the reference algorithm's CPU port (oracle/, op-for-op the reference's PyTorch ops) on
the host cores of the box.
``--dump-outputs DIR`` writes what the last timed step returned (rank 0: logits, similarity, occurrence_map) as
DIR/<name>.npy in float32 (32 MB for the batch of 1024); inputs and weights are seeded, so two builds can be compared
output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

WORKLOAD = "cfg3_video_b1024"
BATCH = 1024
PUSH_CLIPS = 50000


def flops_bytes_per_clip(d):
    C, D, P, K, S = d.C, d.D, d.P, d.K, d.S
    addon = 2 * C * D * S + 2 * D * D * S
    occ = 2 * C * D * S + 2 * D * (D // 2) * S + 2 * (D // 2) * P * S
    pool = 2 * P * D * S
    tail = 6 * P * D + 2 * P * K
    nbytes = C * S * 2 + P * S * 2 + (P + K) * 4
    return addon + occ + pool + tail, nbytes


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        j = json.load(open(p))
        return {"hbm_gbs": j["hbm_gbs"], "bf16_tflops": j["bf16_tflops"],
                "bf16_tflops_sustained": j.get("bf16_tflops_sustained", j["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 100 ms while the timed regions run."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [t.strip() for t in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        # "under load" = samples in the upper half of what we saw
        load = [v for v in sm if v >= 0.5 * max(sm)] if sm else []
        return {"sm_mhz": float(np.median(load)) if load else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def make_model(dims, device, path):
    import protoasnet_b200 as pasn
    from protoasnet_b200 import synth, _lib

    sd = synth.make_head_params(dims, seed=200, bias_scale=0.02, bf16_round=True)
    m = pasn.construct_Video_XProtoNet(pasn.FeatureInput(dims.C), pretrained=False, prototype_shape=dims.prototype_shape,
                                       num_classes=dims.K)
    m.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()})
    m = m.to(device).eval()
    m.kernel_path = {"auto": _lib.PASN_PATH_AUTO, "generic": _lib.PASN_PATH_GENERIC, "tcgen05": _lib.PASN_PATH_TCGEN05}[path]
    return m, sd


class _VideoStub(torch.nn.Module):
    """Identity backbone whose repr contains RESNET2P1D and whose last Conv3d has C out-channels (what the reference's
    PPNet.get_cnn_backbone_out_channels looks for, src/models/ProtoPNet.py:152-162)."""

    def __init__(self, C):
        super().__init__()
        self.resnet2p1d_marker = torch.nn.Conv3d(1, C, 1)

    def forward(self, x):
        return x

    def __repr__(self):
        return "RESNET2P1D_identity_stub(" + super().__repr__() + ")"


def reference_head(dims, sd):
    """-> (callable features -> (logits, similarity, occurrence_map), kind).  kind "reference": the UNMODIFIED reference
    class (staged under oracle/_ref by build(), see oracle/make_ref.py) with an identity backbone; kind "port": the
    oracle's op-for-op restatement when the staged files are absent."""
    from oracle import head_oracle as ho
    from oracle import make_ref

    tsd = ho.to_torch_sd(sd)
    classes = None
    try:
        classes = make_ref.load_reference_classes()
    except Exception:
        classes = None
    if classes is not None:
        Video_XProtoNet, _ = classes
        m = Video_XProtoNet(cnn_backbone=_VideoStub(dims.C), img_size=112, prototype_shape=dims.prototype_shape,
                            proto_layer_rf_info=None, num_classes=dims.K, init_weights=True)
        own = m.state_dict()
        m.load_state_dict({k: (tsd[k] if k in tsd else v) for k, v in own.items()})
        m.eval()
        return (lambda x: m(x)), "reference"
    return (lambda x: ho.head_forward_torch(x, tsd)), "port"


def cpu_head_clips_per_sec(dims, sd, clips_per_run, min_seconds, max_runs, threads):
    """The reference's head on the host CPU (its own class when staged, else the oracle port: the same PyTorch ops),
    fp32, no_grad, in chunks of 64 clips (batch 1024 would allocate 8 GB for the reference's broadcast product)."""
    from protoasnet_b200 import synth

    torch.set_num_threads(threads)
    fwd, kind = reference_head(dims, sd)
    x = torch.from_numpy(synth.make_features(dims, min(64, clips_per_run), seed=0, bf16_round=True))
    chunks = max(1, clips_per_run // x.shape[0])
    with torch.no_grad():
        fwd(x)  # warm-up
        times = []
        t_all = time.perf_counter()
        while len(times) < max_runs and (len(times) < 3 or time.perf_counter() - t_all < min_seconds):
            t0 = time.perf_counter()
            for _ in range(chunks):
                fwd(x)
            times.append(time.perf_counter() - t0)
    return chunks * x.shape[0] / float(np.median(times)), chunks * x.shape[0], len(times), kind


def cpu_push_seconds_per_50k(dims, sd, n_sample, threads):
    """Push CPU baseline (BASELINE.md section 5): the restated reference loop (oracle/push_oracle.py, following
    src/utils/push_abs_revision.py:226-307) with the video push loader's batch size 5
    (src/configs/Ours_ProtoASNet_Video.yml:25) over a sample of the 50k set, extrapolated linearly."""
    from oracle import push_oracle as po
    from protoasnet_b200 import synth

    torch.set_num_threads(threads)
    x = synth.make_features(dims, n_sample, seed=1000, bf16_round=True)
    labels = synth.push_labels(n_sample, dims.K - 1, seed=7)
    t0 = time.perf_counter()
    po.push_prototypes_oracle(x, labels, sd, dims.K, batch=5)
    dt = time.perf_counter() - t0
    return dt * (50000.0 / n_sample), dt


def _bind_host_memory_to_gpu_node(dev):
    """Best effort: prefer host memory on the NUMA node of this rank's GPU for the pinned staging buffers allocated from here
    on (set_mempolicy(MPOL_PREFERRED)).  With N ranks copying their batches host -> device at once, buffers that all sit on
    the node the launcher happened to run on share one memory controller and cross the socket link.  Returns the node or None."""
    try:
        import ctypes
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(dev.index if dev.index is not None else 0)
        pci = pynvml.nvmlDeviceGetPciInfo(h).busId
        pci = (pci.decode() if isinstance(pci, bytes) else str(pci)).lower()
        if len(pci.split(":")[0]) == 8:
            pci = pci[4:]
        node = int(open(f"/sys/bus/pci/devices/{pci}/numa_node").read().strip())
        if node < 0:
            return None
        libc = ctypes.CDLL(None, use_errno=True)
        mask = ctypes.c_ulong(1 << node)
        rc = libc.syscall(238, 1, ctypes.byref(mask), ctypes.c_ulong(64))   # set_mempolicy(MPOL_PREFERRED) on x86_64
        return node if rc == 0 else None
    except Exception:   # noqa: BLE001 -- purely an optimisation
        return None


def dump_outputs(directory, outputs):
    """outputs: (logits, similarity, occurrence_map) as a caller of the head receives them -> DIR/<name>.npy, float32."""
    os.makedirs(directory, exist_ok=True)
    for name, t in zip(("logits", "similarity", "occurrence_map"), outputs):
        np.save(os.path.join(directory, name + ".npy"), t.detach().float().cpu().numpy())


def run_reference(args, rank):
    from protoasnet_b200 import synth

    if rank != 0:
        return
    dims = synth.CONFIGS[WORKLOAD]
    sd = synth.make_head_params(dims, seed=200, bias_scale=0.02, bf16_round=True)
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    fwd, kind = reference_head(dims, sd)
    sample = 128
    x = torch.from_numpy(synth.make_features(dims, 64, seed=0, bf16_round=True))
    with torch.no_grad():
        for _ in range(args.warmup):
            fwd(x)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            for _ in range(sample // 64):
                out = fwd(x)
        dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, out)
    v = args.steps * sample / dt
    what = "the reference's own Video_XProtoNet class (oracle/_ref, identity backbone)" if kind == "reference" else \
        "oracle port of the reference's ops"
    desc = f"{sample} clips per step (2 chunks of 64) of the cfg-3 batch-1024 workload, fp32, torch CPU, {cores} threads, {what}"
    print(json.dumps({
        "impl": "reference", "metric": "head_fwd_clips_per_sec", "value": v, "unit": "clips/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{WORKLOAD}: prototype head fwd, feature map 512x4x7x7, D=256 P=40 K=4", "sample": desc},
        "cpu_baseline": {"value": v, "unit": "clips/s", "cores": cores, "kind": kind, "sample": desc},
        "e2e": {"value": v, "unit": "clips/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--path", default="auto", choices=["auto", "generic", "tcgen05"])
    ap.add_argument("--push-clips", type=int, default=PUSH_CLIPS)
    ap.add_argument("--no-push", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs (rank 0) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank)
        return

    import torch.distributed as dist
    from protoasnet_b200 import _lib, synth
    from protoasnet_b200.push import push_resident

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(v):
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    lib = _lib.load()
    dims = synth.CONFIGS[WORKLOAD]
    model, sd = make_model(dims, dev, args.path)
    peaks = load_peaks()
    flops_clip, bytes_clip = flops_bytes_per_clip(dims)

    g = torch.Generator(device=dev).manual_seed(1234 + rank)
    x = torch.relu(torch.randn((BATCH, dims.C) + dims.spatial, device=dev, generator=g)).bfloat16()
    dims_struct = model._rt.make_dims(x, model.kernel_path)[0]
    tc = bool(lib.pasn_tcgen05_supported(dims_struct)) and args.path != "generic"

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()

    # ---------------- device-resident head forward ----------------
    with torch.no_grad():
        # ranks leave their set-up (imports, weights, NCCL) seconds apart: line them up BEFORE the warm-up, otherwise the early
        # ones sit idle at the timed region's barrier until their clocks have dropped, and the 20 timed steps (3.4 ms) are
        # run on a GPU that is still ramping up (2- and 4-GPU records of round 2: 216 / 248 us per step against 172 on one)
        barrier()
        for _ in range(args.warmup):
            model(x)
        l0 = lib.pasn_debug_launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for _ in range(args.steps):
            out = model(x)
        e1.record()
        barrier()
        ms_total = e0.elapsed_time(e1)
        launches = int(lib.pasn_debug_launch_count() - l0)
        last_out = out
        # dominant kernel, per launch, CUDA events recorded inside the library on the launch stream
        lib.pasn_debug_time_main_kernel(1)
        main_ms = []
        for _ in range(args.steps):
            model(x)
            main_ms.append(float(lib.pasn_debug_last_main_kernel_ms()))
        lib.pasn_debug_time_main_kernel(0)
    ms_step = max_over_ranks(ms_total / args.steps)
    value = world * BATCH / (ms_step * 1e-3)
    main_ms_avg = float(np.mean(main_ms))
    # side measurement (not the headline): the same batch handed over as a channels_last_3d tensor ([N,S,C] in memory,
    # what a channels_last bf16 backbone emits) -- the fused path gathers it with 16-byte L1-bypassing cp.async;
    # measured right after the headline loop, before the 2 s sustained loop heats the part
    channels_last = None
    if tc and rank == 0:
        xcl = x.contiguous(memory_format=torch.channels_last_3d)
        with torch.no_grad():
            for _ in range(3):
                model(xcl)
            torch.cuda.synchronize(dev)
            e0.record()
            for _ in range(args.steps):
                model(xcl)
            e1.record()
            torch.cuda.synchronize(dev)
            cl_ms = e0.elapsed_time(e1) / args.steps
            lib.pasn_debug_time_main_kernel(1)
            cl_main = []
            for _ in range(args.steps):
                model(xcl)
                cl_main.append(float(lib.pasn_debug_last_main_kernel_ms()))
            lib.pasn_debug_time_main_kernel(0)
        channels_last = {"value_one_gpu": BATCH / (cl_ms * 1e-3), "unit": "clips/s", "ms_per_step": cl_ms,
                         "kernel_ms": float(np.mean(cl_main)),
                         "frac_of_burst": BATCH * flops_clip / (cl_ms * 1e-3) / 1e12 / peaks["bf16_tflops"],
                         "frac_k1": BATCH * flops_clip / (float(np.mean(cl_main)) * 1e-3) / 1e12 / peaks["bf16_tflops"],
                         "definition": "frac_of_burst = whole-head FLOPs / ms_per_step / burst peak (step level, as roofline.frac); "
                                       "frac_k1 = same FLOPs / dominant-kernel time"}
        del xcl

    # the same step back to back for >= 2 s: the number to hold against the SUSTAINED peak (clocks / power settle)
    sustained = None
    if rank == 0:
        n_sus = int(2.2 / (ms_step * 1e-3))
        with torch.no_grad():
            torch.cuda.synchronize(dev)
            e0.record()
            for _ in range(n_sus):
                model(x)
            e1.record()
            torch.cuda.synchronize(dev)
        sus_ms = e0.elapsed_time(e1) / n_sus
        sustained = {"steps": n_sus, "seconds": e0.elapsed_time(e1) * 1e-3, "ms_per_step": sus_ms,
                     "value_one_gpu": BATCH / (sus_ms * 1e-3),
                     "frac_of_sustained_peak": BATCH * flops_clip / (sus_ms * 1e-3) / 1e12 / peaks["bf16_tflops_sustained"]}

    # ---------------- end to end through the public API with host buffers ----------------
    # protoasnet_b200.HostPipeline: pinned host batch in, pinned host logits + similarities out; the batch is cut in
    # four pieces so that the H2D copy of one piece overlaps the kernels of the previous one.  Every step copies the
    # whole batch host->device and the results device->host inside the timed region.  The plain sequence (one copy,
    # one forward call, copy back) is timed as well and reported next to it.
    from protoasnet_b200 import HostPipeline
    numa = _bind_host_memory_to_gpu_node(dev) if world > 1 else None   # N ranks copying at once: keep each batch NUMA-local
    x_host = x.cpu().pin_memory()
    lg_host = torch.empty((BATCH, dims.K), dtype=torch.float32).pin_memory()
    sm_host = torch.empty((BATCH, dims.P), dtype=torch.float32).pin_memory()
    x_dev = torch.empty_like(x)
    e2e_steps = max(3, min(args.steps, 10))
    pipe = HostPipeline(model, chunks=4)
    with torch.no_grad():
        barrier()   # (pinning the host buffers takes a different time on every rank)
        for _ in range(2):
            x_dev.copy_(x_host, non_blocking=True)
            model(x_dev)
            pipe(x_host)
        barrier()
        e0.record()
        for _ in range(e2e_steps):
            x_dev.copy_(x_host, non_blocking=True)
            logits, sim, occ = model(x_dev)
            lg_host.copy_(logits, non_blocking=True)
            sm_host.copy_(sim, non_blocking=True)
        e1.record()
        barrier()
        plain_ms = max_over_ranks(e0.elapsed_time(e1) / e2e_steps)
        e0.record()
        for _ in range(e2e_steps):
            lg_p, sm_p = pipe(x_host)
        e1.record()
        barrier()
    e2e_ms = max_over_ranks(e0.elapsed_time(e1) / e2e_steps)
    e2e = {"value": world * BATCH / (e2e_ms * 1e-3), "unit": "clips/s", "ms_per_step": e2e_ms,
           "h2d_bytes_per_step": int(x_host.numel() * 2), "d2h_bytes_per_step": int(lg_host.numel() * 4 + sm_host.numel() * 4),
           "api": "protoasnet_b200.HostPipeline(model, chunks=4)(pinned host features) -> pinned host logits + similarity",
           "h2d_gbs": x_host.numel() * 2 / (e2e_ms * 1e-3) / 1e9, "host_numa_node": numa,
           "single_copy_then_forward": {"value": world * BATCH / (plain_ms * 1e-3), "ms_per_step": plain_ms}}
    del pipe
    del x_host, x_dev

    # ---------------- push over PUSH_CLIPS clips sharded across ranks ----------------
    push = None
    if not args.no_push:
        n_total = args.push_clips
        lo, hi = synth.shard_range(n_total, rank, world)
        labels_all = synth.push_labels(n_total, dims.K - 1, seed=7)
        feats = torch.empty((hi - lo, dims.C) + dims.spatial, dtype=torch.bfloat16, device=dev)
        pos = lo
        while pos < hi:  # chunk c holds global clips [c*1000, (c+1)*1000); identical for any sharding
            c = pos // synth.PUSH_CHUNK
            gg = torch.Generator(device=dev).manual_seed(1000 + c)
            chunk = torch.relu(torch.randn((synth.PUSH_CHUNK, dims.C) + dims.spatial, device=dev, generator=gg)).bfloat16()
            a, b = pos - c * synth.PUSH_CHUNK, min(hi, (c + 1) * synth.PUSH_CHUNK) - c * synth.PUSH_CHUNK
            feats[pos - lo: pos - lo + (b - a)] = chunk[a:b]
            pos += b - a
        del chunk
        labels = torch.from_numpy(labels_all[lo:hi]).to(dev)
        proto0 = model.prototype_vectors.data.clone()
        times, idx_ref = [], None
        with torch.no_grad():
            n_warm, n_timed = 2, 5   # NCCL / allocator first-use effects last into the second push
            for it in range(n_warm + n_timed):
                model.prototype_vectors.data.copy_(proto0)
                barrier()
                e0.record()
                res = push_resident(model, feats, labels, global_offset=lo, chunk=8192, replace_prototypes=True)
                e1.record()
                barrier()
                if it >= n_warm:
                    times.append(e0.elapsed_time(e1))
                if idx_ref is None:
                    idx_ref = res["index"].clone()
                assert torch.equal(idx_ref, res["index"])
        push_ms = max_over_ranks(float(np.median(times)))
        f_push = n_total * (flops_clip - 0)  # same head FLOPs per clip (no occurrence-map store)
        push = {"seconds_per_50k": push_ms * 1e-3 * (50000 / n_total), "clips": n_total, "ms": push_ms, "n_gpus": world,
                "ms_runs_rank0": [round(t, 3) for t in times],
                "clips_per_sec": n_total / (push_ms * 1e-3), "scaling": "strong",
                "tensor_frac_of_sustained": f_push / (push_ms * 1e-3) / 1e12 / (world * peaks["bf16_tflops_sustained"]),
                "winners_sample": idx_ref[:8].tolist(),
                # the merge: one kernel over NVLink peer memory (no collective call), or one all-gather of the records
                "collectives_per_push": 0 if (world == 1 or model.__dict__.get("_pasn_peer_records")
                                              and any(v is not None for v in model.__dict__["_pasn_peer_records"].values())) else 1,
                "merge": "single GPU" if world == 1 else
                         ("one kernel over NVLink peer memory (pasn_push_merge_peers)"
                          if any(v is not None for v in model.__dict__.get("_pasn_peer_records", {}).values())
                          else "one NCCL all-gather of [key | vector] records + pasn_push_reduce")}
        model.prototype_vectors.data.copy_(proto0)
        del feats

    clocks = sampler.stop() if rank == 0 else None

    # ---------------- CPU baseline (rank 0, N == 1) ----------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cores = os.cpu_count() or 1
        v, n_clips, runs, kind = cpu_head_clips_per_sec(dims, sd, 256, 10.0, 12, cores)
        who = "the reference's own Video_XProtoNet class (oracle/_ref)" if kind == "reference" else "oracle port of the reference's ops"
        cpu = {"value": v, "unit": "clips/s", "cores": cores, "kind": kind,
               "sample": f"{n_clips} clips per run in chunks of 64 (cfg-3 shape, fp32, torch CPU, {who}), median of {runs} runs"}
        if push is not None:
            n_sample = 1000
            s50, dt = cpu_push_seconds_per_50k(dims, sd, n_sample, cores)
            push["cpu_baseline"] = {"value": s50, "unit": "s per 50k clips (extrapolated)", "cores": cores, "kind": "port",
                                    "sample": f"restated reference push loop, batch 5, {n_sample} clips in {dt:.1f} s, "
                                              "extrapolated linearly to 50 000"}

    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, last_out)

    if rank == 0:
        # whole-head algorithmic FLOPs over the time in which all of them run (the step), against the burst peak for a
        # short timed loop; the dominant kernel alone is reported as frac_k1 / kernel_ms
        achieved_tf = BATCH * flops_clip / (ms_step * 1e-3) / 1e12
        k1_tf = BATCH * flops_clip / (main_ms_avg * 1e-3) / 1e12
        timed_s = ms_step * args.steps * 1e-3
        peak = peaks["bf16_tflops"] if timed_s < 1.0 else peaks["bf16_tflops_sustained"]
        traffic, traffic_src, l2sm = None, None, None
        tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")
        if tc and os.path.exists(tpath):   # dram__bytes_read+write of the dominant kernel from the committed ncu capture
            tj = json.load(open(tpath))
            traffic, traffic_src = tj.get("dram_bytes_per_launch"), tj.get("source")
            l2sm = tj.get("l2_to_sm_bytes")
        line = {
            "metric": "head_fwd_clips_per_sec", "value": value, "unit": "clips/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": f"{WORKLOAD}: video prototype head fwd, batch {BATCH} per GPU, feature map 512x4x7x7 bf16 "
                                   "(NCDHW), D=256 P=40 K=4, weights bf16-rounded, fp32 accumulate",
                       "batch_per_gpu": BATCH, "layout": "NCDHW", "kernel_path": "tcgen05" if tc else "generic",
                       "l2": "input 205 MB per step > 126 MB L2: re-read from HBM every step"},
            "roofline": {"bound": "tensor", "achieved": achieved_tf, "peak": peak, "unit": "TFLOP/s",
                         "frac": achieved_tf / peak, "traffic": traffic, "traffic_source": traffic_src,
                         "traffic_algorithmic_bytes": BATCH * bytes_clip,
                         "peak_source": f"MEASURED_PEAKS.json ({peaks['source']}), "
                                        + ("burst" if timed_s < 1.0 else "sustained"),
                         "definition": "whole-head algorithmic FLOPs / ms_per_step / peak (step level); "
                                       "frac_k1 = same FLOPs / dominant-kernel time",
                         "frac_of_sustained": achieved_tf / peaks["bf16_tflops_sustained"],
                         "frac_k1": k1_tf / peak, "kernel_ms": main_ms_avg, "algorithmic_flop_per_clip": flops_clip,
                         "hbm_gbs": BATCH * bytes_clip / (ms_step * 1e-3) / 1e9,
                         "hbm_frac": BATCH * bytes_clip / (ms_step * 1e-3) / 1e9 / peaks["hbm_gbs"],
                         # what the dominant kernel actually leans on besides the tensor pipe (DESIGN.md section 7): every SM
                         # re-streams the layer weights for each 128-voxel tile, L2 -> SM bytes per launch from the same ncu
                         # capture as `traffic`, over the kernel's live duration and the SM clock sampled during the run
                         "l2_to_sm": None if not (l2sm and clocks and clocks.get("sm_mhz")) else {
                             "bytes_per_launch": l2sm, "bytes_per_clk": l2sm / (main_ms_avg * 1e-3 * clocks["sm_mhz"] * 1e6),
                             "fabric_limit_bytes_per_clk": 6300,
                             "frac": l2sm / (main_ms_avg * 1e-3 * clocks["sm_mhz"] * 1e6) / 6300.0}},
            "sustained": sustained,
            "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": launches, "clocks": clocks, "push": push,
            "channels_last": channels_last,
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
