"""Wall-clock time of push_prototypes over a data loader, with a save directory (prototypes_info.pickle written), under
torchrun at 1 / 2 / 4 / 8 ranks: this tree against another checkout (--parent, e.g. the parent commit, built), the two
alternating in one job.  Prints the card and its power limit first, then per run the seconds per push (slowest rank,
device synchronised before and after each push) and the clips / batches each rank fetched from the dataset.
``--backend gloo`` runs the ranks on gloo, sharing the node's GPUs round-robin (the merge then takes the all-gather,
PASN_PUSH_PEER=0): on a node with fewer GPUs than ranks it still shows how loading divides among the ranks.

The dataset is map-style: seeded config-3 feature maps ([512,4,7,7], relu(N(0,1)) rounded to bf16; 1024 distinct maps,
item i = map i % 1024), handed out as fp32 because the pickle stores the input clip as a numpy array and numpy has no
bf16.  The backbone is a FeatureInput that passes the map to the head as bf16, so the head runs in bf16 mode.
``--item-ms`` adds a fixed CPU cost per item, a stand-in for the .mat decoding of the reference's loader.

    python tools/time_push_loader.py --parent ../parent_checkout [--worlds 1 2 4 8] [--clips 4096] [--batch 64]
                                     [--item-ms 0.25] [--pushes 2] [--reps 1] [--backend nccl] [--out report.txt]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

HERE = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _worker(a):
    import torch
    import torch.distributed as dist

    import protoasnet_b200 as pasn
    from protoasnet_b200 import push as pushmod
    from protoasnet_b200 import synth

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")) % torch.cuda.device_count())
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group(a.backend, device_id=dev if a.backend == "nccl" else None)
    dims = synth.CONFIGS["cfg3_video_b1024"]

    class BF16Input(pasn.FeatureInput):
        def forward(self, x):
            return x.bfloat16()

    class MapSet(torch.utils.data.Dataset):
        def __init__(self, n):
            self.n, self.fetched = n, 0
            self.maps = torch.from_numpy(synth.make_features(dims, 1024, seed=5, bf16_round=True)).bfloat16()
            self.labels = torch.from_numpy(synth.push_labels(n, dims.K - 1, seed=7))

        def __len__(self):
            return self.n

        def __getitem__(self, i):
            self.fetched += 1
            t_end = time.perf_counter() + a.item_ms * 1e-3
            while time.perf_counter() < t_end:      # fixed per-item CPU cost (decoding stand-in)
                pass
            return {"cine": self.maps[i % 1024].float(), "target_AS": self.labels[i], "filename": f"clip_{i}"}

    sd = synth.make_head_params(dims, seed=200, bias_scale=0.02, bf16_round=True)
    m = pasn.construct_Video_XProtoNet(BF16Input(dims.C), pretrained=False, prototype_shape=dims.prototype_shape,
                                       num_classes=dims.K)
    m.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()})
    m = m.to(dev).eval()
    ds = MapSet(a.clips)
    loader = torch.utils.data.DataLoader(ds, batch_size=a.batch, pin_memory=True)
    times, fetched = [], []
    with tempfile.TemporaryDirectory() as tmp:
        for it in range(a.pushes + 1):            # push 0 warms up (weight packing, peer memory, NCCL communicators)
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            ds.fetched = 0
            t0 = time.perf_counter()
            pushmod.push_prototypes(loader, m, root_dir_for_saving_prototypes=tmp, epoch_number=it, log=lambda *x: None,
                                    replace_prototypes=False)
            torch.cuda.synchronize()
            if it > 0:
                times.append(time.perf_counter() - t0)
                fetched.append(ds.fetched)
        files = sorted(os.listdir(os.path.join(tmp, f"epoch-{a.pushes}")))
    mine = {"rank": rank, "times": times, "fetched": fetched, "files": files}
    every = [None] * world
    if world > 1:
        dist.all_gather_object(every, mine)
        dist.destroy_process_group()
    else:
        every = [mine]
    if rank == 0:
        print("RESULT " + json.dumps({
            "world": world, "push_s": [max(r["times"][i] for r in every) for i in range(a.pushes)],
            "fetched_per_rank": [r["fetched"][-1] for r in every],
            "files_per_rank": [r["files"] for r in every]}), flush=True)


def _run(tree, world, a):
    env = dict(os.environ, PYTHONPATH=tree)
    if a.backend == "gloo":
        env["PASN_PUSH_PEER"] = "0"
    cmd = [sys.executable, "-m", "torch.distributed.run", "--standalone", f"--nproc_per_node={world}",
           os.path.abspath(__file__), "--worker", "--clips", str(a.clips), "--batch", str(a.batch),
           "--item-ms", str(a.item_ms), "--pushes", str(a.pushes), "--backend", a.backend]
    r = subprocess.run(cmd, env=env, capture_output=True, text=True, cwd=tree)
    for line in r.stdout.splitlines():
        if line.startswith("RESULT "):
            return json.loads(line[7:])
    raise RuntimeError(f"{tree} at {world} ranks failed (exit {r.returncode}):\n{r.stdout[-3000:]}\n{r.stderr[-6000:]}")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--worker", action="store_true")
    ap.add_argument("--parent", default=None, help="another built checkout to time in alternation with this one")
    ap.add_argument("--worlds", type=int, nargs="+", default=[1, 2, 4, 8])
    ap.add_argument("--clips", type=int, default=4096)
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--item-ms", type=float, default=0.25)
    ap.add_argument("--pushes", type=int, default=2)
    ap.add_argument("--reps", type=int, default=1)
    ap.add_argument("--backend", default="nccl", choices=["nccl", "gloo"])
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if a.worker:
        return _worker(a)
    import torch
    ngpu = torch.cuda.device_count()
    if ngpu == 0:
        raise SystemExit("time_push_loader needs CUDA devices")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    lines = [f"cards ({ngpu}): " + ("; ".join(sorted(set(q))) if q else torch.cuda.get_device_name()) +
             f"; {os.cpu_count()} host cores",
             f"push_prototypes with a save directory: {a.clips} clips of config 3 (bf16 head), batch {a.batch} "
             f"({-(-a.clips // a.batch)} batches), {a.item_ms} ms CPU per item, pin_memory, no workers; "
             f"{a.pushes} timed pushes after one warm-up push per launch; {a.backend} ranks"
             + (" sharing the GPUs round-robin" if a.backend == "gloo" else "")]
    trees = [("this tree", HERE)] + ([("parent", os.path.abspath(a.parent))] if a.parent else [])
    print("\n".join(lines), flush=True)
    for rep in range(a.reps):
        for world in [w for w in a.worlds if w <= ngpu or a.backend == "gloo"]:
            for lab, tree in trees:
                r = _run(tree, world, a)
                files = sorted({f for fs in r["files_per_rank"] for f in fs})
                line = (f"{lab:9s} R={world}: push " + ", ".join(f"{t:.3f}" for t in r["push_s"]) + " s | clips fetched "
                        f"per rank {r['fetched_per_rank']} (batches {[-(-c // a.batch) for c in r['fetched_per_rank']]}) | "
                        f"files {files}")
                print(line, flush=True)
                lines.append(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
