"""One fine-tuning step written as ordinary PyTorch -- ``TripletMarginLoss(model(a), model(p), model(n))``, ``backward()``,
``torch.optim.Adam`` on ``nomad.model.parameters()`` -- against the fused ``TripletTrainer.step`` (one C call for the
three forwards, the loss and every parameter gradient), alternated in one process at the reference's training shape
(8 triplets x 10 s) and two shorter ones, with the conv feature encoder frozen and trained.

Reports ms/step (CUDA events around whole steps, each ending in the loss read-back), kernel launches per step and the
saved-buffer memory held between the forwards and the backward (three save-mode forwards).  ``--profile DIR``: a
torch.profiler table of one autograd step per configuration of ``--shape`` (a separate run: tracing slows the host)."""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from nomad_b200 import _lib  # noqa: E402
from nomad_b200.nomad import Nomad  # noqa: E402
from nomad_b200.triplet import TripletTrainer  # noqa: E402
from nomad_b200.weights import random_state_dict  # noqa: E402

SHAPES = ((8, 10), (8, 4), (32, 2))
LR = 1e-5
MARGIN = 0.2


def _setup(sd, conv):
    a = Nomad(state_dict=sd, keep_state_dict=True)
    a.model.requires_grad_()
    if not conv:
        for k, p in a.model.named_parameters():
            if "feature_extractor" in k:
                p.requires_grad_(False)
    opt = torch.optim.Adam(a.model.parameters(), lr=LR, fused=True)
    b = Nomad(state_dict=sd, keep_state_dict=True)
    tr = TripletTrainer(b, lr=LR, margin=MARGIN, lr_pretrained=LR, freeze_convnet=not conv)
    loss_fn = torch.nn.TripletMarginLoss(margin=MARGIN)

    def autograd_step(A, P, N):
        opt.zero_grad(set_to_none=True)
        loss = loss_fn(a.model(A), a.model(P), a.model(N))
        loss.backward()
        opt.step()
        return float(loss.item())

    return a, autograd_step, b, (lambda A, P, N: tr.step(A, P, N))


def _time(fn, eng, args, reps):
    torch.cuda.synchronize()
    n0 = eng.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn(*args)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps, (eng.launch_count() - n0) // reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=4)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--profile", default=None)
    ap.add_argument("--shape", default="8x10")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()[0]
    sd = random_state_dict(1234)
    lib = _lib.load()
    results = []
    shapes = SHAPES if args.profile is None else [tuple(int(x) for x in args.shape.split("x"))]
    for B, secs in shapes:
        N = 16000 * secs
        g = torch.Generator().manual_seed(0)
        A, P, Nn = ((0.1 * torch.randn(B, N, generator=g)).cuda() for _ in range(3))
        for conv in (False, True):
            a, step_a, b, step_b = _setup(sd, conv)
            for _ in range(2):   # warm-up: module loads, allocator growth, the trainer's first refresh
                step_a(A, P, Nn)
                step_b(A, P, Nn)
            if args.profile is not None:
                from torch.profiler import ProfilerActivity, profile
                with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
                    step_a(A, P, Nn)
                    torch.cuda.synchronize()
                os.makedirs(args.profile, exist_ok=True)
                path = os.path.join(args.profile, f"r06_profile_autograd_{B}x{secs}s_{'conv' if conv else 'frozen'}.txt")
                with open(path, "w") as f:
                    f.write(f"# {gpu}; one autograd step, B={B} x {secs} s, conv encoder {'trained' if conv else 'frozen'}\n")
                    f.write(prof.key_averages().table(sort_by="cuda_time_total", row_limit=40))
                print("wrote", path)
                continue
            ta, tb = [], []
            for _ in range(args.rounds):
                ms, la = _time(step_a, a.engine, (A, P, Nn), args.reps)
                ta.append(ms)
                ms, lb = _time(step_b, b.engine, (A, P, Nn), args.reps)
                tb.append(ms)
            flags = _lib.SAVE_PARAMS | (_lib.SAVE_CONV if conv else 0)
            saved = 3 * lib.nomad_b200_layers_saved_bytes_ex(B, N, flags)
            row = {"B": B, "seconds": secs, "conv_trained": conv, "autograd_ms": sorted(ta)[len(ta) // 2],
                   "trainer_ms": sorted(tb)[len(tb) // 2], "autograd_ms_all": ta, "trainer_ms_all": tb,
                   "autograd_launches_per_step": la, "trainer_launches_per_step": lb,
                   "saved_buffers_gb_per_step": saved / 1e9}
            row["ratio"] = row["autograd_ms"] / row["trainer_ms"]
            print(json.dumps(row), flush=True)
            results.append(row)
            del a, b, step_a, step_b
            torch.cuda.empty_cache()
    if args.profile is None:
        out = {"gpu": gpu, "config": "autograd: TripletMarginLoss(model(a), model(p), model(n)) + backward + fused Adam on "
                                     "nomad.model.parameters(); trainer: TripletTrainer.step; lr 1e-5, margin 0.2; "
                                     "median of rounds, each round = reps steps of one then reps of the other",
               "results": results}
        print(json.dumps(out))
        if args.out:
            with open(args.out, "w") as f:
                json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
