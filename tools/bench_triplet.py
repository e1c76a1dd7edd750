"""Timing of the triplet fine-tuning step at the reference's training shape (src/config/train_triplet.yaml: train_bs 8,
clips trimmed to 10 s): three forwards + TripletMarginLoss + all parameter gradients in one C-ABI call.

``--train-conv``: the conv feature encoder trained too (freeze_convnet: False) against the frozen step, the two
alternated on the same inputs, plus a torch.profiler breakdown of the conv-encoder gradient kernels of one step."""
import json, os, subprocess, sys, time
import torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from nomad_b200.engine import Engine
from nomad_b200.triplet import triplet_loss_and_grads
from nomad_b200.weights import flops_embed, random_state_dict

SHAPES = ((8, 10), (8, 4), (32, 2))


def frozen():
    sd = random_state_dict(1234)
    eng = Engine(sd, 0)
    out = []
    for B, secs in SHAPES:
        N = 16000 * secs
        g = torch.Generator().manual_seed(0)
        A, P, Nn = (0.1 * torch.randn(B, N, generator=g) for _ in range(3))
        A, P, Nn = A.cuda(), P.cuda(), Nn.cuda()
        for _ in range(2):
            triplet_loss_and_grads(eng, sd, A, P, Nn)
        torch.cuda.synchronize()
        n0 = eng.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(5):
            lib_loss, _ = triplet_loss_and_grads(eng, sd, A, P, Nn)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / 5
        # forward of 3B utterances + dgrad + wgrad of everything after the conv encoder (conv: forward only)
        t = eng.num_frames(N)
        conv = 2.0 * (5120 * ((N - 10) // 5 + 1)) + 0  # conv0 only term of F(N); the rest of the conv stack below
        fwd = flops_embed(N)
        enc = 786432.0 * t + 9437184.0 * t + 12.0 * (4718592.0 * t + 9437184.0 * t + 3072.0 * t * t) + 393216.0
        flops = 3 * B * (fwd + 2.0 * enc)
        out.append({"B": B, "seconds": secs, "frames_per_utt": t, "ms_per_step": ms, "launches_per_step": (eng.launch_count() - n0) // 5,
                    "tflops_algorithmic": flops / (ms / 1e3) / 1e12, "triplets_per_s": B / (ms / 1e3)})
    print(json.dumps({"config": "triplet step: 3B forwards + TripletMarginLoss + all parameter gradients (conv encoder frozen), "
                                "flops = 3B * (F(N) + 2 * F_encoder(N))", "results": out}))


def conv_wgrad_flops(N):
    """Algorithmic FLOPs of the conv1-6 weight gradients of one utterance: 2 * 512 * 512 k * T_l over the valid rows."""
    T, f = (N - 10) // 5 + 1, 0.0
    for k in (3, 3, 3, 3, 2, 2):
        T = (T - k) // 2 + 1
        f += 2.0 * 512 * 512 * k * T
    return f


def train_conv():
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()[0]
    sd = random_state_dict(1234)
    eng = Engine(sd, 0)
    out = []
    for B, secs in SHAPES:
        N = 16000 * secs
        g = torch.Generator().manual_seed(0)
        A, P, Nn = ((0.1 * torch.randn(B, N, generator=g)).cuda() for _ in range(3))
        step = {"frozen": lambda: triplet_loss_and_grads(eng, sd, A, P, Nn),
                "conv": lambda: triplet_loss_and_grads(eng, sd, A, P, Nn, freeze_convnet=False, feature_grad_mult=0.1)}
        for fn in step.values():
            for _ in range(2):
                fn()
        times, launches = {k: [] for k in step}, {}
        for _ in range(4):   # alternate the two modes: the spread of each is measured against the same background
            for mode, fn in step.items():
                torch.cuda.synchronize()
                n0 = eng.launch_count()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(5):
                    fn()
                e1.record()
                torch.cuda.synchronize()
                times[mode].append(e0.elapsed_time(e1) / 5)
                launches[mode] = (eng.launch_count() - n0) // 5
        # kernel breakdown of one conv-training step (separate from the timed runs: tracing slows the host)
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            step["conv"]()
            torch.cuda.synchronize()
        ev = sorted((e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and e.device_time > 0),
                    key=lambda e: e.time_range.start)
        part = {"wgrad_gemm_ms": 0.0, "wgrad_transpose_ms": 0.0, "wgrad_reduce_ms": 0.0, "conv0_groupnorm_ms": 0.0}
        pending = 0.0   # GEMM time since the last transpose: the wgrad GEMM when a reduce follows
        for e in ev:
            us = e.device_time / 1e3
            if "conv_wgrad_transpose" in e.name:
                part["wgrad_transpose_ms"] += us
                pending = 0.0
            elif "conv_wgrad_reduce" in e.name:
                part["wgrad_reduce_ms"] += us
                part["wgrad_gemm_ms"] += pending
                pending = 0.0
            elif "gemm" in e.name.lower() or "tc_kernel" in e.name.lower():
                pending += us
            elif "conv0_wgrad_stats" in e.name or "conv0_param_grad" in e.name:
                part["conv0_groupnorm_ms"] += us
        fl = 3 * B * conv_wgrad_flops(N)
        med = {k: sorted(v)[len(v) // 2] for k, v in times.items()}
        out.append({"B": B, "seconds": secs, "ms_frozen": med["frozen"], "ms_conv": med["conv"],
                    "ms_frozen_all": times["frozen"], "ms_conv_all": times["conv"],
                    "extra_ms": med["conv"] - med["frozen"], "launches_frozen": launches["frozen"],
                    "launches_conv": launches["conv"], "conv_wgrad_gemm_flops": fl,
                    "conv_wgrad_gemm_tflops": fl / (part["wgrad_gemm_ms"] / 1e3) / 1e12 if part["wgrad_gemm_ms"] else None,
                    **part})
    print(json.dumps({"config": "triplet step, conv feature encoder frozen vs trained (feature_grad_mult 0.1), alternated; "
                                "ms = median of 4 x 5 steps; kernel breakdown from torch.profiler on one separate step; "
                                "conv_wgrad_gemm_flops = 3B * sum_l 2 * 512 * 512 k_l * T_l (valid rows)",
                      "gpu": gpu, "results": out}))


if __name__ == "__main__":
    train_conv() if "--train-conv" in sys.argv[1:] else frozen()
