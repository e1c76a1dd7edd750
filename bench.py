#!/usr/bin/env python
"""Benchmark of the NOMAD scoring hot path on B200 (BASELINE.json configs[1]: "batch embedding: 256 x 4 s synthetic
16 kHz clips, wav2vec2-base NOMAD head"), with the scoring tail (distance rows against a resident 1 k NMR set).

    python bench.py --gpus N --steps K --warmup W            # this framework (CUDA, C ABI)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU arithmetic (oracle port)
    python bench.py --impl library ...                       # the reference's arithmetic as torch library kernels
                                                             # (cuDNN / cuBLAS TF32 + SDPA) on the same B200
    python bench.py ... --dump-outputs DIR                   # also write the results of the last timed step as
                                                             # DIR/{emb,dm,mean}.npy (rank 0; inputs are seeded)

One "step" (every N) = one pass of the hot path over one batch per GPU: 256 synthetic 4-second clips -> wav2vec 2.0
base -> NOMAD embedding -> distance rows + row means against the (M, 256) NMR embeddings resident on every rank
(``nomad_b200_score``).  With N > 1 (torchrun, one process per GPU, NCCL) the step ends with the path's exchange:
every rank sends its row means and matrix rows to rank 0 (point-to-point in the NCCL communicator, exact sizes; the
matrix is never all-gathered).  Per-GPU work is fixed as N grows ("weak").  The NMR set is embedded sharded and
all-gathered ONCE before the timed region (that is when `Nomad.predict` does it); its time is reported separately.

Rank 0 prints ONE JSON line:

* ``value``   : utterance-seconds embedded per second, whole job, waveforms resident in HBM, CUDA-event timed, max over
                ranks.
* ``e2e``     : same step through ``nomad_b200_score_host`` with pinned HOST buffers: H2D of the waveforms, D2H of
                embeddings + matrix rows + means inside the timed region (row-sharded host results per rank).
* ``roofline``: the dominant kernel class (tcgen05 GEMM) timed in situ with one CUDA-event pair per launch on the
                launching stream; achieved = sum(2MNK) / sum(duration), against the measured sustained tensor peak.
* ``sharded_c3`` : BASELINE configs[2] as a FIXED global workload (strong scaling): C3_DEG variable-length (1-20 s)
                degraded utterances vs C3_NMR NMR utterances through ``nomad_b200.dist.score_sharded`` -- LPT shard ->
                embed NMR shard -> NCCL all-gather -> embed degraded shard -> row-slice cdist + means -> rows to rank 0.
* ``pairwise``: BASELINE configs[4] slice, fixed global PAIR_N x PAIR_M (strong scaling): rows sharded, means to rank 0.
* ``loss``    : BASELINE configs[3] (N = 1 only; the loss lives inside a user's training step: replicas).
* ``cpu_baseline`` / ``parity``: the oracle on the host cores over a bounded sample of the same batch, and the achieved
                embedding error of this library against it on those clips.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "utterance-seconds embedded per second"
UNIT = "utt-s/s"
CLIPS = 256
CLIP_SECONDS = 4
SR = 16000
NMR_M = 1000
WORKLOAD = ("configs[1]: batch embedding, 256 x 4 s synthetic 16 kHz clips, wav2vec2-base + NOMAD head, scored against "
            "1000 resident NMR embeddings")
CPU_SAMPLE_CLIPS = 16
C3_DEG, C3_NMR = 4096, NMR_M          # fixed global workload of the strong-scaling leg
PAIR_N, PAIR_M = 800_000, NMR_M       # fixed global workload of the pairwise leg (1e5 x 1e3 per GPU at N = 8)
LOSS_B, LOSS_SECONDS = 32, 2
FALLBACK_PEAK_TFLOPS = 1400.0  # B200_PROFILING.md: sustained ~1.4 PFLOP/s (burst fallback 1590)
FALLBACK_HBM_GBS = 6500.0
# dram__bytes_read.sum + dram__bytes_write.sum per tensor-core GEMM launch, averaged over the GEMM launches of one
# step, from the ncu pass named in TRAFFIC_SOURCE (not measured in this run; the algorithmic operand + result bytes of
# those launches are 33.7 GB per step, see DESIGN.md section 4)
GEMM_DRAM_TRAFFIC_BYTES = 559.7e6
TRAFFIC_SOURCE = "ncu profile profiles/r02c_gemm_dram.csv (30.8 GB over the 55 GEMM launches of one step)"


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def synth_batch(clips: int, seed: int):
    import torch
    g = torch.Generator().manual_seed(seed)
    return 0.1 * torch.randn(clips, CLIP_SECONDS * SR, generator=g)


def shared_config(weights: str):
    """The SAME dict in every arm (ours / reference / library), so the driver's same_config check can hold."""
    return {"workload": WORKLOAD, "clips_per_gpu_per_step": CLIPS, "clip_seconds": CLIP_SECONDS, "frames_per_clip": 199,
            "nmr_embeddings": NMR_M, "weights": weights,
            "parallelism": "dp over utterances (one 256-clip batch per GPU); NMR embeddings all-gathered once (NCCL) before "
                           "the timed region; per step every rank sends its row means + matrix rows to rank 0",
            "l2": "per-step working set ~6 GB of activations >> 126 MB L2 (inputs larger than L2, no explicit flush)",
            "reference_arm": f"CPU arms time a bounded sample of this workload per step ({CPU_SAMPLE_CLIPS} of the {CLIPS} "
                             "clips, same seed) and report the same per-utterance-second metric"}


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled every 200 ms while the timed region runs."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.rows = []
        self.proc = None
        self.gpu = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception as e:  # pragma: no cover
            log("clock sampler unavailable:", e)

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 9:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        busy = [x for x in sm if x > 0.5 * (max(mx) if mx else 1)] or sm
        return {"sm_mhz": statistics.median(busy) if busy else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def cpu_reference_rate(steps: int, warmup: int, min_seconds: float = 0.0):
    """Oracle port on the host cores: `steps` passes over the first CPU_SAMPLE_CLIPS clips of rank 0's batch, each
    followed by the scoring tail.  -> (utt-s/s, ms/step, cores, passes, embeddings of the sample)"""
    import torch

    from nomad_b200.weights import random_state_dict
    from oracle import w2v_oracle as O  # CPU baseline leg: the one place bench.py may execute oracle/
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    sd = random_state_dict(1234)
    wav = synth_batch(CLIPS, 0)[:CPU_SAMPLE_CLIPS].contiguous()
    g = torch.Generator().manual_seed(4242)
    nmr = torch.nn.functional.normalize(torch.randn(NMR_M, 256, generator=g), dim=1).numpy()
    emb = None
    with torch.no_grad():
        for _ in range(warmup):
            O.embed(sd, wav)
        times = []
        t_all = time.perf_counter()
        i = 0
        while i < steps or (time.perf_counter() - t_all) < min_seconds:
            t0 = time.perf_counter()
            emb = O.embed(sd, wav)
            O.cdist_mean(emb.numpy(), nmr)
            times.append(time.perf_counter() - t0)
            i += 1
    sec = sum(times) / len(times)
    return CPU_SAMPLE_CLIPS * CLIP_SECONDS / sec, sec * 1e3, cores, len(times), emb


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    steps = max(1, args.steps)
    rate, ms, cores, n, _ = cpu_reference_rate(steps, min(args.warmup, 1))
    sample = (f"{CPU_SAMPLE_CLIPS} x {CLIP_SECONDS} s clips per step (1/16 of the 256-clip batch, same seed) + their distance "
              f"rows against {NMR_M} NMR embeddings; oracle port of the reference's torch-CPU fp32 path (the reference itself "
              f"needs fairseq, absent here), {cores} threads")
    line = {
        "impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": args.gpus, "steps": n,
        "warmup": min(args.warmup, 1), "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": shared_config("random-init(seed=1234)"),
        "cpu_baseline": {"value": rate, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)
    return 0


# ----------------------------------------------------------------------------------------------------------------------
# library arm: the reference's arithmetic dispatched to the vendor libraries on the same GPU (SURVEY.md 8d: "the
# existing Blackwell path" -- cuDNN convs, cuBLAS TF32 GEMMs, fused SDPA attention).  Plain torch ops, none of this
# repo's kernels.
def library_embed(sd, wav):
    import torch
    import torch.nn.functional as F
    P = "ssl_model."
    x = wav.unsqueeze(1)
    for i, (k, s) in enumerate(zip((10, 3, 3, 3, 3, 2, 2), (5, 2, 2, 2, 2, 2, 2))):
        x = F.conv1d(x, sd[P + f"feature_extractor.conv_layers.{i}.0.weight"], stride=s)
        if i == 0:
            x = F.group_norm(x, 512, sd[P + "feature_extractor.conv_layers.0.2.weight"],
                             sd[P + "feature_extractor.conv_layers.0.2.bias"], eps=1e-5)
        x = F.gelu(x)
    x = x.transpose(1, 2)
    x = F.layer_norm(x, (512,), sd[P + "layer_norm.weight"], sd[P + "layer_norm.bias"], 1e-5)
    x = F.linear(x, sd[P + "post_extract_proj.weight"], sd[P + "post_extract_proj.bias"])
    B, T, Cc = x.shape
    pc = F.conv1d(x.transpose(1, 2), sd["_pos_w"], sd[P + "encoder.pos_conv.0.bias"], padding=64, groups=16)[..., :T]
    x = x + F.gelu(pc).transpose(1, 2)
    x = F.layer_norm(x, (Cc,), sd[P + "encoder.layer_norm.weight"], sd[P + "encoder.layer_norm.bias"], 1e-5)
    for l in range(12):
        q_ = P + f"encoder.layers.{l}."
        lin = lambda t, n: F.linear(t, sd[q_ + n + ".weight"], sd[q_ + n + ".bias"])
        q = lin(x, "self_attn.q_proj").view(B, T, 12, 64).transpose(1, 2)
        k = lin(x, "self_attn.k_proj").view(B, T, 12, 64).transpose(1, 2)
        v = lin(x, "self_attn.v_proj").view(B, T, 12, 64).transpose(1, 2)
        a = F.scaled_dot_product_attention(q, k, v).transpose(1, 2).reshape(B, T, Cc)
        x = F.layer_norm(x + lin(a, "self_attn.out_proj"), (Cc,), sd[q_ + "self_attn_layer_norm.weight"],
                         sd[q_ + "self_attn_layer_norm.bias"], 1e-5)
        h = lin(F.gelu(lin(x, "fc1")), "fc2")
        x = F.layer_norm(x + h, (Cc,), sd[q_ + "final_layer_norm.weight"], sd[q_ + "final_layer_norm.bias"], 1e-5)
    e = F.linear(F.relu(x.mean(1)), sd["embedding_layer.1.weight"], sd["embedding_layer.1.bias"])
    return F.normalize(e, dim=1)


def run_library(args):
    import torch

    from nomad_b200.weights import fold_pos_conv_weight, random_state_dict
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    torch.backends.cuda.matmul.allow_tf32 = True
    torch.backends.cudnn.allow_tf32 = True
    dev = torch.device("cuda", 0)
    sd_cpu = random_state_dict(1234)
    sd = {k: v.to(dev) for k, v in sd_cpu.items()}
    sd["_pos_w"] = fold_pos_conv_weight(sd_cpu).to(dev)
    wav_pin = synth_batch(CLIPS, 0).pin_memory()
    wav_dev = wav_pin.to(dev)
    g = torch.Generator().manual_seed(4242)
    nmr = torch.nn.functional.normalize(torch.randn(NMR_M, 256, generator=g), dim=1).to(dev)
    emb_pin = torch.empty((CLIPS, 256)).pin_memory()
    dm_pin = torch.empty((CLIPS, NMR_M)).pin_memory()

    def step_dev():
        with torch.no_grad():
            e = library_embed(sd, wav_dev)
            d = torch.cdist(e, nmr)
            return e, d, d.mean(1)

    def step_host():
        with torch.no_grad():
            w = wav_pin.to(dev, non_blocking=True)
            e = library_embed(sd, w)
            d = torch.cdist(e, nmr)
            emb_pin.copy_(e, non_blocking=True)
            dm_pin.copy_(d, non_blocking=True)
            torch.cuda.synchronize()

    def timed(fn, steps):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / steps

    for _ in range(max(3, args.warmup)):
        step_dev()
    step_host()
    sampler = ClockSampler(0)
    sampler.start()
    time.sleep(0.3)
    ms = timed(step_dev, args.steps)
    e2e_ms = timed(step_host, args.steps)
    clocks = sampler.stop()
    utt_s = CLIPS * CLIP_SECONDS
    line = {"impl": "library", "metric": METRIC, "value": utt_s / (ms / 1e3), "unit": UNIT, "n_gpus": 1, "steps": args.steps,
            "warmup": max(3, args.warmup), "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "tf32", "data": "synthetic", "config": shared_config("random-init(seed=1234)"),
            "library": "torch eager on cuda:0: cuDNN conv1d, cuBLAS TF32 linears, fused scaled_dot_product_attention, "
                       "torch.cdist; fp32 storage",
            "e2e": {"value": utt_s / (e2e_ms / 1e3), "unit": UNIT, "h2d_bytes_per_step": int(CLIPS * CLIP_SECONDS * SR * 4),
                    "d2h_bytes_per_step": int(CLIPS * 256 * 4 + CLIPS * NMR_M * 4)},
            "clocks": clocks}
    print(json.dumps(line), flush=True)
    return 0


# ----------------------------------------------------------------------------------------------------------------------
def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    from nomad_b200 import _lib
    from nomad_b200 import dist as nd
    from nomad_b200.engine import Engine
    from nomad_b200.nomad import plan_batches
    from nomad_b200.weights import flops_embed, load_state_dict

    # stdout carries exactly ONE JSON line: anything a library prints there meanwhile (NCCL's version banner on the
    # first collective) goes to stderr instead
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    rank, world, local = nd.init_from_env("nccl")
    if world != args.gpus:
        log(f"warning: --gpus {args.gpus} but WORLD_SIZE={world}; using WORLD_SIZE")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    sd, source = load_state_dict(None, 1234)
    eng = Engine(sd, local)
    lib = _lib.load()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        """K steps bracketed by barrier + sync; device time via CUDA events; max over ranks."""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    # ------------------------------------------------------------------ configs[2] slice: fixed global workload, sharded
    # every rank derives the same lengths; utterance i's samples are a slice of a shared noise bank (content does not
    # change the arithmetic performed; identical on every N so the scores can be compared across N)
    rng = np.random.default_rng(0)
    deg_len = (SR * rng.uniform(1.0, 20.0, size=C3_DEG)).astype(np.int64)
    nmr_len = (SR * rng.uniform(1.0, 20.0, size=C3_NMR)).astype(np.int64)
    bank = (0.1 * torch.randn(64, 20 * SR, generator=torch.Generator().manual_seed(99))).to(dev)
    max_batch_samples = 2000 * SR

    def embed_from_bank(lengths, salt):
        def fn(idx):
            out = torch.empty((len(idx), 256), dtype=torch.float32, device=dev)
            lens = [int(lengths[i]) for i in idx]
            for b in plan_batches(lens, max_batch_samples):
                wav = torch.cat([bank[(idx[j] + salt) % 64, : lens[j]] for j in b])
                off = Engine.offsets([lens[j] for j in b])
                out[torch.as_tensor(b, device=dev)] = eng.embed_packed(wav, off)
            return out
        return fn

    cdist_fn = lambda a, b, wm: eng.cdist_mean(a, b, wm)
    c3_res = {}

    def c3_pass():
        res = nd.score_sharded(nmr_len.tolist(), embed_from_bank(nmr_len, 7), deg_len.tolist(), embed_from_bank(deg_len, 0),
                               cdist_fn, dev, matrix="root")
        c3_res.update(res)
        if rank == 0:  # the consumer reads the means on the host (D2H inside the timed region)
            c3_res["mean_host"] = res["mean"].cpu()

    c3_pass()  # warm-up (NCCL communicators, workspaces)
    c3_ms = timed(c3_pass, 2) / 2
    nmr_emb = c3_res["nmr"].contiguous()  # (C3_NMR, 256) on every rank, listing order: the resident NMR set below
    c3_utt_s = float(deg_len.sum() + nmr_len.sum()) / SR
    c3_flops = float(sum(flops_embed(int(n)) for n in deg_len) + sum(flops_embed(int(n)) for n in nmr_len))
    c3_check = float(c3_res["mean_host"].double().mean()) if rank == 0 else None
    # the exchange on its own: all-gather of the NMR shards, and the rows-to-root transfer of one step
    nmr_shards = nd.shard_by_cost(nmr_len.tolist(), world)
    local_nmr = nmr_emb[torch.as_tensor(nmr_shards[rank], device=dev)].contiguous()
    for _ in range(3):
        nd.all_gather_shards(local_nmr, nmr_shards)
    allgather_ms = timed(lambda: nd.all_gather_shards(local_nmr, nmr_shards), 20) / 20

    # ------------------------------------------------------------------ primary: configs[1] batch per GPU + scoring tail
    N = CLIP_SECONDS * SR
    wav_cpu = synth_batch(CLIPS, seed=rank)
    off = np.arange(CLIPS + 1, dtype=np.int64) * N
    wav_dev = wav_cpu.reshape(-1).to(dev)
    wav_pin = wav_cpu.reshape(-1).pin_memory()
    wav_pin_np = wav_pin.numpy()
    emb_pin = torch.empty((CLIPS, 256), dtype=torch.float32).pin_memory()
    dm_pin = torch.empty((CLIPS, NMR_M), dtype=torch.float32).pin_memory()
    mean_pin = torch.empty((CLIPS,), dtype=torch.float64).pin_memory()
    emb_pin_np, dm_pin_np, mean_pin_np = emb_pin.numpy(), dm_pin.numpy(), mean_pin.numpy()
    row_counts = [CLIPS] * world   # rank r owns global rows [r * CLIPS, (r + 1) * CLIPS): rank order = listing order
    last = {}

    def step_dev():
        emb, dm, mean = eng.score_packed(wav_dev, off, nmr_emb)
        if world > 1:  # the path's exchange: this rank's rows of the result go to rank 0
            got = nd.gather_rows_to_root([dm, mean.reshape(-1, 1)], row_counts)  # one NCCL group call
            last["dm"], last["mean"] = got if got is not None else (None, None)
        else:
            last["mean"], last["dm"] = mean, dm
        last["emb"] = emb

    def step_host():
        eng.score_host(wav_pin_np, off, nmr_emb, emb_pin_np, dm_pin_np, mean_pin_np)

    for _ in range(max(3, args.warmup)):
        step_dev()
    step_host()
    barrier()

    sampler = ClockSampler(local)
    if rank == 0 and os.environ.get("NOMAD_B200_BENCH_NO_SAMPLER") != "1":
        sampler.start()
        time.sleep(0.3)
    n0 = eng.launch_count()
    total_ms = timed(step_dev, args.steps)
    launches = eng.launch_count() - n0
    dumped = dict(last)  # the last timed step's result tensors (every step allocates new ones)
    e2e_ms = timed(step_host, args.steps)
    # roofline leg: the same K steps again with one CUDA-event pair around every tensor-core GEMM launch (kept out
    # of the `value` region: ~1100 extra event records per 10 steps cost ~5 % of the step)
    lib.nomad_b200_profile_gemm(1)
    prof_ms = timed(step_dev, args.steps)
    g_ms, g_fl, g_n = C.c_double(), C.c_double(), C.c_int64()
    lib.nomad_b200_profile_gemm_read(C.byref(g_ms), C.byref(g_fl), C.byref(g_n))
    lib.nomad_b200_profile_gemm(0)
    clocks = sampler.stop() if rank == 0 else None
    exchange_ms = None
    if world > 1:
        emb, dm, mean = eng.score_packed(wav_dev, off, nmr_emb)

        def xchg():
            nd.gather_rows_to_root([dm, mean.reshape(-1, 1)], row_counts)
        exchange_ms = timed(xchg, 20) / 20

    # ------------------------------------------------------------------ configs[4] slice: fixed global PAIR_N x PAIR_M
    pair_counts = [(r + 1) * PAIR_N // world - r * PAIR_N // world for r in range(world)]  # contiguous row ranges
    n_loc = pair_counts[rank]
    gq = torch.Generator().manual_seed(100 + rank)
    deg_e = torch.nn.functional.normalize(torch.randn(n_loc, 256, generator=gq), dim=1).to(dev)
    nmr_e = torch.nn.functional.normalize(torch.randn(PAIR_M, 256, generator=torch.Generator().manual_seed(5)), dim=1).to(dev)

    pair_dm = torch.empty((n_loc, PAIR_M), dtype=torch.float32, device=dev)     # row-sharded result, reused every step
    pair_mu = torch.empty((n_loc,), dtype=torch.float64, device=dev)

    def pair_step(want_matrix, exchange=True):
        def fn():
            # matrix rows stay with the rank that computed them; the means go to rank 0
            eng.cdist_mean(deg_e, nmr_e, want_matrix=want_matrix, out_dm=pair_dm, out_mean=pair_mu)
            if exchange:
                nd.gather_rows_to_root(pair_mu.reshape(-1, 1), pair_counts)
        return fn
    for _ in range(3):
        pair_step(True)()
    pair_ms = timed(pair_step(True), 10) / 10
    pair_mean_ms = timed(pair_step(False), 10) / 10
    pair_local_ms = timed(pair_step(True, exchange=False), 10) / 10      # kernels only (max over ranks), no exchange
    del deg_e, pair_dm

    # ------------------------------------------------------------------ configs[3]: loss fwd + bwd (single GPU by nature)
    loss = None
    if world == 1:
        gl = torch.Generator().manual_seed(11)
        est = (0.1 * torch.randn(LOSS_B, LOSS_SECONDS * SR, generator=gl)).to(dev)
        cln = (0.1 * torch.randn(LOSS_B, LOSS_SECONDS * SR, generator=gl)).to(dev)
        hw = 0.03 * torch.randn(256, 768, generator=gl)
        eng.set_loss_head(hw, torch.zeros(256))
        for _ in range(3):
            eng.loss_fwd_bwd(est, cln, 0.1)
        n1 = eng.launch_count()
        loss_ms = timed(lambda: eng.loss_fwd_bwd(est, cln, 0.1), 10) / 10
        loss_launches = (eng.launch_count() - n1) // 10
        loss_flops = 3.0 * LOSS_B * flops_embed(LOSS_SECONDS * SR)
        loss = {"workload": f"configs[3]: NOMAD loss fwd+bwd, {LOSS_B} x {LOSS_SECONDS} s estimate/clean pairs, "
                            "feature_grad_mult 0.1", "ms_per_step": loss_ms, "pairs_per_s": LOSS_B / (loss_ms / 1e3),
                "tflops_algorithmic": loss_flops / (loss_ms / 1e3) / 1e12, "launches_per_step": int(loss_launches),
                "flops_definition": "fwd(clean) + fwd(est) + dgrad(est) = 3 * B * F(N); weight gradients excluded"}

    # ------------------------------------------------------------------ the same batch in fp32-class mode (N = 1 only)
    fp32_mode = None
    if world == 1:
        del eng._ws
        eng._ws = None
        torch.cuda.empty_cache()
        eng32 = Engine(sd, local, precision="fp32")
        out32 = torch.empty((CLIPS, 256), dtype=torch.float32, device=dev)
        for _ in range(2):
            eng32.embed_packed(wav_dev, off, out32)
        ms32 = timed(lambda: eng32.embed_packed(wav_dev, off, out32), 3) / 3
        fp32_mode = {"workload": "the configs[1] batch with precision_mode = fp32 (hi + lo operand planes, 3 MMA passes, fp32 "
                                 "attention, erff GELU): embeddings within 1e-5 of the reference arithmetic",
                     "ms_per_step": ms32, "value": CLIPS * CLIP_SECONDS / (ms32 / 1e3), "unit": UNIT,
                     "emb_max_abs_diff_vs_fp16_mode": float((out32 - last["emb"]).abs().max())}
        eng32.close()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0
    sys.stdout.flush()
    os.dup2(saved_stdout, 1)

    if args.dump_outputs:
        # what a caller of the timed path receives: rank 0's embeddings, and the distance rows + row means of every
        # rank (256 x 1000 fp32, 256 fp64 per rank)
        os.makedirs(args.dump_outputs, exist_ok=True)
        dumped["mean"] = dumped["mean"].reshape(-1)  # gathered from N > 1 ranks as an (N * 256, 1) column
        for name in ("emb", "dm", "mean"):
            np.save(os.path.join(args.dump_outputs, f"{name}.npy"), dumped[name].cpu().numpy())

    utt_s_per_step = CLIPS * CLIP_SECONDS * world
    ms_per_step = total_ms / args.steps
    value = utt_s_per_step / (ms_per_step / 1e3)
    e2e_value = utt_s_per_step / (e2e_ms / args.steps / 1e3)

    peaks = {}
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(peaks_path):
        peaks = json.load(open(peaks_path))
    if "bf16_tflops_sustained" in peaks:
        peak = float(peaks["bf16_tflops_sustained"])
        peak_src = "measured (MEASURED_PEAKS.json bf16_tflops_sustained: kernel timed inside a long step)"
    else:
        peak, peak_src = FALLBACK_PEAK_TFLOPS, "fallback (B200_PROFILING.md sustained figure)"
    hbm = float(peaks.get("hbm_gbs", FALLBACK_HBM_GBS))
    achieved = (g_fl.value / 1e12) / (g_ms.value / 1e3) if g_ms.value > 0 else 0.0
    step_flops = CLIPS * flops_embed(N)

    # CPU baseline + achieved parity: rank 0, single-GPU runs only (a reported baseline, not the target)
    cpu, parity = None, None
    if world == 1:
        cpu_rate, cpu_ms, cores, cpu_n, ref_emb = cpu_reference_rate(1, 1, min_seconds=10.0)
        cpu = {"value": cpu_rate, "unit": UNIT, "cores": cores, "kind": "port",
               "sample": f"{cpu_n} pass(es) over the first {CPU_SAMPLE_CLIPS} x {CLIP_SECONDS} s clips of the batch (1/16) + "
                         f"their distance rows vs {NMR_M} NMR embeddings, oracle torch-CPU fp32, {cores} threads, "
                         f"{cpu_ms:.0f} ms/pass"}
        err = float((last["emb"][:CPU_SAMPLE_CLIPS].cpu() - ref_emb).abs().max())
        parity = {"emb_max_abs_err_vs_oracle_fp32": err, "clips_compared": CPU_SAMPLE_CLIPS, "tolerance": 1e-3,
                  "note": "fp16 operands / fp32 accumulate class of north_star (<= 1e-3); checked again in tests/"}
        if fp32_mode is not None:
            fp32_mode["emb_max_abs_err_vs_oracle_fp32"] = float((out32[:CPU_SAMPLE_CLIPS].cpu() - ref_emb).abs().max())
            fp32_mode["tolerance"] = 1e-5

    pair_total = float(PAIR_N) * PAIR_M
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "fp16", "data": "synthetic",
        "config": shared_config(source), "accumulate": "fp32",
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(CLIPS * N * 4),
                "d2h_bytes_per_step": int(CLIPS * 256 * 4 + CLIPS * NMR_M * 4 + CLIPS * 8),
                "api": "nomad_b200_score_host (pinned host waveforms in; embeddings, distance rows, means out to host)"},
        "gpu_launches": int(launches),
        "step_tflops": step_flops * world / (ms_per_step / 1e3) / 1e12,
        "roofline": {"bound": "tensor", "kernel": "gemm_tc_pair_kernel (tcgen05 cta_group::2, all GEMM launches of the step)",
                     "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak if peak else None,
                     "traffic": GEMM_DRAM_TRAFFIC_BYTES, "traffic_source": TRAFFIC_SOURCE, "peak_source": peak_src,
                     "launches_timed": int(g_n.value), "kernel_ms_per_step": g_ms.value / args.steps,
                     "kernel_share_of_step": g_ms.value / prof_ms, "profiled_ms_per_step": prof_ms / args.steps},
        "exchange": {"nmr_allgather_ms": allgather_ms, "nmr_allgather_bytes": int(C3_NMR * 256 * 4),
                     "rows_to_root_ms_per_step": exchange_ms, "rows_to_root_bytes_per_rank": int(CLIPS * NMR_M * 4 + CLIPS * 8),
                     "collective": "NCCL all_gather_into_tensor + batched isend/irecv to rank 0" if world > 1 else "none (1 rank)"},
        "sharded_c3": {"workload": f"configs[2] slice, FIXED global: {C3_DEG} degraded + {C3_NMR} NMR utterances, 1-20 s "
                                   f"(seed 0), masked varlen, through nomad_b200.dist.score_sharded", "scaling": "strong",
                       "n_gpus": world, "ms": c3_ms, "utt_s": c3_utt_s, "value": c3_utt_s / (c3_ms / 1e3), "unit": UNIT,
                       "tflops_algorithmic": c3_flops / (c3_ms / 1e3) / 1e12, "pairs": C3_DEG * C3_NMR,
                       "mean_of_means": c3_check,
                       "timed": "LPT shard -> embed NMR shard -> all-gather -> embed degraded shard -> cdist rows + means -> "
                                "means + matrix rows to rank 0 -> D2H of the means; max over ranks"},
        "pairwise": {"metric": "pairwise distances per second", "workload": f"configs[4] slice, FIXED global {PAIR_N} x {PAIR_M}",
                     "scaling": "strong", "n": PAIR_N, "m": PAIR_M, "n_gpus": world,
                     "value": pair_total / (pair_ms / 1e3), "unit": "pairs/s", "ms": pair_ms, "ms_without_exchange": pair_local_ms,
                     "write_GBps_per_gpu": pair_total / world * 4 / (pair_ms / 1e3) / 1e9,
                     "hbm_frac_per_gpu": pair_total / world * 4 / (pair_ms / 1e3) / 1e9 / hbm,
                     "means_only_value": pair_total / (pair_mean_ms / 1e3), "means_only_ms": pair_mean_ms,
                     "means_only_tensor_frac": 1536.0 * pair_total / world / (pair_mean_ms / 1e3) / 1e12 / peak,
                     "roof": "3-pass split-fp16 Gram: 1536 FLOP/pair on the tensor roof, 4 B/pair written on the HBM roof; "
                             "rows sharded across ranks, matrix rows stay with the rank, means to rank 0"},
        "loss": loss,
        "fp32_mode": fp32_mode,
        "cpu_baseline": cpu,
        "parity": parity,
        "clocks": clocks,
    }
    print(json.dumps(line), flush=True)
    sys.stdout.flush()
    os.dup2(2, 1)  # NCCL_DEBUG=INFO logs communicator teardown to stdout: keep the ONE JSON line clean
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", type=str, default="ours", choices=["ours", "reference", "library"])
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the embeddings, distance rows and row means of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    if args.impl == "reference":
        return run_reference(args)
    if args.impl == "library":
        return run_library(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
