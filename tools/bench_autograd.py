"""Device-event timings of the differentiable paths, per call (forward + backward):

  (a) ``nomad.forward(est, clean)`` fused loss step, replayed CUDA graph and eager (``NOMAD_B200_LOSS_GRAPH=0``, read
      once per process: measured in a child process);
  (b) the reference composition ``nomad_loss(lossnet_layers(clean), lossnet_layers(est))`` with ``est`` requiring grad;
  (c) the same with both ``est`` and ``clean`` requiring grad;
  (d) ``model(wav)`` forward + backward of ``(emb * c).sum()``.

Shapes: 32 x 2 s (the loss configuration) and 8 x 10 s.  Also reports the saved-activation bytes of one
differentiable forward, and the card's name and power limit read in the same run.
``python tools/bench_autograd.py --out profiles/bench_autograd.json``"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

SHAPES = [(32, 32000), (8, 160000)]


def timed(fn, warmup, iters):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ms = []
    for _ in range(iters):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ms.append(a.elapsed_time(b))
    ms.sort()
    return {"ms_median": ms[len(ms) // 2], "ms_min": ms[0], "ms_max": ms[-1], "iters": iters}


def run(which, warmup, iters):
    from nomad_b200.nomad import Nomad
    from nomad_b200.weights import random_state_dict
    nomad = Nomad(state_dict=random_state_dict(1234), feature_grad_mult=0.1)
    out = {}
    for B, N in SHAPES:
        g = torch.Generator(device="cuda").manual_seed(1)
        clean = 0.1 * torch.randn(B, 1, N, device="cuda", generator=g)
        est = clean + 0.03 * torch.randn(B, 1, N, device="cuda", generator=g)
        key = f"{B}x{N / 16000:g}s"
        r = {}

        def fused():
            e = est.clone().requires_grad_(True)
            nomad.forward(e, clean).backward()

        def composition(both):
            e = est.clone().requires_grad_(True)
            c = clean.clone().requires_grad_(both)
            nomad.nomad_loss(nomad.lossnet_layers(c), nomad.lossnet_layers(e)).backward()

        cot = torch.randn(B, 256, device="cuda", generator=g)

        def model():
            w = est.clone().requires_grad_(True)
            (nomad.model(w) * cot).sum().backward()

        if which == "eager":
            r["a_fused_eager"] = timed(fused, warmup, iters)
        else:
            r["a_fused_graph"] = timed(fused, warmup, iters)
            r["b_composition_est_grad"] = timed(lambda: composition(False), warmup, iters)
            r["c_composition_both_grads"] = timed(lambda: composition(True), warmup, iters)
            r["d_model_fwd_bwd"] = timed(model, warmup, iters)
            r["saved_bytes_per_forward"] = int(nomad.engine.lib.nomad_b200_layers_saved_bytes(B, N))
            r["bwd_workspace_bytes"] = int(nomad.engine.lib.nomad_b200_layers_bwd_workspace_bytes(B, N))
            r["peak_allocated_bytes"] = int(torch.cuda.max_memory_allocated())
        out[key] = r
        torch.cuda.reset_peak_memory_stats()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--out", default=None)
    ap.add_argument("--only", choices=["eager"], default=None, help=argparse.SUPPRESS)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_autograd needs a CUDA device")
    if args.only == "eager":
        print(json.dumps(run("eager", args.warmup, args.iters)))
        return
    res = run("graph", args.warmup, args.iters)
    env = dict(os.environ, NOMAD_B200_LOSS_GRAPH="0")
    child = subprocess.run([sys.executable, __file__, "--only", "eager", "--warmup", str(args.warmup), "--iters",
                            str(args.iters)], env=env, capture_output=True, text=True, check=True)
    eager = json.loads(child.stdout.strip().splitlines()[-1])
    for key, r in eager.items():
        res[key].update(r)
        res[key]["b_over_a_eager"] = res[key]["b_composition_est_grad"]["ms_median"] / r["a_fused_eager"]["ms_median"]
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    doc = {"device": torch.cuda.get_device_name(0), "nvidia_smi_name_power_limit": smi[0] if smi else None,
           "torch": torch.__version__, "feature_grad_mult": 0.1, "results": res}
    print(json.dumps(doc, indent=1))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(doc, f, indent=1)


if __name__ == "__main__":
    main()
