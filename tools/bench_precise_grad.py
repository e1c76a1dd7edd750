"""Cost of the fp32-class waveform gradients: device-event time per call (forward + backward) of

  (a) the fused loss step ``nomad.forward(est, clean)`` (fp16 mode replays its CUDA graph, fp32 mode runs eagerly);
  (b) the composition ``nomad_loss(lossnet_layers(clean), lossnet_layers(est))`` with ``est`` requiring grad;
  (c) ``model(wav)`` forward + backward of ``(emb * c).sum()``;

in fp16 and fp32 mode on ONE handle, the two modes alternated call by call, at 32 x 2 s and 8 x 10 s.  Also: the saved
bytes of one differentiable forward per mode, and the library path the fp32 mode competes with -- the oracle's
IEEE-fp32 torch autograd of (a) on the same GPU with TF32 off.  The card's name and power limit are read in the same run.
``python tools/bench_precise_grad.py --out profiles/bench_precise_grad.json``"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

SHAPES = [(32, 32000), (8, 160000)]
MODES = ("fp16", "fp32")


def _event_ms(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b)


def _stats(ms):
    ms = sorted(ms)
    return {"ms_median": ms[len(ms) // 2], "ms_min": ms[0], "ms_max": ms[-1], "iters": len(ms)}


def alternated(engine, fn, warmup, iters):
    """fn timed in both modes, the modes alternated call by call after `warmup` calls of each."""
    for mode in MODES:
        engine.set_precision(mode)
        for _ in range(warmup):
            fn()
    torch.cuda.synchronize()
    ms = {m: [] for m in MODES}
    for _ in range(iters):
        for mode in MODES:
            engine.set_precision(mode)
            ms[mode].append(_event_ms(fn))
    engine.set_precision("fp32")
    out = {m: _stats(v) for m, v in ms.items()}
    out["fp32_over_fp16"] = out["fp32"]["ms_median"] / out["fp16"]["ms_median"]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_precise_grad needs a CUDA device")
    from nomad_b200.nomad import Nomad
    from nomad_b200.weights import random_state_dict
    from oracle import w2v_oracle as O

    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    sd = random_state_dict(1234)
    nomad = Nomad(state_dict=sd, feature_grad_mult=0.1, precision="fp32")
    eng = nomad.engine
    sd_dev = {k: v.cuda() for k, v in sd.items() if torch.is_tensor(v)}
    lin = nomad.lossnet_layers.embedding_layer[1]
    hw, hb = lin.weight.detach().cuda(), lin.bias.detach().cuda()
    res = {}
    for B, N in SHAPES:
        g = torch.Generator(device="cuda").manual_seed(1)
        clean = 0.1 * torch.randn(B, 1, N, device="cuda", generator=g)
        est = clean + 0.03 * torch.randn(B, 1, N, device="cuda", generator=g)
        cot = torch.randn(B, 256, device="cuda", generator=g)
        r = {}

        def fused():
            e = est.clone().requires_grad_(True)
            nomad.forward(e, clean).backward()

        def composition():
            e = est.clone().requires_grad_(True)
            nomad.nomad_loss(nomad.lossnet_layers(clean), nomad.lossnet_layers(e)).backward()

        def model():
            w = est.clone().requires_grad_(True)
            (nomad.model(w) * cot).sum().backward()

        def oracle_fp32():
            e = est.clone().requires_grad_(True)
            O.nomad_forward(sd_dev, hw, hb, e, clean, dtype=torch.float32, feature_grad_mult=0.1).backward()

        r["a_fused_loss"] = alternated(eng, fused, args.warmup, args.iters)
        r["b_composition_est_grad"] = alternated(eng, composition, args.warmup, args.iters)
        r["c_model_fwd_bwd"] = alternated(eng, model, args.warmup, args.iters)
        for _ in range(args.warmup):
            oracle_fp32()
        torch.cuda.synchronize()
        r["oracle_ieee_fp32_autograd_fused_loss"] = _stats([_event_ms(oracle_fp32) for _ in range(args.iters)])
        r["fp32_mode_fused_over_oracle_fp32"] = (r["a_fused_loss"]["fp32"]["ms_median"]
                                                 / r["oracle_ieee_fp32_autograd_fused_loss"]["ms_median"])
        r["saved_bytes_per_forward"] = {m: int(eng.lib.nomad_b200_layers_saved_bytes_mode(B, N, i)) for i, m in enumerate(MODES)}
        r["loss_workspace_bytes"] = {m: int(eng.lib.nomad_b200_loss_workspace_bytes_mode(B, N, 1, i)) for i, m in enumerate(MODES)}
        r["peak_allocated_bytes"] = int(torch.cuda.max_memory_allocated())
        torch.cuda.reset_peak_memory_stats()
        res[f"{B}x{N / 16000:g}s"] = r
        print(json.dumps({f"{B}x{N / 16000:g}s": r}), flush=True)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    doc = {"device": torch.cuda.get_device_name(0), "nvidia_smi_name_power_limit": smi[0] if smi else None,
           "torch": torch.__version__, "tf32": False, "feature_grad_mult": 0.1, "results": res}
    print(json.dumps(doc, indent=1))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(doc, f, indent=1)


if __name__ == "__main__":
    main()
