"""End-to-end scoring FROM FILES (VERDICT r1 weak 12): `nomad.predict('dir')` over a synthetic corpus of wavs written to
/dev/shm -- file reads, ingest (decode, channel mix, resampling), H2D, embedding, distance matrix, CSV writing all inside
the clock.  The corpus encoding is 16 kHz mono PCM16 unless --encoding says otherwise; "mixed" cycles through every
encoding below.

    python tools/bench_files.py [n_deg] [n_nmr] [--encoding s16-16k-mono|s16-48k-stereo|s24-48k-mono|f32-16k-mono|mixed]
"""
import argparse, json, os, shutil, sys, tempfile, time, wave
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch
from nomad_b200.nomad import Nomad
from nomad_b200.weights import random_state_dict

# encoding -> (description, sample format, rate, channels)
ENCODINGS = {
    "s16-16k-mono": ("16 kHz mono PCM16", "s16", 16000, 1),
    "s16-48k-stereo": ("48 kHz stereo PCM16", "s16", 48000, 2),
    "s24-48k-mono": ("48 kHz mono PCM24", "s24", 48000, 1),
    "f32-16k-mono": ("16 kHz mono float32", "f32", 16000, 1),
}
ap = argparse.ArgumentParser()
ap.add_argument("n_deg", type=int, nargs="?", default=3000)
ap.add_argument("n_nmr", type=int, nargs="?", default=300)
ap.add_argument("--encoding", choices=sorted(ENCODINGS) + ["mixed"], default="s16-16k-mono")
args = ap.parse_args()
n_deg, n_nmr = args.n_deg, args.n_nmr
mixed = list(ENCODINGS.values())


def write_wav(path, x, kind, sr):
    """x: (frames, channels) float noise at the scale of the default corpus (PCM16 units / 32768)"""
    if kind == "f32":
        from scipy.io import wavfile
        wavfile.write(path, sr, x.astype(np.float32))
        return
    if kind == "s16":
        raw, width = (x * 32768).astype(np.int16).tobytes(), 2
    else:
        v = np.clip(x * (1 << 23), -(1 << 23), (1 << 23) - 1).astype("<i4")
        raw, width = v.view(np.uint8).reshape(-1, 4)[:, :3].tobytes(), 3
    with wave.open(path, "wb") as w:
        w.setnchannels(x.shape[1]); w.setsampwidth(width); w.setframerate(sr); w.writeframes(raw)


base = "/dev/shm" if os.path.isdir("/dev/shm") else tempfile.gettempdir()
root = tempfile.mkdtemp(prefix="nomad_files_", dir=base)
rng = np.random.default_rng(0)
secs = 0.0
for sub, n in (("nmr", n_nmr), ("deg", n_deg)):
    os.makedirs(os.path.join(root, sub))
    for i in range(n):
        d = rng.uniform(1.0, 20.0)
        path = os.path.join(root, sub, f"{sub}_{i:05d}.wav")
        desc, kind, sr, ch = mixed[i % len(mixed)] if args.encoding == "mixed" else ENCODINGS[args.encoding]
        if (kind, sr, ch) == ("s16", 16000, 1):   # the default corpus, sample for sample
            pcm = (rng.standard_normal(int(16000 * d)) * 3000).astype(np.int16)
            with wave.open(path, "wb") as w:
                w.setnchannels(1); w.setsampwidth(2); w.setframerate(16000); w.writeframes(pcm.tobytes())
            secs += len(pcm) / 16000.0
            continue
        x = rng.standard_normal((int(sr * d), ch)) * (3000 / 32768)
        write_wav(path, x, kind, sr)
        secs += x.shape[0] / sr
corpus = "mixed encodings (" + ", ".join(e[0] for e in mixed) + ")" if args.encoding == "mixed" else ENCODINGS[args.encoding][0]
out = os.path.join(root, "out"); os.makedirs(out)
nomad = Nomad(state_dict=random_state_dict(1234))
res = {}
for threads in (1, nomad.reader_threads):
    nomad.reader_threads = threads
    nomad.predict("dir", os.path.join(root, "nmr"), os.path.join(root, "deg"), out)   # warm-up (page cache, workspaces)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    nomad.predict("dir", os.path.join(root, "nmr"), os.path.join(root, "deg"), out)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    res[f"reader_threads_{threads}"] = {"seconds": dt, "utt_s_per_s": secs / dt}
print(json.dumps({"config": f"predict('dir') from files: {n_deg} degraded + {n_nmr} NMR wavs, 1-20 s, {corpus} on {base}, "
                            f"wall clock incl. reads, ingest, embedding, {n_deg}x{n_nmr} distances and both CSVs",
                  **({} if args.encoding == "s16-16k-mono" else {"encoding": args.encoding}),
                  "utt_s": secs, "cores": os.cpu_count(), **res}))
shutil.rmtree(root, ignore_errors=True)
