"""Waveform ingest: ``Nomad.load_processing`` (reference ``nomad.py:192-212``).

``torchaudio.load`` needs torchcodec, which this image does not have, so PCM wav files are decoded
with the standard library (``torchaudio.load`` semantics: integer PCM scaled to [-1, 1) float32,
shape (channels, N)); anything else is handed to torchaudio / scipy if they can read it.
Resampling uses ``torchaudio.transforms.Resample`` exactly like the reference.
"""
from __future__ import annotations

import wave

import numpy as np
import torch


def load_wav(filepath: str):
    """-> (float32 tensor (channels, N), sample_rate)"""
    try:
        with wave.open(str(filepath), "rb") as w:
            ch, sr, n, sw = w.getnchannels(), w.getframerate(), w.getnframes(), w.getsampwidth()
            raw = w.readframes(n)
        if sw == 2:
            pcm = np.frombuffer(raw, dtype="<i2").astype(np.float32) / 32768.0
        elif sw == 4:
            pcm = np.frombuffer(raw, dtype="<i4").astype(np.float32) / 2147483648.0
        elif sw == 1:
            pcm = (np.frombuffer(raw, dtype=np.uint8).astype(np.float32) - 128.0) / 128.0
        elif sw == 3:
            b = np.frombuffer(raw, dtype=np.uint8).reshape(-1, 3).astype(np.int32)
            v = b[:, 0] | (b[:, 1] << 8) | (b[:, 2] << 16)
            v = np.where(v >= 1 << 23, v - (1 << 24), v)
            pcm = v.astype(np.float32) / 8388608.0
        else:
            raise wave.Error(f"unsupported sample width {sw}")
        return torch.from_numpy(pcm.reshape(-1, ch).T.copy()), sr
    except wave.Error:
        pass
    try:  # float / extensible wav
        from scipy.io import wavfile
        sr, data = wavfile.read(str(filepath))
        if data.dtype.kind == "i":
            data = data.astype(np.float32) / float(2 ** (8 * data.dtype.itemsize - 1))
        elif data.dtype == np.uint8:
            data = (data.astype(np.float32) - 128.0) / 128.0
        data = np.asarray(data, dtype=np.float32)
        if data.ndim == 1:
            data = data[:, None]
        return torch.from_numpy(data.T.copy()), int(sr)
    except Exception:
        import torchaudio
        return torchaudio.load(filepath)


def load_processing_device(engine, filepath, target_sr: int = 16000, trim: bool = False) -> torch.Tensor:
    """``load_processing`` with the sample decode, channel mix, resampling and trim on the GPU
    (``Engine.ingest_wav_files``) for every wav file the native reader handles (PCM of 8, 16, 24 or 32 bits, float of
    32 or 64 bits) -- the file's own data bytes are what crosses PCIe; any other file takes the host path below and is
    moved to the device.  Returns a (1, N) fp32 CUDA tensor."""
    from . import _lib
    if isinstance(filepath, np.ndarray):
        filepath = filepath[0]
    probe = _lib.wav_probe_format([str(filepath)], 1)
    if probe.frames[0] < 0:
        return load_processing(filepath, target_sr, trim).to(engine.device)
    n_out = _lib.ingest_out_samples(probe.frames, probe.sample_rate, target_sr, trim)
    out = torch.empty((1, int(n_out[0])), dtype=torch.float32, device=engine.device)
    engine.ingest_wav_files([str(filepath)], probe, n_out, out, np.zeros(1, np.int64), 1, target_sr)
    return out


def load_processing(filepath, target_sr: int = 16000, trim: bool = False) -> torch.Tensor:
    """Mono 16 kHz float32 (1, N): mean of the first two channels if multi-channel
    (``nomad.py:199-200``), resample if needed (``:203-205``), optional 10 s trim (``:208-210``)."""
    if isinstance(filepath, np.ndarray):
        filepath = filepath[0]  # nomad.py:194-195: a DataFrame row
    wave_, sr = load_wav(filepath)
    if wave_.shape[0] > 1:
        wave_ = ((wave_[0, :] + wave_[1, :]) / 2).unsqueeze(0)
    if sr != target_sr:
        import torchaudio
        wave_ = torchaudio.transforms.Resample(sr, target_sr)(wave_)
        sr = target_sr
    if trim:
        if wave_.shape[1] > sr * 10:
            wave_ = wave_[:, : sr * 10]
    return wave_
