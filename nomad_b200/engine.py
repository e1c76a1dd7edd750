"""Thin host wrapper over the C ABI: owns the handle, torch-allocated workspaces and streams.

PyTorch is used for device memory, streams and (in ``dist.py``) ``torch.distributed`` only; every
arithmetic step of the path runs in ``libnomad_b200.so``.  There is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
from typing import List, Optional, Sequence

import numpy as np
import torch

from . import _lib
from .weights import EMB_DIM, NUM_LAYERS, SSL_OUT_DIM

MIN_SAMPLES = 400
PRECISIONS = {"fp16": 0, "fp32": 1}   # NOMAD_B200_PRECISION_FP16 / _FP32


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream_ptr():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


class Engine:
    """One NOMAD model resident on one GPU."""

    def __init__(self, state_dict, device: Optional[int] = None, precision: str = "fp16"):
        """``precision``: "fp16" (fp16 tensor-core operands, embeddings within 1e-3 of the fp32 reference) or "fp32"
        (split hi + lo operands, within 1e-5; ~3x the time).  An "fp32" engine holds both weight sets and can be
        switched with :meth:`set_precision`."""
        self.lib = _lib.load()
        if precision not in PRECISIONS:
            raise ValueError(f"precision must be one of {sorted(PRECISIONS)}, got {precision!r}")
        self.precision = precision
        if not torch.cuda.is_available():
            raise _lib.NomadB200Error("nomad_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
        self.device_index = torch.cuda.current_device() if device is None else int(device)
        self.device = torch.device("cuda", self.device_index)
        names, arrays = [], []
        for k, v in state_dict.items():
            if not torch.is_tensor(v) or k.endswith("mask_emb"):
                continue
            names.append(k.encode())
            arrays.append(np.ascontiguousarray(v.detach().to(torch.float32).cpu().numpy()))
        tens = (_lib.Tensor * len(names))()
        for i, (n, a) in enumerate(zip(names, arrays)):
            tens[i].name = n
            tens[i].data = a.ctypes.data_as(C.c_void_p)
            tens[i].numel = a.size
        h = C.c_void_p()
        with torch.cuda.device(self.device):
            _lib.check(self.lib.nomad_b200_create(C.byref(h), tens, len(names), PRECISIONS[precision], self.device_index),
                       "nomad_b200_create")
        self.handle = h
        self._ws: Optional[torch.Tensor] = None
        self._pinned: Optional[torch.Tensor] = None
        self._pinned_out: Optional[torch.Tensor] = None
        # bumped by every weight refresh: an autograd graph recorded under an older generation cannot be differentiated
        self.weight_generation = 0
        # called before every call that runs the network (Nomad's parameter store: push edited parameters to the device)
        self.sync_hook = None

    def sync_weights(self):
        if self.sync_hook is not None:
            self.sync_hook()

    def close(self):
        if getattr(self, "handle", None):
            self.lib.nomad_b200_destroy(self.handle)
            self.handle = None

    def __del__(self):  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------ helpers
    def set_gemm_impl(self, impl: int):
        _lib.check(self.lib.nomad_b200_set_gemm_impl(self.handle, int(impl)), "set_gemm_impl")

    def set_precision(self, precision: str):
        _lib.check(self.lib.nomad_b200_set_precision(self.handle, PRECISIONS[precision]), "set_precision")
        self.precision = precision

    @property
    def _mode(self) -> int:
        return PRECISIONS[self.precision]

    def refresh_weights(self, state_dict_dev):
        """Rebuild the kernel-ready weights from fp32 master tensors on THIS device (``nomad_b200_refresh_weights``): the step
        after an optimiser update.  ``state_dict_dev``: {state_dict key: contiguous fp32 CUDA tensor}.  Everything after
        the conv feature encoder; ``refresh_conv_weights`` rebuilds the encoder."""
        self._refresh(state_dict_dev, False)

    def refresh_conv_weights(self, state_dict_dev):
        """The same for the conv feature encoder (``nomad_b200_refresh_conv_weights``), in place: pointers captured by
        loss-step CUDA graphs stay valid."""
        self._refresh(state_dict_dev, True)

    def _refresh(self, state_dict_dev, conv: bool):
        names, ptrs, keep = [], [], []
        for k, v in state_dict_dev.items():
            if not torch.is_tensor(v) or k.endswith("mask_emb") or ("feature_extractor" in k) != conv:
                continue
            t = v.detach()
            assert t.is_cuda and t.device == self.device and t.dtype == torch.float32 and t.is_contiguous(), k
            names.append(k.encode()); ptrs.append(t.data_ptr()); keep.append(t)
        tens = (_lib.Tensor * len(names))()
        for i, (n, p_, t) in enumerate(zip(names, ptrs, keep)):
            tens[i].name = n
            tens[i].data = C.c_void_p(p_)
            tens[i].numel = t.numel()
        with torch.cuda.device(self.device):
            fn = "nomad_b200_refresh_conv_weights" if conv else "nomad_b200_refresh_weights"
            _lib.check(getattr(self.lib, fn)(self.handle, tens, len(names), _stream_ptr()), fn)
        self.weight_generation += 1

    def set_loss_head(self, weight: torch.Tensor, bias: torch.Tensor):
        w = np.ascontiguousarray(weight.detach().to(torch.float32).cpu().numpy())
        b = np.ascontiguousarray(bias.detach().to(torch.float32).cpu().numpy())
        assert w.shape == (EMB_DIM, SSL_OUT_DIM) and b.shape == (EMB_DIM,)
        _lib.check(self.lib.nomad_b200_set_loss_head(self.handle, w.ctypes.data_as(C.c_void_p),
                                                     b.ctypes.data_as(C.c_void_p)), "set_loss_head")

    def workspace(self, nbytes: int) -> torch.Tensor:
        """Grow-only device scratch (torch caching allocator), 1024-byte aligned."""
        if self._ws is None or self._ws.numel() < nbytes + 1024:
            self._ws = None
            self._ws = torch.empty(int(nbytes * 1.05) + 2048, dtype=torch.uint8, device=self.device)
        return self._ws

    @staticmethod
    def _aligned(ws: torch.Tensor):
        base = ws.data_ptr()
        off = (-base) % 1024
        return C.c_void_p(base + off), ws.numel() - off

    @staticmethod
    def offsets(lengths: Sequence[int]):
        off = np.zeros(len(lengths) + 1, dtype=np.int64)
        np.cumsum(np.asarray(lengths, dtype=np.int64), out=off[1:])
        return off

    # ------------------------------------------------------------------ scoring
    def embed_packed(self, wav: torch.Tensor, offsets: np.ndarray, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """``wav``: 1-D fp32 CUDA tensor holding the utterances back to back; ``offsets``: B+1 int64 (host)."""
        self.sync_weights()
        assert wav.is_cuda and wav.dtype == torch.float32 and wav.is_contiguous()
        B = len(offsets) - 1
        offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        off_p = offsets.ctypes.data_as(C.POINTER(C.c_int64))
        need = self.lib.nomad_b200_embed_workspace_bytes_mode(off_p, B, self._mode)
        if need == 0:
            raise _lib.NomadB200Error(self.lib.nomad_b200_last_error().decode())
        ws = self.workspace(need)
        wp, wbytes = self._aligned(ws)
        if out is None:
            out = torch.empty((B, EMB_DIM), dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.nomad_b200_embed(self.handle, _ptr(wav), off_p, B, _ptr(out), wp, wbytes, _stream_ptr()),
                       "nomad_b200_embed")
        return out

    def embed(self, waves: Sequence[torch.Tensor]) -> torch.Tensor:
        """Variable-length batch: list of 1-D (or (1, N)) fp32 tensors on any device -> (B, 256) CUDA tensor."""
        flat = [w.reshape(-1).to(torch.float32) for w in waves]
        offsets = self.offsets([int(w.numel()) for w in flat])
        wav = torch.cat([w.to(self.device, non_blocking=True) for w in flat])
        return self.embed_packed(wav, offsets)

    def embed_host(self, wav_host: np.ndarray, offsets: np.ndarray, emb_host: Optional[np.ndarray] = None) -> np.ndarray:
        """HOST buffers in and out through ``nomad_b200_embed_host`` (H2D + compute + D2H + sync inside)."""
        self.sync_weights()
        B = len(offsets) - 1
        offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        off_p = offsets.ctypes.data_as(C.POINTER(C.c_int64))
        need = self.lib.nomad_b200_embed_workspace_bytes_mode(off_p, B, self._mode)
        if need == 0:
            raise _lib.NomadB200Error(self.lib.nomad_b200_last_error().decode())
        total = int(offsets[-1] - offsets[0])
        ws = self.workspace(need + 4 * total + 1024 * B + 8192)
        wp, wbytes = self._aligned(ws)
        if emb_host is None:
            emb_host = np.empty((B, EMB_DIM), dtype=np.float32)
        assert wav_host.dtype == np.float32 and wav_host.flags.c_contiguous
        with torch.cuda.device(self.device):
            _lib.check(self.lib.nomad_b200_embed_host(self.handle, wav_host.ctypes.data_as(C.c_void_p), off_p, B,
                                                      emb_host.ctypes.data_as(C.c_void_p), wp, wbytes, _stream_ptr()),
                       "nomad_b200_embed_host")
        return emb_host

    def score_packed(self, wav: torch.Tensor, offsets: np.ndarray, nmr: torch.Tensor, want_matrix: bool = True):
        """One batch of ``Nomad.predict`` on device-resident data: -> (emb (B, 256), dm (B, m) | None, mean (B,) fp64)."""
        self.sync_weights()
        assert wav.is_cuda and wav.dtype == torch.float32 and wav.is_contiguous()
        assert nmr.is_cuda and nmr.dtype == torch.float32 and nmr.is_contiguous() and nmr.shape[1] == EMB_DIM
        B, m = len(offsets) - 1, nmr.shape[0]
        offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        off_p = offsets.ctypes.data_as(C.POINTER(C.c_int64))
        need = self.lib.nomad_b200_score_workspace_bytes_mode(off_p, B, m, self._mode)
        if need == 0:
            raise _lib.NomadB200Error(self.lib.nomad_b200_last_error().decode())
        wp, wbytes = self._aligned(self.workspace(need))
        emb = torch.empty((B, EMB_DIM), dtype=torch.float32, device=self.device)
        dm = torch.empty((B, m), dtype=torch.float32, device=self.device) if want_matrix else None
        mean = torch.empty((B,), dtype=torch.float64, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.nomad_b200_score(self.handle, _ptr(wav), off_p, B, _ptr(nmr), m, _ptr(emb), _ptr(dm),
                                                 _ptr(mean), wp, wbytes, _stream_ptr()), "nomad_b200_score")
        return emb, dm, mean

    def score_host(self, wav_host: np.ndarray, offsets: np.ndarray, nmr: torch.Tensor, emb_host: Optional[np.ndarray],
                   dm_host: Optional[np.ndarray], mean_host: np.ndarray):
        """Same with HOST waveforms in and HOST results out (H2D + compute + D2H + sync inside the C call)."""
        self.sync_weights()
        assert wav_host.dtype == np.float32 and wav_host.flags.c_contiguous and mean_host.dtype == np.float64
        assert nmr.is_cuda and nmr.dtype == torch.float32 and nmr.is_contiguous() and nmr.shape[1] == EMB_DIM
        B, m = len(offsets) - 1, nmr.shape[0]
        offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        off_p = offsets.ctypes.data_as(C.POINTER(C.c_int64))
        need = self.lib.nomad_b200_score_workspace_bytes_mode(off_p, B, m, self._mode)
        if need == 0:
            raise _lib.NomadB200Error(self.lib.nomad_b200_last_error().decode())
        wp, wbytes = self._aligned(self.workspace(need))
        hp = lambda a: None if a is None else a.ctypes.data_as(C.c_void_p)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.nomad_b200_score_host(self.handle, hp(wav_host), off_p, B, _ptr(nmr), m, hp(emb_host),
                                                      hp(dm_host), hp(mean_host), wp, wbytes, _stream_ptr()),
                       "nomad_b200_score_host")

    # ------------------------------------------------------------------ pinned staging ring
    def pinned(self, nbytes: int) -> torch.Tensor:
        """A pinned host staging buffer (ring of 3, grow-only) that no in-flight H2D copy is still reading; after
        issuing the copy call :meth:`pinned_release` so the slot is fenced by an event on the current stream."""
        if not hasattr(self, "_ring"):
            self._ring, self._ring_ev, self._ring_i = [None] * 3, [None] * 3, 0
        self._ring_i = (self._ring_i + 1) % 3
        i = self._ring_i
        if self._ring_ev[i] is not None:
            self._ring_ev[i].synchronize()
        if self._ring[i] is None or self._ring[i].numel() < nbytes:
            self._ring[i] = torch.empty(int(nbytes * 1.25) + 4096, dtype=torch.uint8).pin_memory()
        return self._ring[i]

    def pinned_release(self):
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream())
        self._ring_ev[self._ring_i] = ev

    def ingest_wav_files(self, paths, probe: "_lib.WavProbe", n_out, out: torch.Tensor, out_offset, threads: int = 0,
                         target_sr: int = 16000):
        """``load_processing`` on the device for wav files the native reader handles (``probe.frames >= 0``): their data
        bytes are read by the library's host threads into the pinned staging ring (each file at a 16-byte aligned
        offset), cross PCIe in ONE copy and are decoded, mixed and resampled by ONE ``nomad_b200_ingest_batch`` call
        (one launch per source rate) into ``out[out_offset[i]:][:n_out[i]]`` (fp32 CUDA).  Nothing synchronises."""
        n_bytes = probe.frames * probe.channels * _lib.FORMAT_BYTES[probe.format]
        staged = (n_bytes + 15) // 16 * 16
        dst = np.zeros(len(paths), np.int64)
        np.cumsum(staged[:-1], out=dst[1:])
        total = int(staged.sum())
        stage = self.pinned(total)
        _lib.wav_read(paths, probe.data_offset, n_bytes, dst, stage.data_ptr(), threads)
        src = stage[:total].to(self.device, non_blocking=True)
        self.pinned_release()
        items = np.zeros(len(paths), _lib.INGEST_ITEM)
        items["byte_offset"], items["n_frames"], items["out_offset"], items["out_samples"] = dst, probe.frames, out_offset, n_out
        items["channels"], items["format"], items["sample_rate"] = probe.channels, probe.format, probe.sample_rate
        ip = items.ctypes.data_as(C.c_void_p)
        need = self.lib.nomad_b200_ingest_workspace_bytes(ip, len(items), int(target_sr))
        if need == 0:
            raise _lib.NomadB200Error(self.lib.nomad_b200_last_error().decode())
        wp, wbytes = self._aligned(self.workspace(need))
        assert out.is_cuda and out.dtype == torch.float32 and out.is_contiguous()
        with torch.cuda.device(self.device):
            _lib.check(self.lib.nomad_b200_ingest_batch(_ptr(src), ip, len(items), int(target_sr), _ptr(out), wp, wbytes,
                                                        _stream_ptr()), "nomad_b200_ingest_batch")

    def embed_wav_files(self, paths, probe: "_lib.WavProbe", threads: int = 0, out: Optional[torch.Tensor] = None,
                        waves=None) -> torch.Tensor:
        """Embed one batch of wav files (``load_processing`` + ``model`` of nomad.py:172-186) -> (B, 256) CUDA tensor.
        Files with ``probe.frames >= 0`` go through :meth:`ingest_wav_files`; the others must come decoded in ``waves``
        ({position in ``paths``: 1-D or (1, N) fp32 tensor at 16 kHz}) and are copied into the same packed buffer, so
        the whole batch is one ``nomad_b200_embed`` call."""
        waves = waves or {}
        native = np.flatnonzero(probe.frames >= 0)
        lens = np.zeros(len(paths), np.int64)
        lens[native] = _lib.ingest_out_samples(probe.frames[native], probe.sample_rate[native])
        for i, w in waves.items():
            lens[i] = w.numel()
        offsets = self.offsets(lens)
        wav = torch.empty((int(offsets[-1]),), dtype=torch.float32, device=self.device)
        if len(native):
            self.ingest_wav_files([paths[i] for i in native], probe.take(native), lens[native], wav, offsets[native],
                                  threads)
        for i, w in waves.items():
            wav[offsets[i]:offsets[i + 1]].copy_(w.reshape(-1), non_blocking=True)
        return self.embed_packed(wav, offsets, out)

    # ------------------------------------------------------------------ ingest
    def ingest_pcm16(self, pcm: np.ndarray, sr: int, target_sr: int = 16000, trim: bool = False) -> torch.Tensor:
        """``load_processing`` on the device: (n_frames, channels) or (n_frames,) int16 HOST samples at ``sr`` ->
        (1, N) fp32 CUDA tensor at ``target_sr`` (mono mix, torchaudio-default resampling, optional 10 s trim)."""
        pcm = np.ascontiguousarray(pcm, dtype=np.int16)
        if pcm.ndim == 1:
            pcm = pcm[:, None]
        n, ch = pcm.shape
        n_out = int(self.lib.nomad_b200_ingest_out_samples(n, int(sr), int(target_sr), 1 if trim else 0))
        out = torch.empty((1, max(n_out, 0)), dtype=torch.float32, device=self.device)
        if n_out > 0:
            dev = torch.from_numpy(pcm if pcm.flags.writeable else pcm.copy()).to(self.device, non_blocking=True)
            with torch.cuda.device(self.device):
                _lib.check(self.lib.nomad_b200_ingest_pcm16(_ptr(dev), n, ch, int(sr), int(target_sr), 1 if trim else 0,
                                                            _ptr(out), _stream_ptr()), "nomad_b200_ingest_pcm16")
        return out

    # ------------------------------------------------------------------ loss-side forward
    def num_frames(self, n: int) -> int:
        return int(self.lib.nomad_b200_num_frames(int(n)))

    def layers(self, wav: torch.Tensor, want_layers: bool = True, want_emb: bool = True):
        """``LossNetLayers.forward`` for a (B, N) or (B, 1, N) CUDA batch -> ((12, B, T, 768) | None, (B, 256) | None)."""
        self.sync_weights()
        if wav.dim() == 3:
            wav = wav.squeeze(1)
        wav = wav.to(self.device, torch.float32).contiguous()
        B, N = wav.shape
        T = self.num_frames(N)
        need = self.lib.nomad_b200_layers_workspace_bytes_mode(B, N, self._mode)
        if need == 0:
            raise _lib.NomadB200Error(self.lib.nomad_b200_last_error().decode())
        ws = self.workspace(need)
        wp, wbytes = self._aligned(ws)
        layers = torch.empty((NUM_LAYERS, B, T, SSL_OUT_DIM), dtype=torch.float32, device=self.device) if want_layers else None
        emb = torch.empty((B, EMB_DIM), dtype=torch.float32, device=self.device) if want_emb else None
        with torch.cuda.device(self.device):
            _lib.check(self.lib.nomad_b200_layers_fwd(self.handle, _ptr(wav), B, N, _ptr(layers), _ptr(emb), wp, wbytes,
                                                      _stream_ptr()), "nomad_b200_layers_fwd")
        return layers, emb

    def layers_fwd_save(self, wav: torch.Tensor, head: int, want_layers: bool = True, flags: int = 0):
        """Save-mode forward of a (B, N) CUDA batch for autograd (``nomad_b200_layers_fwd_save``, in the engine's precision;
        with ``flags`` fp16 operands whatever the precision).  ``head``: 0 = NOMAD head, 1 = loss head.  -> ((12, B, T, 768) | None, (B, 256), saved):
        ``saved`` is a uint8 CUDA tensor owned by the caller that :meth:`layers_bwd` needs; keep it until then.
        ``flags`` (``_lib.SAVE_*``, ``nomad_b200_layers_fwd_save_ex``): also save for :meth:`layers_bwd_params`."""
        self.sync_weights()
        wav = wav.to(self.device, torch.float32).contiguous()
        B, N = wav.shape
        T = self.num_frames(N)
        nbytes = (self.lib.nomad_b200_layers_saved_bytes_ex(B, N, int(flags)) if flags
                  else self.lib.nomad_b200_layers_saved_bytes_mode(B, N, self._mode))
        if nbytes == 0:
            raise _lib.NomadB200Error(self.lib.nomad_b200_last_error().decode())
        saved = torch.empty(nbytes + 1024, dtype=torch.uint8, device=self.device)
        sp, sbytes = self._aligned(saved)
        layers = torch.empty((NUM_LAYERS, B, T, SSL_OUT_DIM), dtype=torch.float32, device=self.device) if want_layers else None
        emb = torch.empty((B, EMB_DIM), dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            if flags:
                _lib.check(self.lib.nomad_b200_layers_fwd_save_ex(self.handle, _ptr(wav), B, N, int(head), _ptr(layers),
                                                                  _ptr(emb), sp, sbytes, int(flags), _stream_ptr()),
                           "nomad_b200_layers_fwd_save_ex")
            else:
                _lib.check(self.lib.nomad_b200_layers_fwd_save(self.handle, _ptr(wav), B, N, int(head), _ptr(layers),
                                                               _ptr(emb), sp, sbytes, _stream_ptr()), "nomad_b200_layers_fwd_save")
        return layers, emb, saved

    def layers_bwd(self, saved: torch.Tensor, wav: torch.Tensor, g_layers: Sequence[Optional[torch.Tensor]],
                   g_emb: Optional[torch.Tensor], feature_grad_mult: float) -> torch.Tensor:
        """d(<g_layers, layers> + <g_emb, emb>) / d wav for the forward that filled ``saved`` (``nomad_b200_layers_bwd``):
        ``g_layers``: 12 entries of (B, T, 768) or None, ``g_emb``: (B, 256) or None.  -> (B, N) fp32 CUDA tensor.  Runs
        in the precision the forward was saved in, which must still be the engine's (the library refuses otherwise)."""
        wav = wav.to(self.device, torch.float32).contiguous()
        B, N = wav.shape

        gl = [self._grad_in(g) for g in g_layers]
        ge = self._grad_in(g_emb)
        need = self.lib.nomad_b200_layers_bwd_workspace_bytes_mode(B, N, self._mode)
        if need == 0:
            raise _lib.NomadB200Error(self.lib.nomad_b200_last_error().decode())
        wp, wbytes = self._aligned(self.workspace(need))
        sp, sbytes = self._aligned(saved)
        ptrs = (C.c_void_p * NUM_LAYERS)(*[None if g is None else g.data_ptr() for g in gl])
        d_wav = torch.empty((B, N), dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.nomad_b200_layers_bwd(self.handle, sp, sbytes, _ptr(wav), B, N, ptrs, _ptr(ge),
                                                      C.c_float(feature_grad_mult), _ptr(d_wav), wp, wbytes, _stream_ptr()),
                       "nomad_b200_layers_bwd")
        return d_wav

    def _grad_in(self, g):  # fp32, contiguous, 16-byte aligned (the kernels read rows as float4)
        if g is None:
            return None
        g = g.to(self.device, torch.float32).contiguous()
        return g if g.data_ptr() % 16 == 0 else g.clone()

    def layers_bwd_params(self, saved: torch.Tensor, wav: torch.Tensor, g_layers: Sequence[Optional[torch.Tensor]],
                          g_emb: Optional[torch.Tensor], feature_grad_mult: float, flags: int, want_wav: bool,
                          want_params: bool, want_conv: bool):
        """:meth:`layers_bwd` plus the parameter gradients (``nomad_b200_layers_bwd_params``) for a forward saved with
        ``flags``.  -> (d_wav (B, N) | None, grads (flat, ``triplet.grad_segments()`` layout) | None, conv_grads (flat,
        ``grad_segments(conv=True)``) | None, S (0-dim CUDA tensor)): every result is multiplied by S."""
        wav = wav.to(self.device, torch.float32).contiguous()
        B, N = wav.shape
        gl = [self._grad_in(g) for g in g_layers]
        ge = self._grad_in(g_emb)
        need = self.lib.nomad_b200_layers_bwd_params_workspace_bytes(B, N, int(flags))
        if need == 0:
            raise _lib.NomadB200Error(self.lib.nomad_b200_last_error().decode())
        wp, wbytes = self._aligned(self.workspace(need))
        sp, sbytes = self._aligned(saved)
        ptrs = (C.c_void_p * NUM_LAYERS)(*[None if g is None else g.data_ptr() for g in gl])
        f32 = dict(dtype=torch.float32, device=self.device)
        d_wav = torch.empty((B, N), **f32) if want_wav else None
        grads = torch.empty((int(self.lib.nomad_b200_triplet_grad_floats()),), **f32) if want_params else None
        conv = torch.empty((int(self.lib.nomad_b200_triplet_conv_grad_floats()),), **f32) if want_conv else None
        scale = torch.empty((), **f32)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.nomad_b200_layers_bwd_params(self.handle, sp, sbytes, _ptr(wav), B, N, ptrs, _ptr(ge),
                                                             C.c_float(feature_grad_mult), _ptr(d_wav), _ptr(grads), _ptr(conv),
                                                             _ptr(scale), wp, wbytes, _stream_ptr()),
                       "nomad_b200_layers_bwd_params")
        return d_wav, grads, conv, scale

    def loss_fwd_bwd(self, est: torch.Tensor, clean: torch.Tensor, feature_grad_mult: float, with_grad: bool = True):
        self.sync_weights()
        if est.dim() == 3:
            est = est.squeeze(1)
        if clean.dim() == 3:
            clean = clean.squeeze(1)
        est = est.detach().to(self.device, torch.float32).contiguous()
        clean = clean.detach().to(self.device, torch.float32).contiguous()
        assert est.shape == clean.shape
        B, N = est.shape
        need = self.lib.nomad_b200_loss_workspace_bytes_mode(B, N, 1 if with_grad else 0, self._mode)
        if need == 0:
            raise _lib.NomadB200Error(self.lib.nomad_b200_last_error().decode())
        ws = self.workspace(need)
        wp, wbytes = self._aligned(ws)
        loss = torch.empty((), dtype=torch.float32, device=self.device)
        grad = torch.empty_like(est) if with_grad else None
        with torch.cuda.device(self.device):
            _lib.check(self.lib.nomad_b200_loss_fwd_bwd(self.handle, _ptr(est), _ptr(clean), B, N,
                                                        C.c_float(feature_grad_mult), _ptr(loss), _ptr(grad), wp, wbytes,
                                                        _stream_ptr()), "nomad_b200_loss_fwd_bwd")
        return loss, grad

    # ------------------------------------------------------------------ distance
    def cdist_mean(self, deg: torch.Tensor, nmr: torch.Tensor, want_matrix: bool = True, gemm_impl: int = 0,
                   out_dm: Optional[torch.Tensor] = None, out_mean: Optional[torch.Tensor] = None):
        """(n, 256), (m, 256) fp32 CUDA -> ((n, m) fp32 | None, (n,) fp64 row means); ``out_dm`` / ``out_mean``:
        caller-owned result tensors (a scoring service reuses them across batches)."""
        deg = deg.to(self.device, torch.float32).contiguous()
        nmr = nmr.to(self.device, torch.float32).contiguous()
        if deg.dim() != 2 or nmr.dim() != 2 or deg.shape[1] != EMB_DIM or nmr.shape[1] != EMB_DIM:
            # the kernels address rows of exactly 256 floats (nomad.py:55 EMB_DIM); anything else would be read misaligned
            raise ValueError(f"cdist_mean needs (n, {EMB_DIM}) and (m, {EMB_DIM}) embeddings, got {tuple(deg.shape)} "
                             f"and {tuple(nmr.shape)}")
        n, m = deg.shape[0], nmr.shape[0]
        dm = None
        if want_matrix:
            dm = out_dm if out_dm is not None else torch.empty((n, m), dtype=torch.float32, device=self.device)
            assert dm.shape == (n, m) and dm.dtype == torch.float32 and dm.is_contiguous() and dm.device == self.device
        mean = out_mean if out_mean is not None else torch.empty((n,), dtype=torch.float64, device=self.device)
        assert mean.shape == (n,) and mean.dtype == torch.float64 and mean.device == self.device
        need = self.lib.nomad_b200_cdist_workspace_bytes(n, m)
        ws = self.workspace(need)
        wp, wbytes = self._aligned(ws)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.nomad_b200_cdist_mean(_ptr(deg), n, _ptr(nmr), m, _ptr(dm), _ptr(mean), wp, wbytes,
                                                      gemm_impl, _stream_ptr()), "nomad_b200_cdist_mean")
        return dm, mean

    def paired_dist(self, a: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
        """(n, 256), (n, 256) fp32 -> (n,) fp64 distances of matching rows (the diagonal of ``cdist``)."""
        a = a.to(self.device, torch.float32).contiguous()
        b = b.to(self.device, torch.float32).contiguous()
        assert a.shape == b.shape and a.shape[1] == EMB_DIM
        out = torch.empty((a.shape[0],), dtype=torch.float64, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.nomad_b200_paired_dist(_ptr(a), _ptr(b), a.shape[0], _ptr(out), _stream_ptr()),
                       "nomad_b200_paired_dist")
        return out

    def launch_count(self) -> int:
        return int(self.lib.nomad_b200_launch_count())
