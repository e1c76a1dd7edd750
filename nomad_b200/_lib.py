"""ctypes binding of ``libnomad_b200.so`` (the C ABI declared in ``include/nomad_b200.h``).

The product path has no CPU fallback: if the shared library is missing this module raises, it never
routes around it.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import NamedTuple

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("NOMAD_B200_LIB") or os.path.join(_HERE, "csrc", "libnomad_b200.so")  # override: kernel A/B probes

c_i64 = C.c_int64
c_vp = C.c_void_p


# NOMAD_B200_WAV_* sample formats -> bytes per sample
WAV_U8, WAV_S16, WAV_S24, WAV_S32, WAV_F32, WAV_F64 = 1, 2, 3, 4, 5, 6
FORMAT_BYTES = np.array([0, 1, 2, 3, 4, 4, 8], np.int64)

# ``nomad_b200_ingest_item``
INGEST_ITEM = np.dtype([("byte_offset", "<i8"), ("n_frames", "<i8"), ("out_offset", "<i8"), ("out_samples", "<i8"),
                        ("channels", "<i4"), ("format", "<i4"), ("sample_rate", "<i4"), ("reserved", "<i4")])


class Tensor(C.Structure):
    """``nomad_b200_tensor``"""
    _fields_ = [("name", C.c_char_p), ("data", c_vp), ("numel", c_i64)]


# name -> (restype, argtypes): mirrors include/nomad_b200.h one to one
PROTOTYPES = {
    "nomad_b200_last_error": (C.c_char_p, []),
    "nomad_b200_version": (C.c_char_p, []),
    "nomad_b200_create": (C.c_int, [C.POINTER(c_vp), C.POINTER(Tensor), C.c_int, C.c_int, C.c_int]),
    "nomad_b200_set_precision": (C.c_int, [c_vp, C.c_int]),
    "nomad_b200_get_precision": (C.c_int, [c_vp]),
    "nomad_b200_destroy": (C.c_int, [c_vp]),
    "nomad_b200_set_gemm_impl": (C.c_int, [c_vp, C.c_int]),
    "nomad_b200_set_loss_head": (C.c_int, [c_vp, c_vp, c_vp]),
    "nomad_b200_embed_workspace_bytes": (C.c_size_t, [C.POINTER(c_i64), C.c_int]),
    "nomad_b200_embed_workspace_bytes_mode": (C.c_size_t, [C.POINTER(c_i64), C.c_int, C.c_int]),
    "nomad_b200_layers_workspace_bytes_mode": (C.c_size_t, [C.c_int, c_i64, C.c_int]),
    "nomad_b200_score_workspace_bytes_mode": (C.c_size_t, [C.POINTER(c_i64), C.c_int, c_i64, C.c_int]),
    "nomad_b200_embed": (C.c_int, [c_vp, c_vp, C.POINTER(c_i64), C.c_int, c_vp, c_vp, C.c_size_t, c_vp]),
    "nomad_b200_embed_host": (C.c_int, [c_vp, c_vp, C.POINTER(c_i64), C.c_int, c_vp, c_vp, C.c_size_t, c_vp]),
    "nomad_b200_loss_workspace_bytes": (C.c_size_t, [C.c_int, c_i64, C.c_int]),
    "nomad_b200_loss_fwd_bwd": (C.c_int, [c_vp, c_vp, c_vp, C.c_int, c_i64, C.c_float, c_vp, c_vp, c_vp,
                                          C.c_size_t, c_vp]),
    "nomad_b200_layers_workspace_bytes": (C.c_size_t, [C.c_int, c_i64]),
    "nomad_b200_num_frames": (c_i64, [c_i64]),
    "nomad_b200_layers_fwd": (C.c_int, [c_vp, c_vp, C.c_int, c_i64, c_vp, c_vp, c_vp, C.c_size_t, c_vp]),
    "nomad_b200_cdist_workspace_bytes": (C.c_size_t, [c_i64, c_i64]),
    "nomad_b200_cdist_mean": (C.c_int, [c_vp, c_i64, c_vp, c_i64, c_vp, c_vp, c_vp, C.c_size_t, C.c_int, c_vp]),
    "nomad_b200_cdist_mean_host": (C.c_int, [c_vp, c_i64, c_vp, c_i64, c_vp, c_vp, c_vp, C.c_size_t, c_vp]),
    "nomad_b200_score_workspace_bytes": (C.c_size_t, [C.POINTER(c_i64), C.c_int, c_i64]),
    "nomad_b200_score": (C.c_int, [c_vp, c_vp, C.POINTER(c_i64), C.c_int, c_vp, c_i64, c_vp, c_vp, c_vp, c_vp, C.c_size_t,
                                   c_vp]),
    "nomad_b200_score_host": (C.c_int, [c_vp, c_vp, C.POINTER(c_i64), C.c_int, c_vp, c_i64, c_vp, c_vp, c_vp, c_vp,
                                        C.c_size_t, c_vp]),
    "nomad_b200_gemm_f16": (C.c_int, [c_vp, c_i64, c_i64, C.c_int, c_vp, C.c_int, C.c_int, C.c_int, C.c_int,
                                       c_i64, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, c_i64, C.c_int, C.c_int, c_vp]),
    "nomad_b200_refresh_weights": (C.c_int, [c_vp, C.POINTER(Tensor), C.c_int, c_vp]),
    "nomad_b200_debug_read_weight": (C.c_int, [c_vp, C.c_char_p, c_vp, C.c_size_t]),
    "nomad_b200_triplet_grad_floats": (c_i64, []),
    "nomad_b200_triplet_grad_segment": (C.c_int, [C.c_int, C.c_char_p, C.c_int, C.POINTER(c_i64), C.POINTER(c_i64)]),
    "nomad_b200_triplet_workspace_bytes": (C.c_size_t, [C.c_int, c_i64]),
    "nomad_b200_triplet_fwd_bwd": (C.c_int, [c_vp, c_vp, C.c_int, c_i64, C.c_float, c_vp, c_vp, C.POINTER(C.c_float), c_vp,
                                             C.c_size_t, c_vp]),
    "nomad_b200_gemm_split": (C.c_int, [c_vp, c_vp, c_i64, c_vp, c_vp, C.c_int, C.c_int, C.c_int, C.c_float, c_vp, c_vp, c_vp,
                                        c_vp, c_i64, C.c_int, c_vp]),
    "nomad_b200_write_scores_csv": (C.c_int, [C.c_char_p, C.c_char_p, C.POINTER(C.c_char_p), c_i64, C.POINTER(C.c_char_p),
                                               c_i64, c_vp, C.c_int, C.c_int]),
    "nomad_b200_paired_dist": (C.c_int, [c_vp, c_vp, c_i64, c_vp, c_vp]),
    "nomad_b200_ingest_out_samples": (c_i64, [c_i64, C.c_int, C.c_int, C.c_int]),
    "nomad_b200_ingest_pcm16": (C.c_int, [c_vp, c_i64, C.c_int, C.c_int, C.c_int, C.c_int, c_vp, c_vp]),
    "nomad_b200_wav_probe": (C.c_int, [C.POINTER(C.c_char_p), c_i64, c_vp, c_vp, c_vp, c_vp, C.c_int]),
    "nomad_b200_wav_read_pcm16": (C.c_int, [C.POINTER(C.c_char_p), c_i64, c_vp, c_vp, c_vp, c_vp, C.c_int]),
    "nomad_b200_wav_probe_format": (C.c_int, [C.POINTER(C.c_char_p), c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, C.c_int]),
    "nomad_b200_wav_read": (C.c_int, [C.POINTER(C.c_char_p), c_i64, c_vp, c_vp, c_vp, c_vp, C.c_int]),
    "nomad_b200_ingest_workspace_bytes": (C.c_size_t, [c_vp, c_i64, C.c_int]),
    "nomad_b200_ingest_batch": (C.c_int, [c_vp, c_vp, c_i64, C.c_int, c_vp, c_vp, C.c_size_t, c_vp]),
    "nomad_b200_attention_workspace_bytes": (C.c_size_t, [C.POINTER(C.c_int32), C.c_int]),
    "nomad_b200_attention_f16": (C.c_int, [c_vp, c_i64, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.c_int, c_vp, c_vp,
                                            c_vp, C.c_size_t, c_vp]),
    "nomad_b200_profile_gemm": (C.c_int, [C.c_int]),
    "nomad_b200_profile_gemm_read": (C.c_int, [C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(c_i64)]),
    "nomad_b200_launch_count": (c_i64, []),
}

_lib = None


class NomadB200Error(RuntimeError):
    pass


def load() -> C.CDLL:
    """Load the shared library (once) and attach prototypes.  Raises if it was not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise NomadB200Error(
            f"{LIB_PATH} not found: build it with `make -C nomad_b200/csrc` (or `python -c 'import "
            f"__graft_entry__ as g; g.build()'`). nomad_b200 has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)  # AttributeError here = header/library mismatch: fail loudly
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(status: int, what: str = "") -> None:
    if status != 0:
        msg = load().nomad_b200_last_error().decode("utf-8", "replace")
        raise NomadB200Error(f"{what or 'nomad_b200 call'} failed: {msg}")


def write_scores_csv(path, index_name, row_labels, col_labels, values, decimals=3, threads=0) -> None:
    """``DataFrame(values, index=row_labels, columns=col_labels).round(decimals)`` + ``to_csv`` with ``index_name`` as
    the first header cell, byte for byte, from a float64 (n, m) array -- nomad_b200_write_scores_csv."""
    import numpy as np
    values = np.ascontiguousarray(values, dtype=np.float64)
    if values.ndim == 1:
        values = values[:, None]
    n, m = values.shape
    assert len(row_labels) == n and len(col_labels) == m
    rl = (C.c_char_p * max(n, 1))(*[str(x).encode("utf-8") for x in row_labels])
    cl = (C.c_char_p * max(m, 1))(*[str(x).encode("utf-8") for x in col_labels])
    check(load().nomad_b200_write_scores_csv(str(path).encode("utf-8"), str(index_name).encode("utf-8"), rl, n, cl, m,
                                             values.ctypes.data_as(c_vp), int(decimals), int(threads)),
          "nomad_b200_write_scores_csv")


def wav_probe(paths, threads=0):
    """-> (sample_rate int32[n], channels int32[n], frames int64[n] (-1: not 16-bit PCM wav), data_offset int64[n])"""
    import numpy as np
    n = len(paths)
    arr = (C.c_char_p * max(n, 1))(*[str(p).encode("utf-8") for p in paths])
    sr, ch = np.zeros(n, np.int32), np.zeros(n, np.int32)
    fr, off = np.full(n, -1, np.int64), np.zeros(n, np.int64)
    check(load().nomad_b200_wav_probe(arr, n, sr.ctypes.data_as(c_vp), ch.ctypes.data_as(c_vp), fr.ctypes.data_as(c_vp),
                                     off.ctypes.data_as(c_vp), int(threads)), "nomad_b200_wav_probe")
    return sr, ch, fr, off


class WavProbe(NamedTuple):
    """Per-file header fields from ``nomad_b200_wav_probe_format``; frames = -1 (format 0): not read natively."""
    sample_rate: np.ndarray   # int32
    channels: np.ndarray      # int32
    frames: np.ndarray        # int64
    data_offset: np.ndarray   # int64
    format: np.ndarray        # int32, WAV_*

    def take(self, idx) -> "WavProbe":
        return WavProbe(*(a[idx] for a in self))

    @staticmethod
    def unread(n: int) -> "WavProbe":
        """n files left to the host decoder"""
        return WavProbe(np.zeros(n, np.int32), np.zeros(n, np.int32), np.full(n, -1, np.int64), np.zeros(n, np.int64),
                        np.zeros(n, np.int32))


def wav_probe_format(paths, threads=0) -> WavProbe:
    n = len(paths)
    arr = (C.c_char_p * max(n, 1))(*[str(p).encode("utf-8") for p in paths])
    p = WavProbe.unread(n)
    check(load().nomad_b200_wav_probe_format(arr, n, *(a.ctypes.data_as(c_vp) for a in p), int(threads)),
          "nomad_b200_wav_probe_format")
    return p


def ingest_out_samples(frames, sample_rate, target_sr=16000, trim=False) -> np.ndarray:
    """``nomad_b200_ingest_out_samples`` per file (-1 where frames < 0)."""
    frames = np.asarray(frames, np.int64)
    sample_rate = np.asarray(sample_rate, np.int64)
    out = np.where(frames >= 0, frames, -1)
    f = load().nomad_b200_ingest_out_samples
    for i in np.flatnonzero((frames >= 0) & ((sample_rate != target_sr) | bool(trim))):
        out[i] = f(int(frames[i]), int(sample_rate[i]), int(target_sr), int(bool(trim)))
    return out


def wav_read(paths, src_offset, n_bytes, dst_offset, dst_ptr, threads=0):
    """Read n_bytes[i] bytes of file i from byte src_offset[i] to (char*) dst_ptr + dst_offset[i] with host threads."""
    n = len(paths)
    arr = (C.c_char_p * max(n, 1))(*[str(p).encode("utf-8") for p in paths])
    a = [np.ascontiguousarray(x, dtype=np.int64) for x in (src_offset, n_bytes, dst_offset)]
    check(load().nomad_b200_wav_read(arr, n, *(x.ctypes.data_as(c_vp) for x in a), c_vp(dst_ptr), int(threads)),
          "nomad_b200_wav_read")


def wav_read_pcm16(paths, data_offset, n_samples, dst_offset, dst_ptr, threads=0):
    """Read the samples of every file into (int16*) dst_ptr + dst_offset[i] with host threads."""
    import numpy as np
    n = len(paths)
    arr = (C.c_char_p * max(n, 1))(*[str(p).encode("utf-8") for p in paths])
    a = [np.ascontiguousarray(x, dtype=np.int64) for x in (data_offset, n_samples, dst_offset)]
    check(load().nomad_b200_wav_read_pcm16(arr, n, a[0].ctypes.data_as(c_vp), a[1].ctypes.data_as(c_vp),
                                          a[2].ctypes.data_as(c_vp), c_vp(dst_ptr), int(threads)), "nomad_b200_wav_read_pcm16")
