"""Native wav reader and batched device ingest for every PCM and float encoding (``nomad_b200_wav_probe_format``,
``nomad_b200_wav_read``, ``nomad_b200_ingest_batch``): headers, bytes and decoded waveforms against the host path
``audio.load_wav`` / ``audio.load_processing``, which stands in for ``torchaudio.load`` (nomad.py:192-212).  The corpus
is written by the fixtures: ``wave`` for PCM of 1-4 bytes, scipy for float32 / float64, and a small RIFF writer for
WAVE_FORMAT_EXTENSIBLE, RIFX, u-law, an odd-sized chunk before ``data`` and a truncated ``data`` chunk."""
import os
import struct
import wave

import numpy as np
import pytest
import torch

from nomad_b200 import _lib, audio
from nomad_b200.engine import Engine

RATES = (8000, 16000, 22050, 44100, 48000)
CHANNELS = (1, 2, 3)
FORMATS = (_lib.WAV_U8, _lib.WAV_S16, _lib.WAV_S24, _lib.WAV_S32, _lib.WAV_F32, _lib.WAV_F64)
GUID_TAIL = bytes.fromhex("000010008000" "00aa00389b71")


def _samples(rng, fmt, n, level=None):
    """-> (array of n samples, their little-endian data bytes).  Default: the first 16 samples span the full range of
    the format (decode edge cases), the rest stay within a quarter of it, a speech level like that of
    tests/golden/ref_ingest.npz, for which the 1e-6 bound on resampled output is stated.  ``level``: Gaussian noise of
    that standard deviation (full scale = 1) instead."""
    if level is not None:
        x = np.clip(rng.standard_normal(n) * level, -1.0, 0.99)
        if fmt in (_lib.WAV_F32, _lib.WAV_F64):
            x = x.astype("<f4" if fmt == _lib.WAV_F32 else "<f8")
            return x, x.tobytes()
        bits = 8 * int(_lib.FORMAT_BYTES[fmt])
        v = np.round(x * (1 << (bits - 1))).astype(np.int64)
        if fmt == _lib.WAV_U8:
            v = (v + 128).astype(np.uint8)
            return v, v.tobytes()
        v = v.astype("<i2" if bits == 16 else "<i4")
        return v, (v.view(np.uint8).reshape(-1, 4)[:, :3].tobytes() if bits == 24 else v.tobytes())
    quiet = np.arange(n) >= 16
    if fmt == _lib.WAV_U8:
        x = rng.integers(0, 256, n)
        x = np.where(quiet, 128 + (x - 128) // 4, x).astype(np.uint8)
        return x, x.tobytes()
    if fmt in (_lib.WAV_S16, _lib.WAV_S24, _lib.WAV_S32):
        bits = {_lib.WAV_S16: 16, _lib.WAV_S24: 24, _lib.WAV_S32: 32}[fmt]
        x = rng.integers(-(1 << (bits - 1)), 1 << (bits - 1), n)
        x = np.where(quiet, x // 4, x).astype("<i2" if bits == 16 else "<i4")
        raw = x.view(np.uint8).reshape(-1, 4)[:, :3].tobytes() if bits == 24 else x.tobytes()
        return x, raw
    x = rng.uniform(-1.0, 1.0, n)
    x = np.where(quiet, x * 0.25, x).astype("<f4" if fmt == _lib.WAV_F32 else "<f8")
    return x, x.tobytes()


def _fmt_chunk(tag, ch, sr, bits, sub=None, sub_tail=GUID_TAIL, block_align=None):
    ba = ch * bits // 8 if block_align is None else block_align
    body = struct.pack("<HHIIHH", 0xFFFE if sub is not None else tag, ch, sr, sr * ba, ba, bits)
    if sub is not None:   # WAVE_FORMAT_EXTENSIBLE: cbSize, valid bits, channel mask, sub-format GUID
        body += struct.pack("<HHI", 22, bits, 0) + struct.pack("<I", sub) + sub_tail
    return b"fmt " + struct.pack("<I", len(body)) + body


def _riff(chunks, data, data_size=None, riff=b"RIFF", data_first=False):
    """RIFF/WAVE from a fmt chunk + extra chunks, then the data chunk (``data_size`` overrides its size field)."""
    d = b"data" + struct.pack("<I", len(data) if data_size is None else data_size) + data
    body = (d + chunks) if data_first else (chunks + d)
    return riff + struct.pack("<I", 4 + len(body)) + b"WAVE" + body


def _write(path, fmt, ch, sr, frames, rng, how="plain", level=None):
    """Write one file; -> its data bytes."""
    _, raw = _samples(rng, fmt, frames * ch, level)
    bits = 8 * int(_lib.FORMAT_BYTES[fmt])
    if how == "plain" and fmt in (_lib.WAV_F32, _lib.WAV_F64):
        from scipy.io import wavfile
        x = np.frombuffer(raw, "<f4" if fmt == _lib.WAV_F32 else "<f8").reshape(frames, ch)
        wavfile.write(str(path), sr, x)
    elif how == "plain":
        with wave.open(str(path), "wb") as w:
            w.setnchannels(ch); w.setsampwidth(bits // 8); w.setframerate(sr); w.writeframes(raw)
    elif how == "extensible":
        sub = 3 if fmt in (_lib.WAV_F32, _lib.WAV_F64) else 1
        path.write_bytes(_riff(_fmt_chunk(0, ch, sr, bits, sub=sub), raw))
    elif how == "list":    # odd-sized LIST chunk (plus its pad byte) between fmt and data
        path.write_bytes(_riff(_fmt_chunk(1, ch, sr, bits) + b"LIST" + struct.pack("<I", 5) + b"INFOx\0", raw))
    elif how == "truncated":   # the data chunk claims more bytes than the file holds
        path.write_bytes(_riff(_fmt_chunk(1, ch, sr, bits), raw, data_size=len(raw) + 1000 * ch * bits // 8))
    return raw


def _native_corpus(root, frame_counts, seed=0):
    """Every format x channel count x rate x frame count, plus the EXTENSIBLE / LIST / truncated variants.
    -> list of (path, format, channels, rate, frames, data bytes)"""
    rng = np.random.default_rng(seed)
    out = []
    for fmt in FORMATS:
        for ch in CHANNELS:
            for sr in RATES:
                for n in frame_counts:
                    p = root / f"f{fmt}_c{ch}_r{sr}_n{n}.wav"
                    out.append((str(p), fmt, ch, sr, n, _write(p, fmt, ch, sr, n, rng)))
    for fmt, how, ch, sr in ((_lib.WAV_S24, "extensible", 2, 48000), (_lib.WAV_S16, "extensible", 1, 16000),
                             (_lib.WAV_F32, "extensible", 3, 22050), (_lib.WAV_F64, "extensible", 1, 16000),
                             (_lib.WAV_S16, "list", 2, 44100), (_lib.WAV_S24, "list", 1, 16000),
                             (_lib.WAV_S16, "truncated", 1, 16000), (_lib.WAV_S32, "truncated", 2, 8000)):
        n = max(frame_counts)
        p = root / f"{how}_f{fmt}_c{ch}_r{sr}.wav"
        out.append((str(p), fmt, ch, sr, n, _write(p, fmt, ch, sr, n, rng, how)))
    return out


def _rejected_files(root):
    """Files the native reader must leave to the host path (frames = -1)."""
    rng = np.random.default_rng(5)
    pcm = rng.integers(-3000, 3000, 600).astype(np.int16)
    files = {}
    # RIFX: big-endian container (scipy reads it)
    body = b"fmt " + struct.pack(">IHHIIHH", 16, 1, 1, 16000, 32000, 2, 16)
    body += b"data" + struct.pack(">I", 2 * len(pcm)) + pcm.astype(">i2").tobytes()
    files["rifx"] = b"RIFX" + struct.pack(">I", 4 + len(body)) + b"WAVE" + body
    files["ulaw"] = _riff(_fmt_chunk(7, 1, 8000, 8), bytes(range(256)))
    files["alaw"] = _riff(_fmt_chunk(6, 1, 8000, 8), bytes(range(256)))
    files["adpcm"] = _riff(_fmt_chunk(2, 1, 8000, 4, block_align=256), bytes(512))
    files["data_first"] = _riff(_fmt_chunk(1, 1, 16000, 16), pcm.tobytes(), data_first=True)
    files["float16"] = _riff(_fmt_chunk(3, 1, 16000, 16), pcm.tobytes())
    files["pcm12"] = _riff(_fmt_chunk(1, 1, 16000, 12, block_align=2), pcm.tobytes())
    files["bad_align"] = _riff(_fmt_chunk(1, 2, 16000, 16, block_align=2), pcm.tobytes())
    files["ext_bad_guid"] = _riff(_fmt_chunk(0, 1, 16000, 16, sub=1, sub_tail=bytes(12)), pcm.tobytes())
    files["ext_ulaw"] = _riff(_fmt_chunk(0, 1, 8000, 8, sub=7), bytes(range(256)))
    files["garbage"] = b"not a wav file at all"
    paths = {}
    for k, v in files.items():
        (root / f"{k}.wav").write_bytes(v)
        paths[k] = str(root / f"{k}.wav")
    paths["missing"] = str(root / "missing.wav")
    return paths


@pytest.fixture(scope="module")
def host_corpus(tmp_path_factory):
    root = tmp_path_factory.mktemp("formats")
    return _native_corpus(root, (0, 1, 1001)), _rejected_files(root)


# ---------------------------------------------------------------------------------------------- host, no GPU
def test_probe_format_matches_the_host_decoder(host_corpus):
    native, _ = host_corpus
    probe = _lib.wav_probe_format([c[0] for c in native], 3)
    for i, (path, fmt, ch, sr, n, raw) in enumerate(native):
        w, got_sr = audio.load_wav(path)
        assert (probe.sample_rate[i], probe.channels[i], probe.format[i]) == (got_sr, w.shape[0], fmt), path
        assert probe.frames[i] == w.shape[1] == n, path
        assert probe.data_offset[i] > 0


def test_read_returns_the_data_bytes(host_corpus):
    native, _ = host_corpus
    paths = [c[0] for c in native]
    probe = _lib.wav_probe_format(paths, 2)
    n_bytes = probe.frames * probe.channels * _lib.FORMAT_BYTES[probe.format]
    dst = np.zeros(len(paths), np.int64)
    np.cumsum((n_bytes[:-1] + 15) // 16 * 16, out=dst[1:])
    buf = np.full(int(dst[-1] + n_bytes[-1]) + 16, 0xA5, np.uint8)
    _lib.wav_read(paths, probe.data_offset, n_bytes, dst, buf.ctypes.data, 4)
    for i, c in enumerate(native):
        assert buf[dst[i]: dst[i] + n_bytes[i]].tobytes() == c[5], c[0]
    assert (buf[int(dst[-1] + n_bytes[-1]):] == 0xA5).all()


def test_unhandled_files_are_rejected(host_corpus):
    _, rejected = host_corpus
    probe = _lib.wav_probe_format(list(rejected.values()), 2)
    for k, fr, fmt in zip(rejected, probe.frames, probe.format):
        assert fr == -1 and fmt == 0, k
    # the host path still reads the RIFX file
    w, sr = audio.load_wav(rejected["rifx"])
    assert sr == 16000 and w.shape == (1, 600)


def test_pcm16_probe_still_accepts_only_16_bit_pcm(host_corpus):
    native, rejected = host_corpus
    paths = [c[0] for c in native] + list(rejected.values())
    sr, ch, fr, off = _lib.wav_probe(paths, 3)
    full = _lib.wav_probe_format(paths, 3)
    s16 = full.format == _lib.WAV_S16
    assert s16.sum() > 40
    np.testing.assert_array_equal(fr, np.where(s16, full.frames, -1))
    np.testing.assert_array_equal(off, np.where(s16, full.data_offset, 0))
    np.testing.assert_array_equal(sr[s16], full.sample_rate[s16])
    np.testing.assert_array_equal(ch[s16], full.channels[s16])


def test_shard_cost_is_the_16k_output_length(host_corpus):
    from nomad_b200.dist import shard_costs
    native, rejected = host_corpus
    paths = [c[0] for c in native] + [rejected["rifx"], rejected["ulaw"]]
    costs = shard_costs(paths, 2)
    lib = _lib.load()
    for c, cost in zip(native, costs):
        assert cost == lib.nomad_b200_ingest_out_samples(c[4], c[3], 16000, 0), c[0]
    assert costs[-2:] == [float(os.path.getsize(rejected["rifx"])), float(os.path.getsize(rejected["ulaw"]))]


def test_ingest_workspace_rejects_bad_descriptors():
    lib = _lib.load()
    items = np.zeros(2, _lib.INGEST_ITEM)
    items["n_frames"], items["channels"], items["sample_rate"], items["format"] = 1000, 1, 16000, _lib.WAV_S16
    items["out_samples"], items["byte_offset"] = 1000, (0, 2048)
    ws = lambda it: lib.nomad_b200_ingest_workspace_bytes(it.ctypes.data_as(_lib.c_vp), len(it), 16000)
    assert ws(items) > 0
    for field, value, message in (("out_samples", 1001, b"output samples"), ("format", 9, b"sample format"),
                                  ("byte_offset", 3, b"not aligned"), ("channels", 0, b"bad descriptor")):
        bad = items.copy()
        bad[field][1] = value
        assert ws(bad) == 0 and message in lib.nomad_b200_last_error(), field


# ------------------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def engine(state_dict):
    return Engine(state_dict, 0)


@pytest.mark.gpu
def test_device_ingest_equals_host_path_for_every_encoding(engine, tmp_path):
    """(a) ``load_processing_device`` vs ``load_processing``: bit-identical at 16 kHz, <= 1e-6 resampled."""
    (tmp_path / "one").mkdir()
    native = _native_corpus(tmp_path, (1001,), seed=1)
    native += [c for c in _native_corpus(tmp_path / "one", (1,), seed=2) if c[3] == 16000]   # one frame: 16 kHz only
    worst = 0.0
    for path, fmt, ch, sr, n, _ in native:
        dev = audio.load_processing_device(engine, path).cpu()
        host = audio.load_processing(path)
        assert dev.shape == host.shape, path
        err = float((dev - host).abs().max()) if dev.numel() else 0.0
        if sr == 16000:
            assert torch.equal(dev, host), path
        else:
            assert err <= 1e-6, (path, err)
            worst = max(worst, err)
    # trim (nomad.py:208-210) through the output count, here on a 10.5 s 48 kHz S24 stereo file and a 16 kHz F32 one
    rng = np.random.default_rng(3)
    for fmt, sr in ((_lib.WAV_S24, 48000), (_lib.WAV_F32, 16000)):
        p = tmp_path / f"long_{fmt}.wav"
        _write(p, fmt, 2, sr, int(sr * 10.5), rng, "extensible" if fmt == _lib.WAV_S24 else "plain")
        dev = audio.load_processing_device(engine, str(p), trim=True).cpu()
        host = audio.load_processing(str(p), trim=True)
        assert dev.shape == host.shape == (1, 160000)
        assert float((dev - host).abs().max()) <= (0.0 if sr == 16000 else 1e-6)
    print("max-abs resampled", worst)


@pytest.mark.gpu
def test_batched_s16_items_equal_ingest_pcm16(engine, tmp_path):
    """(b) S16 items of one ``nomad_b200_ingest_batch`` call == ``nomad_b200_ingest_pcm16`` per file, bit for bit."""
    rng = np.random.default_rng(4)
    paths, pcms = [], []
    for sr in RATES:
        for ch in CHANNELS:
            n = int(rng.integers(400, 5000)) | 1
            pcm = rng.integers(-32768, 32768, (n, ch)).astype("<i2")
            p = tmp_path / f"s16_{sr}_{ch}.wav"
            with wave.open(str(p), "wb") as w:
                w.setnchannels(ch); w.setsampwidth(2); w.setframerate(sr); w.writeframes(pcm.tobytes())
            paths.append(str(p)); pcms.append((pcm, sr))
    for trim in (False, True):
        probe = _lib.wav_probe_format(paths, 2)
        n_out = _lib.ingest_out_samples(probe.frames, probe.sample_rate, 16000, trim)
        off = Engine.offsets(n_out)
        out = torch.full((int(off[-1]),), float("nan"), dtype=torch.float32, device=engine.device)
        engine.ingest_wav_files(paths, probe, n_out, out, off[:-1], 3)
        got = out.cpu()
        for i, (pcm, sr) in enumerate(pcms):
            ref = engine.ingest_pcm16(pcm, sr, 16000, trim)[0].cpu()
            assert torch.equal(got[off[i]:off[i + 1]], ref), (paths[i], trim)


@pytest.mark.gpu
def test_launches_per_batch_do_not_grow_with_the_file_count(engine, tmp_path):
    """(d) one launch for the 16 kHz items + one per distinct other rate, whatever the number of files."""
    rng = np.random.default_rng(6)
    paths = []
    for i in range(40):
        fmt, ch, sr = FORMATS[i % 6], CHANNELS[i % 3], (16000, 44100, 48000, 8000)[i % 4]
        p = tmp_path / f"l{i}.wav"
        _write(p, fmt, ch, sr, int(rng.integers(500, 3000)), rng)
        paths.append(str(p))
    for k in (1, 4, 13, 40):
        probe = _lib.wav_probe_format(paths[:k], 2)
        n_out = _lib.ingest_out_samples(probe.frames, probe.sample_rate)
        off = Engine.offsets(n_out)
        out = torch.empty((int(off[-1]),), dtype=torch.float32, device=engine.device)
        n0 = engine.launch_count()
        engine.ingest_wav_files(paths[:k], probe, n_out, out, off[:-1], 2)
        rates = set(int(r) for r in probe.sample_rate)
        assert engine.launch_count() - n0 == int(16000 in rates) + len(rates - {16000}), k


@pytest.mark.gpu
def test_embed_files_mixed_corpus_equals_per_file_loop(state_dict, tmp_path):
    """(c) ``Nomad.embed_files`` on a corpus of every encoding plus RIFX files (host fallback, packed into the same
    batches) vs the reference's per-file host loop: bit-identical at 16 kHz, <= 1e-4 on resampled files.  The model runs
    in precision='fp32': with fp16 operands its own rounding (3.5e-4 against fp32) is of the order of the bound, and the
    <= 1e-6 waveform difference of the resampler was seen to move an embedding of a 22.05 kHz file by 1.2e-4."""
    from nomad_b200.nomad import Nomad
    rng = np.random.default_rng(7)
    paths, rates = [], []
    for i in range(30):
        fmt, ch, sr = FORMATS[i % 6], CHANNELS[i % 3], (16000, 16000, 22050, 44100, 48000)[i % 5]
        p = tmp_path / f"m{i:02d}.wav"
        _write(p, fmt, ch, sr, int(sr * rng.uniform(0.3, 6.0)), rng, "extensible" if i % 7 == 3 else "plain",
               level=3000 / 32768)
        paths.append(str(p)); rates.append(sr)
    for i in range(3):   # RIFX 16-bit: not read natively
        pcm = rng.integers(-20000, 20000, 4000 + 777 * i).astype(np.int16)
        body = b"fmt " + struct.pack(">IHHIIHH", 16, 1, 1, 16000, 32000, 2, 16)
        body += b"data" + struct.pack(">I", 2 * len(pcm)) + pcm.astype(">i2").tobytes()
        p = tmp_path / f"x{i}.wav"
        p.write_bytes(b"RIFX" + struct.pack(">I", 4 + len(body)) + b"WAVE" + body)
        paths.insert(5 * i + 2, str(p)); rates.insert(5 * i + 2, 16000)
    assert (_lib.wav_probe_format(paths).frames < 0).sum() == 3
    nomad = Nomad(state_dict=state_dict, precision="fp32")
    nomad.window_files = 11
    fast = nomad.embed_files(np.array(paths)).cpu().numpy()
    ref = np.stack([nomad.engine.embed([nomad.load_processing(p).reshape(-1)]).cpu().numpy()[0] for p in paths])
    for i, p in enumerate(paths):
        if rates[i] == 16000:
            np.testing.assert_array_equal(fast[i], ref[i], err_msg=p)
        else:
            assert np.abs(fast[i] - ref[i]).max() <= 1e-4, p


@pytest.mark.gpu
def test_short_files_raise_the_reference_error(state_dict, tmp_path):
    """(e) fewer than 400 output samples: today's RuntimeError, whatever the encoding."""
    from nomad_b200.nomad import Nomad
    rng = np.random.default_rng(8)
    nomad = Nomad(state_dict=state_dict)
    ok = tmp_path / "ok.wav"
    _write(ok, _lib.WAV_S16, 1, 16000, 4000, rng)
    for fmt, sr, n in ((_lib.WAV_S24, 48000, 1000), (_lib.WAV_F32, 16000, 399), (_lib.WAV_U8, 8000, 199)):
        p = tmp_path / f"short_{fmt}.wav"
        _write(p, fmt, 2, sr, n, rng)
        with pytest.raises(RuntimeError, match=r"Kernel size can't be greater than actual input size"):
            nomad.embed_files(np.array([str(ok), str(p)]))
