"""Host-side mirror of the reference's ``nomad_audio.nomad`` module (``src/nomad_audio/nomad.py``).

Same class and method names, argument meaning, return values, CSV formats and error messages as the
reference; the arithmetic (wav2vec 2.0 base forward, pooled head, pairwise distance, loss and its
backward) runs in ``libnomad_b200.so`` on a B200.  Differences that are deliberate:

* files are embedded in length-bucketed batches instead of one by one (``nomad.py:166-189``); every
  utterance is still computed exactly as if alone (length-masked), so results equal the per-file loop;
* there is no CPU path: ``device='cpu'`` raises;
* weights come from ``pt-models/nomad_best_model.pt`` (or ``$NOMAD_B200_CHECKPOINT``) when present,
  else seeded random-init of the identical architecture -- nothing is downloaded at import;
* ``forward`` back-propagates to ``estimate`` only (dgrad chain, wheel 0.0.8 semantics: the NOMAD
  network's own parameters receive no ``.grad``).
"""
from __future__ import annotations

import os
from datetime import datetime
from typing import List, Optional, Sequence

import numpy as np
import pandas as pd
import torch
import torch.nn as nn
import torch.nn.functional as F

from . import audio
from .engine import Engine, MIN_SAMPLES
from .weights import EMB_DIM, SSL_OUT_DIM, load_state_dict

w2v_path = 'pt-models/wav2vec_small.pt'        # kept for API compatibility (nomad.py:21); unused
nomad_path = 'pt-models/nomad_best_model.pt'   # nomad.py:29


def plan_batches(lengths: Sequence[int], max_samples: int) -> List[List[int]]:
    """Length-bucketed batches: indices sorted by length, cut when the sample budget is reached.
    Returns index lists; results are scattered back so output order == input order."""
    order = sorted(range(len(lengths)), key=lambda i: (lengths[i], i))
    batches, cur, tot = [], [], 0
    for i in order:
        n = int(lengths[i])
        if cur and tot + n > max_samples:
            batches.append(cur)
            cur, tot = [], 0
        cur.append(i)
        tot += n
    if cur:
        batches.append(cur)
    return batches


class TripletModel:
    """``TripletModel`` (``nomad.py:214-231``): ``model(wav, lengths=None) -> (B, 256)`` unit-norm."""

    def __init__(self, engine: Engine):
        self.engine = engine
        self.ssl_features = SSL_OUT_DIM

    def eval(self):
        return self

    def to(self, *_a, **_k):
        return self

    def __call__(self, wav, lengths=None):  # ``lengths`` accepted and ignored, as in the reference
        return self.forward(wav, lengths)

    @torch.no_grad()
    def forward(self, wav: torch.Tensor, lengths=None) -> torch.Tensor:
        if wav.dim() == 3:
            wav = wav.squeeze(1)  # nomad.py:225
        if wav.dim() == 1:
            wav = wav.unsqueeze(0)
        B, N = wav.shape
        flat = wav.to(self.engine.device, torch.float32).contiguous().reshape(-1)
        return self.engine.embed_packed(flat, np.arange(B + 1, dtype=np.int64) * N)


class LossNetLayers:
    """``LossNetLayers`` (``nomad.py:233-258``): 12 transformer-layer outputs + the head output."""

    def __init__(self, engine: Engine):
        self.engine = engine
        self.ssl_features = SSL_OUT_DIM
        # freshly initialised head, exactly like the reference (nomad.py:238-241)
        self.embedding_layer = nn.Sequential(nn.ReLU(), nn.Linear(SSL_OUT_DIM, EMB_DIM))
        self._synced = None

    def to(self, *_a, **_k):
        return self

    def sync_head(self):
        lin = self.embedding_layer[1]
        key = (lin.weight._version, lin.bias._version, lin.weight.data_ptr(), lin.bias.data_ptr())
        if key != self._synced:
            self.engine.set_loss_head(lin.weight, lin.bias)
            self._synced = key

    def __call__(self, wav):
        return self.forward(wav)

    @torch.no_grad()
    def forward(self, wav: torch.Tensor) -> List[torch.Tensor]:
        self.sync_head()
        layers, emb = self.engine.layers(wav)
        return [layers[i] for i in range(layers.shape[0])] + [emb]


class NomadLoss(nn.Module):
    """``NomadLoss`` (``nomad.py:260-282``) on already-computed feature lists."""

    def __init__(self):
        super().__init__()
        self.L = 13
        self.only_embedding = False

    def forward(self, nomad_ref, nomad_test):
        l1_dist = 0.0
        for i in range(self.L):
            l1_dist = l1_dist + F.l1_loss(nomad_test[i], nomad_ref[i])
        return l1_dist


class _NomadLossFn(torch.autograd.Function):
    """loss = sum_i mean|H_i(est) - H_i(clean)|; d loss / d est comes back from the same C call."""

    @staticmethod
    def forward(ctx, estimate, clean, owner):
        need_grad = estimate.requires_grad
        loss, grad = owner.engine.loss_fwd_bwd(estimate, clean, owner.feature_grad_mult, with_grad=need_grad)
        ctx.shape = estimate.shape
        ctx.out_device = estimate.device
        ctx.out_dtype = estimate.dtype
        ctx.save_for_backward(grad if grad is not None else torch.empty(0))
        out = loss.to(estimate.device)
        return out

    @staticmethod
    def backward(ctx, grad_out):
        (g,) = ctx.saved_tensors
        if g.numel() == 0:
            return None, None, None
        ge = (g * grad_out.to(g.device)).reshape(ctx.shape).to(ctx.out_device, ctx.out_dtype)
        return ge, None, None


class Nomad():
    def __init__(self, device=None, checkpoint: Optional[str] = None, seed: int = 1234,
                 feature_grad_mult: float = 0.1, max_batch_seconds: float = 2000.0, state_dict=None,
                 precision: Optional[str] = None, keep_state_dict: bool = False):
        # *** DEVICE SETTINGS *** (nomad.py:38-49)
        if torch.cuda.is_available():
            self.DEVICE = 'cuda'
        else:
            self.DEVICE = 'cpu'
        if device is not None:
            self.DEVICE = device
        if not str(self.DEVICE).startswith('cuda'):
            raise RuntimeError(f"nomad_b200 runs on CUDA (B200, sm_100a) only; device={self.DEVICE!r} has no "
                               "implementation here (there is no CPU fallback)")
        print(f'NOMAD running on: {self.DEVICE}')
        dev = torch.device(self.DEVICE)
        index = dev.index if dev.index is not None else torch.cuda.current_device()

        # *** LOAD MODEL *** (nomad.py:51-68): tensors only, no fairseq needed
        if state_dict is None:
            state_dict, self.weights_source = load_state_dict(checkpoint, seed)
        else:
            self.weights_source = "state_dict"
        # arithmetic class of the scoring path: "fp16" (tensor-core operands in fp16, scores within 1e-3 of the
        # reference's fp32 arithmetic) or "fp32" (split operands, within 1e-5); the loss path always runs "fp16"
        self.precision = precision or os.environ.get("NOMAD_B200_PRECISION", "fp16")
        self.engine = Engine(state_dict, index, self.precision)
        self.state_dict_ref = state_dict if keep_state_dict else None   # fine-tuning (triplet.py) needs the fp32 tensors
        self.model = TripletModel(self.engine)
        # NOMAD loss model shares the same network (nomad.py:70-72)
        self.lossnet_layers = LossNetLayers(self.engine)
        self.nomad_loss = NomadLoss()
        # fairseq applies GradMultiply(feature_grad_mult) to the conv features (wav2vec 2.0 base: 0.1)
        self.feature_grad_mult = float(feature_grad_mult)
        self.max_batch_samples = int(max_batch_seconds * 16000)
        self.device_ingest = os.environ.get("NOMAD_B200_DEVICE_INGEST", "1") != "0"
        self.window_files = int(os.environ.get("NOMAD_B200_WINDOW_FILES", "1024"))
        self.reader_threads = int(os.environ.get("NOMAD_B200_READER_THREADS", str(min(16, os.cpu_count() or 4))))

    def predict(self, mode='dir', nmr='data/nmr-data', deg='data/test-data', results_path=None):
        if nmr is None:
            raise Exception('nmr_path not specified, you need to pass a valid value to nmr_path')
        if deg is None:
            raise Exception('test_path not specified, you need to pass a valide value to test_path')

        if mode == 'dir':
            if os.path.isdir(nmr) == False:
                raise Exception(f'Path to the non-matching reference files {nmr} does not exist')
            if os.path.isdir(deg) == False:
                raise Exception(f'Path to the test files {deg} does not exist')
        elif mode == 'csv':
            if os.path.isfile(nmr) == False:
                raise Exception(f'File {nmr} does not exist')
            if os.path.isfile(deg) == False:
                raise Exception(f'File {deg} does not exist')
        else:
            raise Exception(f'Mode value {mode} is not valid. Valid values are dir and csv')

        print(f'Compute non-matching reference embeddings from {nmr}')
        nmr_embeddings = self.get_embeddings(nmr).set_index('filename')

        print(f'Compute degraded embeddings from {deg}')
        test_embeddings = self.get_embeddings(deg).set_index('filename')

        # Pairwise distance matrix + row mean (nomad.py:108,111) on the GPU
        distance_matrix, avg_nomad = self.pairwise(test_embeddings, nmr_embeddings)

        return self.write_results(list(test_embeddings.index), list(nmr_embeddings.index), distance_matrix, avg_nomad,
                                  results_path)

    def write_results(self, test_index, nmr_index, distance_matrix, avg_nomad, results_path=None):
        """DataFrame assembly + the two CSVs, byte-compatible with the reference (``nomad.py:113-140``)."""
        test_files = [x.split('/')[-1].split('.')[0] for x in test_index]
        df_avg_nomad = pd.DataFrame({'Test File': test_files, 'NOMAD': avg_nomad}).set_index('Test File').round(3)

        df_dm = None
        if distance_matrix is not None:  # None: the rows were written per rank (dist.predict_sharded, matrix='local')
            df_dm = pd.DataFrame(distance_matrix).round(3)
            df_dm['Test File'] = test_files
            df_dm.set_index('Test File', inplace=True)
            df_dm.columns = [x.split('/')[-1].split('.')[0] for x in nmr_index]

        # Save results (nomad.py:122-139)
        if results_path == None:
            now = datetime.now()
            dt_string = now.strftime("%d-%m-%Y_%H-%M-%S")
            results_avg_path = os.path.join('results-csv', dt_string)
            if os.path.isdir(results_avg_path) == False:
                os.makedirs(results_avg_path)
            results_scores_path = os.path.join('results-csv', dt_string)
            if os.path.isdir(results_scores_path) == False:
                os.makedirs(results_scores_path)
            results_avg_path = os.path.join(results_avg_path, f'{dt_string}_nomad_avg.csv')
            results_scores_path = os.path.join(results_scores_path, f'{dt_string}_nomad_scores.csv')
        else:
            results_avg_path = os.path.join(results_path, 'nomad_avg.csv')
            results_scores_path = os.path.join(results_path, 'nomad_scores.csv')

        # same bytes as ``df.reset_index().to_csv(path, index=False)`` (tests/test_host.py), written by the library's
        # multi-threaded formatter from the unrounded values: pandas takes minutes on a 1e5 x 1e3 frame
        from . import _lib
        _lib.write_scores_csv(results_avg_path, 'Test File', test_files, ['NOMAD'], np.asarray(avg_nomad, dtype=np.float64))
        if df_dm is not None:
            _lib.write_scores_csv(results_scores_path, 'Test File', test_files, list(df_dm.columns),
                                  np.asarray(distance_matrix, dtype=np.float64))
        return df_avg_nomad, df_dm

    def pairwise(self, test_embeddings, nmr_embeddings):
        """``cdist`` + ``np.mean(axis=1)`` -> (float64 (N, M), float64 (N,)) like scipy/numpy return."""
        te = np.ascontiguousarray(np.asarray(test_embeddings, dtype=np.float32))
        ne = np.ascontiguousarray(np.asarray(nmr_embeddings, dtype=np.float32))
        if te.ndim != 2 or ne.ndim != 2 or te.shape[1] != ne.shape[1]:
            raise ValueError('XA and XB must have the same number of columns (i.e. feature dimension.)')
        if te.shape[1] != EMB_DIM:
            raise ValueError(f'NOMAD embeddings have {EMB_DIM} columns, got {te.shape[1]} (an extra csv column?)')
        dm, mean = self.engine.cdist_mean(torch.from_numpy(te), torch.from_numpy(ne))
        return dm.cpu().numpy().astype(np.float64), mean.cpu().numpy()

    def forward(self, estimate, clean):
        """Differentiable NOMAD loss (``nomad.py:142-146``): 0-dim tensor, grad flows to ``estimate``."""
        self.lossnet_layers.sync_head()
        return _NomadLossFn.apply(estimate, clean, self)

    def get_embeddings(self, path):
        # If mode == dir
        if os.path.isdir(path):
            data = pd.DataFrame(os.listdir(path))
            data.columns = ['filename']
            data['filename'] = [os.path.join(path, x) for x in data['filename']]
        # If mode == csv
        elif os.path.isfile(path):
            data = pd.read_csv(path)
            if 'filename' not in data.columns:
                raise Exception('File {path} not including a column called filename. Please pass a csv file with a column called filename that includes the absolute filpaths of the waveforms.')

        embeddings = self.get_embeddings_csv(self.model, data)
        return embeddings

    def embed_waves(self, waves: Sequence[torch.Tensor]) -> np.ndarray:
        """Embed variable-length mono waveforms in length-bucketed batches; output order == input order.
        Batches are enqueued back to back; the only synchronisation is the single device-to-host copy at the end."""
        if len(waves) == 0:
            return np.zeros((0, EMB_DIM), dtype=np.float32)
        lengths = [int(w.numel()) for w in waves]
        out = torch.empty((len(waves), EMB_DIM), dtype=torch.float32, device=self.engine.device)
        for idx in plan_batches(lengths, self.max_batch_samples):
            emb = self.engine.embed([waves[i] for i in idx])
            out[torch.as_tensor(idx, device=self.engine.device)] = emb
        return out.cpu().numpy()

    def embed_files(self, filepaths: Sequence, root=False) -> torch.Tensor:
        """The reference's per-file loop (``nomad.py:172-186``) restructured for throughput -> (n, 256) CUDA tensor in
        input order.  Files are handled in windows of ``self.window_files`` (bounded memory for 100 k-file corpora).
        Per window the headers of all files are parsed by the library's host threads (``nomad_b200_wav_probe_format``).
        Every wav file the native reader handles -- PCM of 8, 16, 24 or 32 bits or float of 32 or 64 bits, any sample
        rate and channel count -- is then read batch by batch straight into a pinned staging buffer, crosses PCIe as
        the file's own bytes in ONE copy per batch and is decoded, mixed to mono and resampled to 16 kHz on the GPU
        (``nomad_b200_ingest_batch``: one launch per batch plus one per distinct other sample rate).  Other files
        (u-law, A-law, RIFX, non-wav containers) are decoded on the host by ``load_processing`` and packed into the
        same batch.  Batches are planned on 16 kHz lengths.  ``NOMAD_B200_DEVICE_INGEST=0`` decodes every file on the
        host.  Nothing synchronises per batch: the GPU works on batch k while the host reads batch k + 1 (the returned
        tensor may still be being computed)."""
        from concurrent.futures import ThreadPoolExecutor

        from . import _lib
        n_files = len(filepaths)
        parts = []
        with ThreadPoolExecutor(max_workers=self.reader_threads) as pool:
            for w0 in range(0, n_files, self.window_files):
                paths = []
                for filename_anchor in filepaths[w0:w0 + self.window_files]:
                    if isinstance(filename_anchor, np.ndarray):
                        filename_anchor = filename_anchor[0]  # nomad.py:194-195: a DataFrame row
                    paths.append(os.path.join(root, filename_anchor) if root else filename_anchor)
                paths = [str(p) for p in paths]
                if self.device_ingest:
                    probe = _lib.wav_probe_format(paths, self.reader_threads)
                else:
                    probe = _lib.WavProbe.unread(len(paths))
                lengths = _lib.ingest_out_samples(probe.frames, probe.sample_rate)
                host_idx = np.flatnonzero(probe.frames < 0)
                waves = dict(zip(host_idx.tolist(), pool.map(self.load_processing, [paths[i] for i in host_idx])))
                for k, w in waves.items():
                    lengths[k] = w.shape[-1]
                for n in lengths:
                    if n < MIN_SAMPLES:
                        raise RuntimeError(f"Calculated padded input size per channel: ({n}). Kernel size: (10). "
                                           "Kernel size can't be greater than actual input size")
                dev_out = torch.empty((len(paths), EMB_DIM), dtype=torch.float32, device=self.engine.device)
                for idx in plan_batches(lengths, self.max_batch_samples):
                    sel = torch.as_tensor(idx, device=self.engine.device)
                    pos = {i: j for j, i in enumerate(idx)}
                    dev_out[sel] = self.engine.embed_wav_files([paths[i] for i in idx], probe.take(idx), self.reader_threads,
                                                               waves={pos[i]: waves[i] for i in idx if i in waves})
                parts.append(dev_out)  # still being computed; the host goes on with the next window
        if not parts:
            return torch.zeros((0, EMB_DIM), dtype=torch.float32, device=self.engine.device)
        return torch.cat(parts) if len(parts) > 1 else parts[0]

    # Function that extract NOMAD embeddings and store them in a DataFrame (nomad.py:166-189)
    def get_embeddings_csv(self, model, file_names, root=False):
        embeddings = self.embed_files(np.array(file_names), root).cpu().numpy()
        embeddings = pd.DataFrame(embeddings)
        df_emb = pd.concat([file_names.reset_index(), embeddings], axis=1).drop('index', axis=1)
        return df_emb

    # Load wave file (nomad.py:192-212)
    def load_processing(self, filepath, target_sr=16000, trim=False):
        return audio.load_processing(filepath, target_sr, trim)
