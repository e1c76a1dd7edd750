"""Multi-GPU scoring: one process per GPU, utterances sharded across ranks, ONE collective exchange.

The reference has no distributed code (SURVEY.md 2.2); this is the natural sharding of its scoring
path (``nomad.py:102-111``, SURVEY.md 8e).  Utterances are independent, so NMR and degraded files are
partitioned across ranks by audio length (LPT greedy; every rank computes the same partition, so no
sizes are exchanged):

1. each rank embeds its NMR shard;
2. ONE all-gather of the (M, 256) fp32 NMR embeddings (NCCL over NVLink/NVSwitch; <= 8 MB, latency
   bound), issued asynchronously so that it overlaps the start of step 3;
3. each rank embeds its degraded shard and computes its rows of the distance matrix and their means
   against the full NMR set;
4. row means -- and, when wanted, the matrix rows -- are sent to rank 0 only (point-to-point inside the
   group communicator, exact sizes, no padding), where listing order is restored.  The distance matrix
   is never all-gathered; for corpora whose matrix should not live on one rank ``matrix='local'``
   leaves each rank's rows with the rank (row-sharded files).

The functions take ``embed`` / ``cdist_fn`` callables so the host logic is exercised by world_size-2
``gloo`` tests on CPU, and so that ``bench.py`` times exactly the code ``predict_sharded`` runs.
"""
from __future__ import annotations

import os
from typing import Callable, List, Optional, Sequence

import numpy as np
import torch
import torch.distributed as dist


def shard_by_cost(costs: Sequence[float], world: int) -> List[List[int]]:
    """Longest-processing-time greedy partition; deterministic; each shard sorted ascending by index."""
    loads = [0.0] * world
    shards: List[List[int]] = [[] for _ in range(world)]
    for i in sorted(range(len(costs)), key=lambda i: (-float(costs[i]), i)):
        r = min(range(world), key=lambda r: (loads[r], r))
        shards[r].append(i)
        loads[r] += float(costs[i])
    return [sorted(s) for s in shards]


def _world(group=None):
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(group), dist.get_world_size(group)
    return 0, 1


def _listing_index(shards: List[List[int]], stride: int, device) -> torch.Tensor:
    """Row of listing position i inside a buffer that stores shard r at rows [r * stride, r * stride + len)."""
    n = sum(len(s) for s in shards)
    src = np.empty((n,), dtype=np.int64)
    for r, s in enumerate(shards):
        if s:
            src[np.asarray(s, dtype=np.int64)] = r * stride + np.arange(len(s), dtype=np.int64)
    return torch.from_numpy(src).to(device)


class _Pending:
    """An all-gather in flight; ``result()`` waits (stream-ordered on CUDA) and restores listing order."""

    def __init__(self, work, buf, index):
        self.work, self.buf, self.index = work, buf, index

    def result(self) -> torch.Tensor:
        if self.work is not None:
            self.work.wait()
            self.work = None
        return self.buf.index_select(0, self.index)


def all_gather_shards(local: torch.Tensor, shards: List[List[int]], group=None, async_op: bool = False):
    """``local`` = this rank's rows (len(shards[rank]), d) in shard order.  ONE all-gather (shards padded to the
    tallest); returns all rows in listing order on every rank -- or a ``_Pending`` when ``async_op``."""
    rank, world = _world(group)
    d = local.shape[1]
    tall = max(1, max(len(s) for s in shards))
    assert local.shape[0] == len(shards[rank])
    index = _listing_index(shards, tall, local.device)
    if world == 1:
        pend = _Pending(None, local, index)
        return pend if async_op else pend.result()
    pad = torch.zeros((tall, d), dtype=local.dtype, device=local.device)
    pad[: local.shape[0]] = local
    buf = torch.empty((world * tall, d), dtype=local.dtype, device=local.device)
    work = dist.all_gather_into_tensor(buf, pad, group=group, async_op=True)
    pend = _Pending(work, buf, index)
    return pend if async_op else pend.result()


def gather_rows_to_root(local, counts: Sequence[int], group=None):
    """Send every rank's row block (``counts[r]`` rows on rank r) to rank 0 only: exact sizes, ONE batch of
    point-to-point operations in the group's communicator (one NCCL group call, also for several tensors).  ``local``
    is a tensor or a list of tensors with the same row count (e.g. matrix rows + their means).  Rank 0 returns the
    blocks concatenated in RANK order (same device); other ranks return ``None``."""
    rank, world = _world(group)
    many = isinstance(local, (list, tuple))
    locs = [t.contiguous() for t in (local if many else [local])]
    assert all(t.shape[0] == counts[rank] for t in locs)
    if world == 1:
        return locs if many else locs[0]
    root = dist.get_global_rank(group, 0) if group is not None else 0
    if rank != 0:
        if counts[rank]:
            for w in dist.batch_isend_irecv([dist.P2POp(dist.isend, t, root, group=group) for t in locs]):
                w.wait()
        return None
    starts = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
    bufs = [torch.empty((int(starts[-1]),) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device) for t in locs]
    ops = []
    for t, buf in zip(locs, bufs):
        buf[: t.shape[0]] = t
    for r in range(1, world):
        if counts[r]:
            peer = dist.get_global_rank(group, r) if group is not None else r
            ops += [dist.P2POp(dist.irecv, buf[starts[r]: starts[r + 1]], peer, group=group) for buf in bufs]
    if ops:
        for w in dist.batch_isend_irecv(ops):
            w.wait()
    return bufs if many else bufs[0]


def gather_shards_to_root(local, shards: List[List[int]], group=None):
    """``gather_rows_to_root`` + restoring listing order: rank 0 returns the rows of all shards in listing order
    (a tensor, or a list of tensors when ``local`` is a list)."""
    got = gather_rows_to_root(local, [len(s) for s in shards], group)
    if got is None:
        return None
    many = isinstance(got, (list, tuple))
    gots = list(got) if many else [got]
    if gots[0].shape[0]:
        starts = np.concatenate([[0], np.cumsum([len(s) for s in shards])]).astype(np.int64)
        src = np.empty((int(starts[-1]),), dtype=np.int64)
        for r, s in enumerate(shards):
            if s:
                src[np.asarray(s, dtype=np.int64)] = starts[r] + np.arange(len(s), dtype=np.int64)
        idx = torch.from_numpy(src).to(gots[0].device)
        gots = [g.index_select(0, idx) for g in gots]
    return gots if many else gots[0]


def sharded_embeddings(costs: Sequence[float], embed: Callable[[List[int]], torch.Tensor], dim: int,
                       device, group=None, async_op: bool = False):
    """Every rank embeds its shard; returns ALL embeddings (len(costs), dim) in listing order on every rank."""
    rank, world = _world(group)
    shards = shard_by_cost(costs, world)
    mine = shards[rank]
    local = embed(mine) if mine else torch.zeros((0, dim), dtype=torch.float32, device=device)
    local = local.to(device=device, dtype=torch.float32).contiguous()
    return all_gather_shards(local, shards, group, async_op=async_op)


def sharded_scores(deg_costs: Sequence[float], embed: Callable[[List[int]], torch.Tensor], nmr_emb,
                   cdist_fn: Callable, device, group=None, matrix: str = "root", want_emb: bool = False):
    """Each rank: embed its degraded shard, distance rows + means against the full NMR set (``nmr_emb``: tensor or
    the pending all-gather).  ``matrix``: "root" (rows sent to rank 0), "local" (rows stay on the rank that computed
    them) or "none".  Returns a dict: on rank 0 ``mean`` (N,) float64 and ``dm`` (N, M) float32 (matrix="root") in
    listing order; on every rank ``local_rows`` (listing indices of its shard), ``local_mean`` and, for
    matrix="local", ``local_dm``.  Tensors stay on ``device``; nothing is synchronised here."""
    assert matrix in ("root", "local", "none")
    rank, world = _world(group)
    shards = shard_by_cost(deg_costs, world)
    mine = shards[rank]
    emb = (embed(mine).to(device=device, dtype=torch.float32) if mine
           else torch.zeros((0, 256), dtype=torch.float32, device=device))
    if isinstance(nmr_emb, _Pending):
        nmr_emb = nmr_emb.result()
    M = nmr_emb.shape[0]
    if mine:
        dm, mean = cdist_fn(emb, nmr_emb, matrix != "none")
    else:
        dm = torch.zeros((0, M), dtype=torch.float32, device=device) if matrix != "none" else None
        mean = torch.zeros((0,), dtype=torch.float64, device=device)
    out = {"local_rows": mine, "local_mean": mean, "local_dm": dm if matrix == "local" else None, "nmr": nmr_emb}
    send = [mean.reshape(-1, 1).to(torch.float64)]   # everything that goes to rank 0 travels in one NCCL group call
    if matrix == "root":
        send.append(dm.to(torch.float32))
    if want_emb:
        send.append(emb)
    got = gather_shards_to_root(send, shards, group)
    out["mean"], out["dm"], out["emb"] = None, None, None
    if got is not None:
        out["mean"] = got[0].reshape(-1)
        if matrix == "root":
            out["dm"] = got[1]
        if want_emb:
            out["emb"] = got[-1]
    return out


def score_sharded(nmr_costs: Sequence[float], embed_nmr: Callable, deg_costs: Sequence[float], embed_deg: Callable,
                  cdist_fn: Callable, device, group=None, matrix: str = "root", want_emb: bool = False):
    """Steps 1-4 of the module docstring.  The NMR all-gather is in flight while the degraded shard is embedded."""
    pending = sharded_embeddings(nmr_costs, embed_nmr, 256, device, group, async_op=True)
    return sharded_scores(deg_costs, embed_deg, pending, cdist_fn, device, group, matrix, want_emb)


def init_from_env(backend: Optional[str] = None):
    """torchrun-style init (RANK / LOCAL_RANK / WORLD_SIZE / MASTER_*).  Returns (rank, world, local_rank)."""
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1 and not dist.is_initialized():
        if backend is None:
            backend = "nccl" if torch.cuda.is_available() else "gloo"
        if backend == "nccl":
            torch.cuda.set_device(local)
            dist.init_process_group(backend, device_id=torch.device("cuda", local))
        else:
            dist.init_process_group(backend)
    return rank, world, local


def shard_costs(files, threads: int = 0) -> List[float]:
    """Work estimate per file for ``shard_by_cost``: the 16 kHz output length for a wav file the native reader handles
    (the embedding's cost does not depend on the file's encoding), the size in bytes for any other file."""
    from . import _lib
    probe = _lib.wav_probe_format(files, threads)
    n_out = _lib.ingest_out_samples(probe.frames, probe.sample_rate)
    return [float(n) if n >= 0 else float(os.path.getsize(f)) for f, n in zip(files, n_out)]


# above this many matrix bytes the rows stay with the ranks and are written as row-sharded files
ROOT_MATRIX_LIMIT_BYTES = 8 << 30


def predict_sharded(nomad, mode: str, nmr: str, deg: str, results_path: Optional[str] = None, group=None,
                    matrix: Optional[str] = None):
    """``Nomad.predict`` across the ranks of the current process group.  Rank 0 returns ``(df_avg_nomad, df_dm)`` and
    writes the CSVs; other ranks return ``None``.  With ``matrix='local'`` (default above ROOT_MATRIX_LIMIT_BYTES)
    every rank writes its own rows to ``nomad_scores.rank<r>.csv`` under ``results_path`` and rank 0 returns
    ``(df_avg_nomad, None)``."""
    import pandas as pd

    rank, world = _world(group)
    device = nomad.engine.device

    def listing(path):
        obj = [None]
        if rank == 0:
            if mode == "dir":
                obj[0] = [os.path.join(path, x) for x in os.listdir(path)]
            else:
                obj[0] = list(pd.read_csv(path)["filename"])
        if world > 1:
            dist.broadcast_object_list(obj, src=0, group=group)
        return obj[0]

    nmr_files, deg_files = listing(nmr), listing(deg)
    if matrix is None:
        matrix = "root" if 4 * len(nmr_files) * len(deg_files) <= ROOT_MATRIX_LIMIT_BYTES else "local"
    if matrix == "local" and results_path is None:
        raise Exception("row-sharded scores need results_path (every rank writes its rows there)")

    # windowed, length-bucketed, device-ingest loader of Nomad.get_embeddings_csv, on this rank's files only
    embed_files = lambda files: (lambda idx: nomad.embed_files([files[i] for i in idx]))
    cost = lambda files: shard_costs(files, nomad.reader_threads)
    res = score_sharded(cost(nmr_files), embed_files(nmr_files), cost(deg_files), embed_files(deg_files),
                        lambda a, b, wm: nomad.engine.cdist_mean(a, b, wm), device, group, matrix)
    if matrix == "local":
        rows = res["local_rows"]
        from . import _lib
        stems = [x.split('/')[-1].split('.')[0] for x in deg_files]
        _lib.write_scores_csv(os.path.join(results_path, f"nomad_scores.rank{rank}.csv"), 'Test File',
                              [stems[i] for i in rows], [x.split('/')[-1].split('.')[0] for x in nmr_files],
                              res["local_dm"].cpu().numpy().astype(np.float64).reshape(len(rows), len(nmr_files)))
    if rank != 0:
        return None
    mean = res["mean"].cpu().numpy()
    if matrix == "local":
        return nomad.write_results(deg_files, nmr_files, None, mean, results_path)
    return nomad.write_results(deg_files, nmr_files, res["dm"].cpu().numpy().astype(np.float64), mean, results_path)
