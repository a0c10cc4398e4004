"""``--gpus N`` for the command-line tools: one worker process per GPU.

The CLI's host work (file parsing, TSV writers) stays in the calling process; the compute stages
fan out over N worker processes, one per GPU (``torch.multiprocessing`` spawn, ranks 0..N-1 on
devices 0..N-1).  Inputs and outputs travel through shared host memory: every worker reads its row
slab of the shared count matrix and writes its rows of the shared result, so the "host gather" of
SURVEY.md section 8e is the result array itself.  Row slabs are cut where no adjacency edge crosses
(sharding.partition_rows), so quant needs no collective at all; pairwise joins a NCCL group for the
one exchange its default correction needs (per-pair Benjamini-Hochberg ranks whole columns:
distributed.bh_columns_sharded) and for the gather of ``--multiple_test_correction all``.

Replaces nothing in the reference (it is single-process, single-threaded): this is how the B200
path spreads SPLICEDICE.calculatePsi (SPLICEDICE.py:297-310) and the pairwise loop
(pairwise_fisher.py:154-191) over the GPUs of one box.
"""
from __future__ import annotations

import os
import socket

import numpy as np


def device_count() -> int:
    import torch
    return torch.cuda.device_count() if torch.cuda.is_available() else 0


def check_gpus(n_gpus: int) -> int:
    n_gpus = int(n_gpus)
    if n_gpus < 1:
        raise ValueError("--gpus must be at least 1")
    have = device_count()
    if n_gpus > have:
        raise RuntimeError(f"--gpus {n_gpus} requested but only {have} CUDA device(s) are visible")
    return n_gpus


def _free_port() -> int:
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _shared(array, dtype):
    import torch
    t = torch.from_numpy(np.ascontiguousarray(array, dtype=dtype))
    return t.share_memory_()


def _spawn(fn, n_gpus, args):
    import torch.multiprocessing as mp
    # the host-buffer pipelines check this to know that several ranks share the host (sd_hostpipe.cu)
    os.environ["LOCAL_WORLD_SIZE"] = str(n_gpus)
    try:
        mp.spawn(fn, args=(n_gpus, *args), nprocs=n_gpus, join=True)
    finally:
        os.environ.pop("LOCAL_WORLD_SIZE", None)


# ---- quant ------------------------------------------------------------------------------------
def _quant_worker(rank, world, counts, row_ptr, col_idx, mask, out, parts):
    import torch
    from . import ops, sharding
    torch.cuda.set_device(rank)
    r0, r1 = parts[rank]
    if r1 == r0:
        return
    rp, ci = sharding.shard_csr(row_ptr.numpy(), col_idx.numpy(), r0, r1)
    ops.quant_ps_host(counts[r0:r1], rp, ci, low_mask=None if mask is None else mask[r0:r1].numpy(),
                      out=out[r0:r1], device=rank)


def quant_ps(counts, row_ptr, col_idx, low_mask=None, n_gpus=2):
    """float32 PS of a host int32 count matrix on ``n_gpus`` GPUs: contiguous row slabs at cluster
    boundaries, balanced by (1 + degree) x samples, each through sd_quant_ps_host on its own GPU."""
    import torch
    from . import sharding
    n_gpus = check_gpus(n_gpus)
    J, S = counts.shape
    parts = sharding.partition_rows(row_ptr, col_idx, n_gpus, sharding.row_weights(row_ptr, S))
    out = torch.empty((J, S), dtype=torch.float32).share_memory_()
    _spawn(_quant_worker, n_gpus, (_shared(counts, np.int32), _shared(row_ptr, np.int32), _shared(col_idx, np.int32),
                                   None if low_mask is None else _shared(low_mask, np.uint8), out, parts))
    return out.numpy()


# ---- pairwise -----------------------------------------------------------------------------------
def _pairwise_worker(rank, world, port, counts, row_ptr, col_idx, correction, test, out, refused):
    import torch
    import torch.distributed as dist
    from . import distributed
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world,
                            device_id=torch.device("cuda", rank))
    try:
        # a rank that meets a refused chi-squared table still finishes every collective (the others would
        # wait for it) and reports the table through shared memory
        ref = torch.full((1,), -1, dtype=torch.int64, device=torch.device("cuda", rank)) if test == "chi2" else None
        p, (r0, r1) = distributed.pairwise_sharded(counts.numpy(), row_ptr.numpy(), col_idx.numpy(), correction,
                                                   device=rank, test=test, refused=ref)
        out[r0:r1] = p.cpu()
        if ref is not None and int(ref.item()) != -1:
            refused[rank] = int(ref.item()) + r0 * out.shape[1]
    finally:
        dist.destroy_process_group()


def pairwise(counts_int, row_ptr, col_idx, n_pairs, correction="pairwise", n_gpus=2, test="fisher"):
    """(float64[J, n_pairs] (corrected) p-values, first refused index) on ``n_gpus`` GPUs
    (distributed.pairwise_sharded).  The index is row * n_pairs + pair of the first table the
    chi-squared test refuses (as sd_chi2_pairwise reports it on one GPU), None when there is none."""
    import torch
    n_gpus = check_gpus(n_gpus)
    J = counts_int.shape[0]
    out = torch.empty((J, n_pairs), dtype=torch.float64).share_memory_()
    refused = torch.full((n_gpus,), -1, dtype=torch.int64).share_memory_()
    _spawn(_pairwise_worker, n_gpus, (_free_port(), _shared(counts_int, np.int64), _shared(row_ptr, np.int32),
                                      _shared(col_idx, np.int32), correction, test, out, refused))
    found = [int(v) for v in refused.tolist() if v != -1]
    return out.numpy(), (min(found) if found else None)
