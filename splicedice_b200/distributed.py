"""One process per GPU: row-slab sharding of the quant / pairwise work over torch.distributed.

The path has no exchange step (adjacency never leaves an overlap component, see sharding.py):
every rank computes its slab independently and results return by host gather.  The only
collective is the optional all-gather of PS row blocks (NCCL over NVLink when the slabs are CUDA
tensors and the backend is nccl; gloo on CPU tensors in the tests), for a consumer that wants the
whole matrix on every GPU.
"""
from __future__ import annotations

import numpy as np
import torch
import torch.distributed as dist

from . import sharding


def bind_to_gpu_numa(device: int = 0):
    """Pin the calling thread (and the threads it starts later) to the CPUs NVML reports as local
    to ``device``, so pinned host buffers allocated afterwards land on the GPU's own NUMA node and
    its PCIe traffic does not cross the socket interconnect.  One process per GPU calls this once,
    before it allocates host buffers.  Performance only: returns the CPU set used, or None when
    NVML / the affinity call is unavailable or the local CPUs are outside this process's cpuset."""
    import os
    if os.environ.get("SD_NO_NUMA_BIND"):
        return None
    try:
        import pynvml
        pynvml.nvmlInit()
        visible = os.environ.get("CUDA_VISIBLE_DEVICES")
        index = device
        if visible:
            ids = [v.strip() for v in visible.split(",") if v.strip()]
            if device < len(ids) and ids[device].isdigit():
                index = int(ids[device])
        handle = pynvml.nvmlDeviceGetHandleByIndex(index)
        n_cpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(handle, (n_cpu + 63) // 64)
        local = {64 * w + b for w, word in enumerate(words) for b in range(64) if (word >> b) & 1}
        allowed = os.sched_getaffinity(0)
        cpus = local & allowed
        if not cpus or cpus == allowed:
            return None if not cpus else sorted(cpus)
        os.sched_setaffinity(0, cpus)
        return sorted(cpus)
    except Exception:                          # noqa: BLE001 - placement hint only
        return None


def _world():
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


def all_gather_rows(local, parts):
    """Row slabs -> the whole [J, ...] tensor on every rank.  ``local`` holds this rank's rows
    ``parts[rank]``; slab heights differ (cuts sit on cluster boundaries).  NCCL: one
    ``dist.all_gather`` whose outputs are the slab views of the result itself -- torch issues it as
    one grouped NCCL call that lands every slab in place, no padding and no second copy.  Other
    backends (gloo in the CPU tests) need equal blocks: slabs are padded to a common height."""
    rank, world = _world()
    if world == 1:
        return local
    J = parts[-1][1]
    if dist.get_backend() == "nccl" and local.is_cuda:
        full = torch.empty((J,) + tuple(local.shape[1:]), dtype=local.dtype, device=local.device)
        dist.all_gather([full[a:b] for a, b in parts], local.contiguous())
        return full
    r0, r1 = parts[rank]
    height = max(b - a for a, b in parts)
    padded = torch.zeros((height,) + tuple(local.shape[1:]), dtype=local.dtype, device=local.device)
    padded[: r1 - r0] = local
    blocks = [torch.empty_like(padded) for _ in range(world)]
    dist.all_gather(blocks, padded)
    return torch.cat([blocks[k][: parts[k][1] - parts[k][0]] for k in range(world)])


def sharded_rows(counts, row_ptr, col_idx, slab_fn, gather=True, weights=None):
    """Run ``slab_fn(counts[r0:r1], local_row_ptr, local_col_idx) -> tensor[r1 - r0, S]`` on this
    rank's slab.  With ``gather`` every rank receives the full [J, S] tensor (all_gather_rows);
    otherwise returns (local tensor, (r0, r1))."""
    rank, world = _world()
    n_samples = counts.shape[1]
    if weights is None:
        weights = sharding.row_weights(row_ptr, n_samples)
    parts = sharding.partition_rows(row_ptr, col_idx, world, weights)
    r0, r1 = parts[rank]
    rp, ci = sharding.shard_csr(row_ptr, col_idx, r0, r1)
    local = slab_fn(counts[r0:r1], rp, ci)
    if not gather:
        return local, (r0, r1)
    return all_gather_rows(local, parts)


def quant_ps_sharded(counts_host, row_ptr, col_idx, device=None, gather=True, low_mask=None):
    """PS of a host int32 count matrix with the rows split over the ranks' GPUs.  Rank r uploads
    only its slab (and its slab of the low-coverage mask: the NaN overwrite of SPLICEDICE.py:307-309
    is per cell, so it shards with the rows).  Returns the full float32 matrix on every rank's GPU
    (``gather``) or the local slab and its row range."""
    from . import ops
    rank, _ = _world()
    dev = torch.device("cuda", torch.cuda.current_device() if device is None else device)
    n_cols = counts_host.shape[1]
    parts = sharding.partition_rows(row_ptr, col_idx, _world()[1], sharding.row_weights(row_ptr, n_cols))

    def slab(counts_slab, rp, ci):
        c = ops.upload_counts(counts_slab, dev)
        mask = None
        if low_mask is not None:
            r0, r1 = parts[rank]
            mask = torch.from_numpy(np.ascontiguousarray(low_mask[r0:r1], dtype=np.uint8)).to(dev)
        return ops.quant_ps(c, rp, ci, low_mask=mask, want_f32=True)["ps_f32"]

    return sharded_rows(counts_host, row_ptr, col_idx, slab, gather=gather)


# ---- pairwise: row-sharded Fisher, column-sharded Benjamini-Hochberg ---------------------------
# The Fisher rows are independent, so every rank computes p[rows_r, P] for its row slab.  The
# per-pair correction (pairwise_fisher.py:186-191) ranks each COLUMN over all junctions, which is
# the path's one real exchange step: an all-to-all turns the row slabs into column blocks
# [J, P_r] (NCCL over NVLink on CUDA tensors), each rank adjusts its columns with sd_bh_adjust,
# and a second all-to-all brings the adjusted values back to the row owners.

def _all_to_all(recv, send):
    """recv[g] <- rank g's send[this rank].  One NCCL all-to-all on CUDA tensors; backends without
    that collective (gloo, in the CPU tests) exchange the same blocks with paired isend / irecv."""
    rank, world = _world()
    if dist.get_backend() == "nccl":
        dist.all_to_all(recv, send)
        return
    recv[rank].copy_(send[rank])
    ops_ = []
    for g in range(world):
        if g != rank:
            ops_.append(dist.P2POp(dist.isend, send[g], g))
            ops_.append(dist.P2POp(dist.irecv, recv[g], g))
    for req in dist.batch_isend_irecv(ops_):
        req.wait()


def column_blocks(n_cols, world):
    """Contiguous, near-equal column ranges, one per rank."""
    base, extra = divmod(n_cols, world)
    cuts = [0]
    for g in range(world):
        cuts.append(cuts[-1] + base + (1 if g < extra else 0))
    return [(cuts[g], cuts[g + 1]) for g in range(world)]


def rows_to_columns(p_local, parts):
    """[rows_r, P] on every rank -> [J, P_r] on every rank (rows in global order)."""
    rank, world = _world()
    blocks = column_blocks(p_local.shape[1], world)
    if world == 1:
        return p_local
    send = [p_local[:, a:b].contiguous() for a, b in blocks]
    c0, c1 = blocks[rank]
    recv = [torch.empty((r1 - r0, c1 - c0), dtype=p_local.dtype, device=p_local.device) for r0, r1 in parts]
    _all_to_all(recv, send)
    return torch.cat(recv, dim=0)


def columns_to_rows(q_cols, parts, n_cols):
    """Inverse of rows_to_columns: [J, P_r] -> [rows_r, P]."""
    rank, world = _world()
    if world == 1:
        return q_cols
    blocks = column_blocks(n_cols, world)
    r0, r1 = parts[rank]
    send = [q_cols[a:b].contiguous() for a, b in parts]
    recv = [torch.empty((r1 - r0, b - a), dtype=q_cols.dtype, device=q_cols.device) for a, b in blocks]
    _all_to_all(recv, send)
    return torch.cat(recv, dim=1)


def bh_columns_sharded(p_local, parts, adjust_fn):
    """Per-column Benjamini-Hochberg of a row-sharded p-value matrix.  ``adjust_fn([J, P_r]) ->
    [J, P_r]`` adjusts whole columns (ops.bh_adjust(..., 'pairwise') in the product; the numpy
    restatement in the gloo test)."""
    n_cols = p_local.shape[1]
    cols = rows_to_columns(p_local, parts)
    return columns_to_rows(adjust_fn(cols), parts, n_cols)


# ---- the same exchange fused into the kernels: peer memory over NVLink -------------------------
# Instead of "Fisher -> all-to-all -> BH -> all-to-all", every rank's Fisher kernel stores each
# p-value straight into the column-block owner's matrix (sd_fisher_pairwise_scatter writes through
# CUDA IPC mappings of the peers' buffers), one barrier orders the GPUs, every rank adjusts its
# column block in place, and the adjusted blocks go back to the row owners through one kernel of
# peer stores (sd_peer_scatter_rows).
# No packing, no staging buffers, no NCCL on the data path (NCCL carries the barriers and the
# one-off exchange of the IPC handles).
_PEER_CACHE = {}
# Measured on B200s, 200,000 x 2,016 cut over N GPUs, whole step (Fisher + exchange + correction), fused
# vs NCCL all-to-alls: N = 2: 24.4 vs 27.9 ms; N = 8: 7.87 vs 7.71 ms (the slabs' Fisher kernels last
# only 2.5 ms there, and the two host-side barriers cost what the small all-to-alls cost).  The fused
# form is the default up to four GPUs.
FUSED_MAX_WORLD = 4


class _RawCuda:
    """A raw device allocation as something torch.as_tensor can alias (__cuda_array_interface__)."""

    def __init__(self, ptr, shape):
        self.__cuda_array_interface__ = {"shape": tuple(int(x) for x in shape), "typestr": "<f8", "data": (int(ptr), False),
                                         "version": 2, "strides": None}


class PeerMatrix:
    """One float64 matrix per rank, every rank able to address all of them: this rank's own
    allocation (sd_peer_alloc; ``own`` is a torch tensor aliasing it) and CUDA IPC mappings of the
    others' (sd_peer_open).  ``ptrs[g]`` / ``lds[g]`` / ``shapes[g]``: rank g's base pointer, leading
    dimension in elements and shape.  Shapes may differ by rank."""

    def __init__(self, shape, dev):
        import ctypes
        from . import native
        rank, world = _world()
        self.dev = dev
        self.shape = tuple(int(x) for x in shape)
        nbytes = max(1, self.shape[0] * self.shape[1] * 8)
        ptr = ctypes.c_void_p()
        handle = (ctypes.c_ubyte * 64)()
        with torch.cuda.device(dev):
            native.call("sd_peer_alloc", nbytes, ctypes.byref(ptr), handle)
        self._own_ptr = ptr.value
        self.own = torch.as_tensor(_RawCuda(ptr.value, self.shape), device=dev) if self.shape[0] * self.shape[1] else \
            torch.empty(self.shape, dtype=torch.float64, device=dev)
        gathered = [None] * world
        dist.all_gather_object(gathered, (bytes(handle), self.shape))
        self.ptrs, self.lds, self.shapes, self._opened = [], [], [], []
        for g, (h, shp) in enumerate(gathered):
            self.shapes.append(shp)
            self.lds.append(shp[1])
            if g == rank:
                self.ptrs.append(self._own_ptr)
                continue
            peer = ctypes.c_void_p()
            buf = (ctypes.c_ubyte * 64).from_buffer_copy(h)
            with torch.cuda.device(dev):
                native.call("sd_peer_open", buf, ctypes.byref(peer))
            self.ptrs.append(peer.value)
            self._opened.append(peer.value)

    def close(self):
        from . import native
        torch.cuda.synchronize(self.dev)
        if dist.is_initialized():
            dist.barrier()                          # nobody is still reading this rank's buffer
        with torch.cuda.device(self.dev):
            for p in self._opened:
                native.call("sd_peer_close", p)
            self._opened = []
            if self._own_ptr:
                self.own = None
                native.call("sd_peer_free", self._own_ptr)
                self._own_ptr = None


def _peer_matrix(tag, shape, dev):
    hit = _PEER_CACHE.get(tag)
    if hit is not None and hit.shape == tuple(shape) and hit.dev == dev:
        return hit
    if hit is not None:
        hit.close()
    _PEER_CACHE[tag] = PeerMatrix(shape, dev)
    return _PEER_CACHE[tag]


def release_peer_buffers():
    """Unmap and free every cached peer buffer (collective: every rank calls it)."""
    for tag in list(_PEER_CACHE):
        _PEER_CACHE.pop(tag).close()


def pairwise_fused(inc, exc, pair_a, pair_b, parts, bound, adjust=True):
    """Fisher + per-pair Benjamini-Hochberg of a row-sharded problem with the exchange fused into the
    kernels' stores.  inc / exc: this rank's slab (CUDA); parts: every rank's (row_begin, row_end).
    Returns float64 CUDA [rows_r, P] (a cached peer buffer: copy it if it must outlive the next call)."""
    import ctypes
    from . import native, ops
    rank, world = _world()
    dev = inc.device
    P = int(len(pair_a))
    J = parts[-1][1]
    r0, r1 = parts[rank]
    blocks = column_blocks(P, world)
    c0, c1 = blocks[rank]
    cols = _peer_matrix(("cols", J, P, world), (J, c1 - c0), dev)
    rows = _peer_matrix(("rows", J, P, world), (r1 - r0, P), dev)
    pa, pb = ops._i32(pair_a, dev), ops._i32(pair_b, dev)
    n = world
    ptrs = (ctypes.c_void_p * n)(*cols.ptrs)
    cuts = (ctypes.c_int64 * (n + 1))(*([b[0] for b in blocks] + [P]))
    lds = (ctypes.c_int64 * n)(*cols.lds)
    with torch.cuda.device(dev):
        native.call("sd_fisher_pairwise_scatter", inc.shape[0], inc.shape[1], native.ptr(inc), inc.stride(0),
                    native.ptr(exc), exc.stride(0), P, native.ptr(pa), native.ptr(pb), n, ptrs, cuts, lds, r0, 0,
                    inc.shape[0], int(bound), native.stream_ptr())
        dist.barrier()                               # every GPU's stores into this rank's column block are done
        if adjust and c1 > c0:
            ops.bh_adjust(cols.own, "pairwise", out=cols.own)
        if c1 > c0:                                  # adjusted block -> the row owners, one kernel of peer stores
            rptrs = (ctypes.c_void_p * n)(*rows.ptrs)
            rcuts = (ctypes.c_int64 * (n + 1))(*([a for a, _ in parts] + [J]))
            rlds = (ctypes.c_int64 * n)(*rows.lds)
            native.call("sd_peer_scatter_rows", native.ptr(cols.own), J, c1 - c0, n, rptrs, rcuts, rlds, c0, native.stream_ptr())
        dist.barrier()                               # every rank's rows are complete
    return rows.own


def pairwise_sharded(counts_host, row_ptr, col_idx, correction="pairwise", device=None, test="fisher", refused=None):
    """``splicedice pairwise`` arithmetic over the ranks' GPUs: exclusion sums + Fisher (or the
    chi-squared test, ``test='chi2'``) on this rank's row slab, then the correction.  counts_host:
    integer [J, S] on every rank (each uploads only its slab).  Returns (float64 CUDA tensor
    [rows_r, P], (r0, r1)).  chi2: ``refused`` as in ops.chi2_pairwise, the index local to the slab."""
    from . import ops
    from .pairwise_fisher import checked_counts, fisher_inputs
    rank, world = _world()
    if correction not in ("none", "pairwise", "all"):
        raise ValueError("correction must be 'none', 'pairwise' or 'all'")
    if test not in ("fisher", "chi2"):
        raise ValueError("test must be 'fisher' or 'chi2'")
    dev = torch.device("cuda", torch.cuda.current_device() if device is None else device)
    parts = sharding.partition_rows(row_ptr, col_idx, world)
    r0, r1 = parts[rank]
    rp, ci = sharding.shard_csr(row_ptr, col_idx, r0, r1)
    inc, exc, pa, pb, bound = fisher_inputs(checked_counts(counts_host[r0:r1]), rp, ci, dev)
    if test == "chi2":                               # the NCCL exchange below: no fused scatter form
        p = ops.chi2_pairwise(inc, exc, pa, pb, refused=refused)
    elif correction == "pairwise" and 1 < world <= FUSED_MAX_WORLD and dist.get_backend() == "nccl" and len(pa) >= world:
        # the exchange rides on the kernels' own stores (peer memory); see pairwise_fused
        return pairwise_fused(inc, exc, pa, pb, parts, bound).clone(), (r0, r1)
    else:
        p = ops.fisher_pairwise(inc, exc, pa, pb, max_cell_bound=bound)
    if correction == "pairwise":
        p = bh_columns_sharded(p, parts, lambda cols: ops.bh_adjust(cols, "pairwise", out=cols))
    elif correction == "all":
        # one ranking over every p-value of the matrix (pairwise_fisher.py:189-191): the row slabs are
        # gathered on every GPU (NCCL), each adjusts the whole matrix and keeps its own rows -- the
        # matrix has to fit one GPU for this mode anyway (sd_bh_adjust: < 2^31 values per segment)
        full = all_gather_rows(p, parts) if world > 1 else p
        ops.bh_adjust(full, "all", out=full)
        p = full[r0:r1].clone() if world > 1 else full
    return p, (r0, r1)
