"""Device-level operators over the C-ABI (torch tensors in, torch tensors out).

torch owns device memory and streams; every computation is a call into
``libsplicedice_b200.so``.  Nothing here computes on the CPU and nothing falls back: without a
CUDA device ``require_cuda`` raises.
"""
from __future__ import annotations

import ctypes

import numpy as np
import torch

from . import native


def require_cuda():
    native.load()
    if not torch.cuda.is_available():
        raise native.NativeLibraryError("splicedice_b200 needs a CUDA device (sm_100a); there is no CPU path")


def _dev(device=None):
    require_cuda()
    if isinstance(device, torch.device):
        return device if device.index is not None else torch.device("cuda", torch.cuda.current_device())
    return torch.device("cuda", torch.cuda.current_device() if device is None else int(device))


def _i32(x, device):
    if isinstance(x, torch.Tensor):
        return x.to(device=device, dtype=torch.int32).contiguous()
    return torch.from_numpy(np.ascontiguousarray(x, dtype=np.int32)).to(device)


def _sp(stream=None):
    return native.stream_ptr(stream)


def device_info(device: int = 0):
    sm, maj, mnr, mem = ctypes.c_int(), ctypes.c_int(), ctypes.c_int(), ctypes.c_size_t()
    native.call("sd_device_info", device, ctypes.byref(sm), ctypes.byref(maj), ctypes.byref(mnr), ctypes.byref(mem))
    return dict(sm_count=sm.value, cc=(maj.value, mnr.value), total_mem=mem.value)


# ---------------------------------------------------------------------------------------
# K1
# ---------------------------------------------------------------------------------------
def cluster_build(chrom_rank, strand_rank, start, end, device=None, with_adjacency=True):
    """Overlap adjacency CSR + output row order on the device (sd_cluster_build / _fill).

    Returns a dict of int32 device tensors (cluster_order, out_row, row_of_pos, comp_id,
    row_ptr, col_idx) and python ints nnz, n_comp.
    """
    dev = _dev(device)
    with torch.cuda.device(dev):
        c, s, st, en = (_i32(x, dev) for x in (chrom_rank, strand_rank, start, end))
        J = int(c.numel())
        if not (s.numel() == J and st.numel() == J and en.numel() == J):
            raise ValueError("cluster_build: arrays differ in length")
        i32 = dict(dtype=torch.int32, device=dev)
        out = dict(cluster_order=torch.empty(J, **i32), out_row=torch.empty(J, **i32),
                   row_of_pos=torch.empty(J, **i32), comp_id=torch.empty(J, **i32),
                   row_ptr=torch.zeros(J + 1, **i32))
        if J == 0:
            out.update(col_idx=torch.empty(0, **i32), nnz=0, n_comp=0)
            return out
        lib = native.load()
        ws_bytes = lib.sd_cluster_workspace_bytes(J)
        if ws_bytes == 0:
            raise native.NativeCallError("sd_cluster_workspace_bytes", -1, native.last_error())
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        nnz, ncomp = ctypes.c_int64(), ctypes.c_int64()
        native.call("sd_cluster_build", J, native.ptr(c), native.ptr(s), native.ptr(st), native.ptr(en),
                    native.ptr(out["cluster_order"]), native.ptr(out["out_row"]), native.ptr(out["row_of_pos"]),
                    native.ptr(out["comp_id"]), native.ptr(out["row_ptr"]), ctypes.byref(nnz), ctypes.byref(ncomp),
                    native.ptr(ws), ws_bytes, _sp())
        out["nnz"], out["n_comp"] = nnz.value, ncomp.value
        col = torch.empty(nnz.value, **i32)
        if with_adjacency and nnz.value:
            fw_bytes = lib.sd_cluster_fill_workspace_bytes(J, nnz.value)
            fw = torch.empty(fw_bytes, dtype=torch.uint8, device=dev)
            native.call("sd_cluster_fill", J, nnz.value, native.ptr(out["row_of_pos"]), native.ptr(out["row_ptr"]),
                        native.ptr(col), native.ptr(ws), ws_bytes, native.ptr(fw), fw_bytes, _sp())
        out["col_idx"] = col
        return out


# ---------------------------------------------------------------------------------------
# K2
# ---------------------------------------------------------------------------------------
def upload_counts(host_matrix, device):
    """int32 CUDA view [J, S] of a host integer matrix (values already checked to fit int32), in a
    zero-padded [J, ceil4(S)] buffer: the tiled count kernels need 16-byte aligned rows."""
    J, S = host_matrix.shape
    buf = torch.zeros((J, (S + 3) // 4 * 4), dtype=torch.int32, device=device)
    buf[:, :S] = torch.from_numpy(np.ascontiguousarray(host_matrix, dtype=np.int32)).to(device)
    return buf[:, :S]


def quant_ps(counts, row_ptr, col_idx, low_mask=None, want_f32=True, want_f64=False, want_exc=False,
             row_begin=0, row_end=None, flags=native.SD_QUANT_AUTO, out_f32=None, out_f64=None, out_exc=None):
    """PS (float32 as SPLICEDICE.calculatePsi, float64 as counts_to_ps) and/or exclusion sums
    for rows [row_begin, row_end) of a device int32 count matrix (sd_quant_ps)."""
    require_cuda()
    if counts.dtype != torch.int32 or not counts.is_cuda or counts.dim() != 2:
        raise TypeError("quant_ps: counts must be a 2-D int32 CUDA tensor")
    if counts.stride(1) != 1:
        raise ValueError("quant_ps: counts must be row-major")
    J, S = counts.shape
    dev = counts.device
    row_end = J if row_end is None else row_end
    row_ptr = _i32(row_ptr, dev)
    col_idx = _i32(col_idx, dev)

    def alloc(want, given, dtype):
        if given is not None:
            return given
        return torch.empty((J, S), dtype=dtype, device=dev) if want else None

    ps32 = alloc(want_f32, out_f32, torch.float32)
    ps64 = alloc(want_f64, out_f64, torch.float64)
    exc = alloc(want_exc, out_exc, torch.int64)
    if low_mask is not None:
        low_mask = low_mask.to(device=dev, dtype=torch.uint8).contiguous()
    ld = lambda t: 0 if t is None else t.stride(0)  # noqa: E731
    with torch.cuda.device(dev):
        native.call("sd_quant_ps", J, S, native.ptr(counts), counts.stride(0), native.ptr(row_ptr),
                    native.ptr(col_idx), native.ptr(low_mask), ld(low_mask), native.ptr(ps32), ld(ps32),
                    native.ptr(ps64), ld(ps64), native.ptr(exc), ld(exc), row_begin, row_end, flags, _sp())
    return dict(ps_f32=ps32, ps_f64=ps64, exc=exc)


def quant_ps_host(counts, row_ptr, col_idx, low_mask=None, out=None, device=0):
    """Host-buffer PS: numpy / pinned torch CPU arrays in and out (sd_quant_ps_host)."""
    require_cuda()
    c = counts if isinstance(counts, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(counts, dtype=np.int32))
    if c.dtype != torch.int32 or c.is_cuda or c.dim() != 2 or c.stride(1) != 1:
        raise TypeError("quant_ps_host: counts must be a row-major 2-D int32 host array")
    J, S = c.shape
    rp = np.ascontiguousarray(row_ptr.cpu().numpy() if isinstance(row_ptr, torch.Tensor) else row_ptr, dtype=np.int32)
    ci = np.ascontiguousarray(col_idx.cpu().numpy() if isinstance(col_idx, torch.Tensor) else col_idx, dtype=np.int32)
    if out is None:
        out = torch.empty((J, S), dtype=torch.float32)
    m = None
    if low_mask is not None:
        m = np.ascontiguousarray(low_mask, dtype=np.uint8)
    native.call("sd_quant_ps_host", device, J, S, native.ptr(c), c.stride(0), native.ptr(rp), native.ptr(ci),
                native.ptr(m), 0 if m is None else m.strides[0], native.ptr(out), out.stride(0))
    return out


# ---------------------------------------------------------------------------------------
# K3
# ---------------------------------------------------------------------------------------
def all_pairs(n_samples: int):
    """Pair order of pairwise_fisher.py:142-145."""
    a, b = np.triu_indices(n_samples, k=1)
    return a.astype(np.int32), b.astype(np.int32)


def fisher_pairwise(inc, exc, pair_a, pair_b, row_begin=0, row_end=None, out=None, max_cell_bound=None):
    """p[j, k] for tables [[inc[j,a_k], inc[j,b_k]], [exc[j,a_k], exc[j,b_k]]] (sd_fisher_pairwise).
    With ``max_cell_bound`` (an upper bound on inc + exc the caller vouches for) the call is fully
    asynchronous (sd_fisher_pairwise_bounded); cells outside the bound give NaN."""
    require_cuda()
    if inc.dtype != torch.int32 or exc.dtype != torch.int64 or not inc.is_cuda or not exc.is_cuda:
        raise TypeError("fisher_pairwise: inc int32 / exc int64 CUDA tensors expected")
    J, S = inc.shape
    dev = inc.device
    # pairs given on the host are validated there; device tensors are trusted (no sync)
    for arr in (pair_a, pair_b):
        if not isinstance(arr, torch.Tensor):
            h = np.asarray(arr)
            if h.size and (h.min() < 0 or h.max() >= S):
                raise ValueError("fisher_pairwise: pair index out of range")
    pa, pb = _i32(pair_a, dev), _i32(pair_b, dev)
    P = int(pa.numel())
    row_end = J if row_end is None else row_end
    if out is None:
        out = torch.empty((J, P), dtype=torch.float64, device=dev)
    with torch.cuda.device(dev):
        if max_cell_bound is None:
            native.call("sd_fisher_pairwise", J, S, native.ptr(inc), inc.stride(0), native.ptr(exc), exc.stride(0),
                        P, native.ptr(pa), native.ptr(pb), native.ptr(out), out.stride(0), row_begin, row_end, _sp())
        else:
            native.call("sd_fisher_pairwise_bounded", J, S, native.ptr(inc), inc.stride(0), native.ptr(exc),
                        exc.stride(0), P, native.ptr(pa), native.ptr(pb), native.ptr(out), out.stride(0), row_begin,
                        row_end, int(max_cell_bound), _sp())
    return out


def chi2_pairwise(inc, exc, pair_a, pair_b, row_begin=0, row_end=None, out=None, refused=None):
    """p[j, k] = Yates-corrected chi-squared p (scipy.stats.chi2_contingency(table)[1]) of the same
    tables as fisher_pairwise (sd_chi2_pairwise; fully asynchronous).  Tables scipy refuses (a zero
    margin with a non-zero total) give NaN; ``refused``, a one-element int64 CUDA tensor the caller sets
    to -1, is lowered to the smallest j * n_pairs + k among them (read as uint64: -1 = none)."""
    require_cuda()
    if inc.dtype != torch.int32 or exc.dtype != torch.int64 or not inc.is_cuda or not exc.is_cuda:
        raise TypeError("chi2_pairwise: inc int32 / exc int64 CUDA tensors expected")
    if refused is not None and (refused.dtype != torch.int64 or refused.device != inc.device or refused.numel() != 1):
        raise TypeError("chi2_pairwise: refused must be a one-element int64 tensor on the counts' device")
    J, S = inc.shape
    dev = inc.device
    for arr in (pair_a, pair_b):
        if not isinstance(arr, torch.Tensor):
            h = np.asarray(arr)
            if h.size and (h.min() < 0 or h.max() >= S):
                raise ValueError("chi2_pairwise: pair index out of range")
    pa, pb = _i32(pair_a, dev), _i32(pair_b, dev)
    P = int(pa.numel())
    row_end = J if row_end is None else row_end
    if out is None:
        out = torch.empty((J, P), dtype=torch.float64, device=dev)
    with torch.cuda.device(dev):
        native.call("sd_chi2_pairwise", J, S, native.ptr(inc), inc.stride(0), native.ptr(exc), exc.stride(0), P,
                    native.ptr(pa), native.ptr(pb), native.ptr(out), out.stride(0), row_begin, row_end,
                    native.ptr(refused), _sp())
    return out


def fisher_pairwise_host(inc, exc, pair_a, pair_b, out=None, device=0):
    require_cuda()
    inc = np.ascontiguousarray(inc, dtype=np.int32) if not isinstance(inc, torch.Tensor) else inc
    exc = np.ascontiguousarray(exc, dtype=np.int64) if not isinstance(exc, torch.Tensor) else exc
    J, S = inc.shape
    pa = np.ascontiguousarray(pair_a, dtype=np.int32)
    pb = np.ascontiguousarray(pair_b, dtype=np.int32)
    if out is None:
        out = torch.empty((J, len(pa)), dtype=torch.float64)
    ld = lambda t: t.stride(0) if isinstance(t, torch.Tensor) else t.strides[0] // t.itemsize  # noqa: E731
    native.call("sd_fisher_pairwise_host", device, J, S, native.ptr(inc), ld(inc), native.ptr(exc), ld(exc),
                len(pa), native.ptr(pa), native.ptr(pb), native.ptr(out), ld(out))
    return out


def pairwise_host(inc, row_ptr, col_idx, pair_a, pair_b, out=None, device=0):
    """sd_pairwise_host: host inclusion counts + cluster CSR -> host p-values (exclusion counts are summed
    on the device)."""
    require_cuda()
    inc = np.ascontiguousarray(inc, dtype=np.int32) if not isinstance(inc, torch.Tensor) else inc
    J, S = inc.shape
    rp = np.ascontiguousarray(row_ptr, dtype=np.int32)
    ci = np.ascontiguousarray(col_idx, dtype=np.int32)
    pa = np.ascontiguousarray(pair_a, dtype=np.int32)
    pb = np.ascontiguousarray(pair_b, dtype=np.int32)
    if out is None:
        out = torch.empty((J, len(pa)), dtype=torch.float64)
    ld = lambda t: t.stride(0) if isinstance(t, torch.Tensor) else t.strides[0] // t.itemsize  # noqa: E731
    native.call("sd_pairwise_host", device, J, S, native.ptr(inc), ld(inc), native.ptr(rp), native.ptr(ci), len(pa),
                native.ptr(pa), native.ptr(pb), native.ptr(out), ld(out))
    return out


BH_COLUMNS, BH_ALL = 0, 1
_BH_MAX_VALUES = 2 ** 31 - 1


def bh_adjust(p, mode="pairwise", out=None):
    """Benjamini-Hochberg adjusted p-values of a CUDA float64 matrix [rows, cols] (sd_bh_adjust):
    ``mode='pairwise'`` adjusts every column on its own, ``'all'`` the flattened matrix
    (pairwise_fisher.py:182-191).  ``out`` may be ``p`` itself.  Column mode splits into column
    blocks when the matrix holds more than 2^31 - 1 values."""
    require_cuda()
    if p.dtype != torch.float64 or not p.is_cuda or p.dim() != 2 or (p.numel() and p.stride(1) != 1):
        raise TypeError("bh_adjust: a 2-D float64 CUDA tensor with unit column stride expected")
    if mode not in ("pairwise", "all"):
        raise ValueError("bh_adjust: mode must be 'pairwise' or 'all'")
    if out is None:
        out = torch.empty_like(p)
    rows, cols = p.shape
    if rows == 0 or cols == 0:
        return out
    kind = BH_COLUMNS if mode == "pairwise" else BH_ALL
    if rows * cols > _BH_MAX_VALUES:
        if kind == BH_ALL or rows > _BH_MAX_VALUES:
            raise ValueError("bh_adjust: more than 2^31 - 1 values in one segment")
        step = _BH_MAX_VALUES // rows
    else:
        step = cols
    with torch.cuda.device(p.device):
        ws = None
        for c0 in range(0, cols, step):
            c1 = min(cols, c0 + step)
            need = native.load().sd_bh_workspace_bytes(rows, c1 - c0, kind)
            if need == 0:
                raise native.NativeCallError("sd_bh_workspace_bytes", 1, native.last_error())
            if ws is None or ws.numel() < need:
                ws = torch.empty(need, dtype=torch.uint8, device=p.device)
            src, dst = p[:, c0:c1], out[:, c0:c1]
            native.call("sd_bh_adjust", rows, c1 - c0, native.ptr(src), p.stride(0), native.ptr(dst), out.stride(0),
                        kind, native.ptr(ws), ws.numel(), _sp())
    return out


def fisher_tables(a, b, c, d, device=None):
    """Element-wise two-sided p of [[a, b], [c, d]] (sd_fisher_tables)."""
    dev = _dev(device)
    ts = [torch.as_tensor(np.ascontiguousarray(x, dtype=np.int64)).to(dev) if not isinstance(x, torch.Tensor)
          else x.to(device=dev, dtype=torch.int64).contiguous() for x in (a, b, c, d)]
    n = ts[0].numel()
    out = torch.empty(n, dtype=torch.float64, device=dev)
    with torch.cuda.device(dev):
        native.call("sd_fisher_tables", n, *(native.ptr(t) for t in ts), native.ptr(out), _sp())
    return out


# ---------------------------------------------------------------------------------------
# K6
# ---------------------------------------------------------------------------------------
def ranksum_rows(ps, cols1, cols2, row_begin=0, row_end=None, out=None):
    """Wilcoxon rank-sum test per row between two column groups of a float32 / float64 CUDA PS matrix
    (sd_ranksum_rows; fully asynchronous): scipy.stats.ranksums(x, y, nan_policy='omit') on the non-NaN
    cells x of ``cols1`` and y of ``cols2``.  Returns a dict of [J] CUDA views n1, n2 (int32) and mean1,
    mean2, z, p (float64); only rows [row_begin, row_end) are written.  ``out`` = (int32 [J, >= 2],
    float64 [J, >= 4]) gives the buffers behind those views.  Host column lists are checked here
    (integers in [0, S), each group non-empty and without repeats, the groups disjoint); CUDA int32
    tensors are taken as they are (the kernel never reads a column outside [0, S))."""
    require_cuda()
    if ps.dtype not in (torch.float32, torch.float64) or not ps.is_cuda or ps.dim() != 2:
        raise TypeError("ranksum_rows: ps must be a 2-D float32 / float64 CUDA tensor")
    J, S = ps.shape
    if J and S and ps.stride(1) != 1:
        raise ValueError("ranksum_rows: ps must be row-major")
    dev = ps.device
    host = {}
    for name, cols in (("cols1", cols1), ("cols2", cols2)):
        if isinstance(cols, torch.Tensor) and cols.is_cuda:
            continue
        h = np.asarray(cols.cpu() if isinstance(cols, torch.Tensor) else cols)
        if h.ndim != 1 or h.size == 0 or not np.issubdtype(h.dtype, np.integer):
            raise ValueError(f"ranksum_rows: {name} must be a non-empty list of column indices")
        if h.min() < 0 or h.max() >= S:
            raise ValueError(f"ranksum_rows: {name} has a column outside [0, {S})")
        if np.unique(h).size != h.size:
            raise ValueError(f"ranksum_rows: {name} lists a column twice")
        host[name] = h
    if len(host) == 2 and np.intersect1d(host["cols1"], host["cols2"]).size:
        raise ValueError("ranksum_rows: cols1 and cols2 share a column")
    c1, c2 = _i32(cols1, dev), _i32(cols2, dev)
    row_end = J if row_end is None else row_end
    if out is None:
        out = (torch.empty((J, 2), dtype=torch.int32, device=dev), torch.empty((J, 4), dtype=torch.float64, device=dev))
    n_out, st = out
    if (n_out.dtype != torch.int32 or st.dtype != torch.float64 or n_out.device != dev or st.device != dev
            or n_out.shape[0] != J or st.shape[0] != J or n_out.stride(1) != 1 or st.stride(1) != 1):
        raise TypeError("ranksum_rows: out must be (int32 [J, >= 2], float64 [J, >= 4]) on the PS device")
    kind = native.SD_RANKSUM_F32 if ps.dtype == torch.float32 else native.SD_RANKSUM_F64
    with torch.cuda.device(dev):
        native.call("sd_ranksum_rows", J, S, native.ptr(ps), ps.stride(0), kind, c1.numel(), native.ptr(c1),
                    c2.numel(), native.ptr(c2), row_begin, row_end, native.ptr(n_out), n_out.stride(0),
                    native.ptr(st), st.stride(0), _sp())
    return dict(n1=n_out[:, 0], n2=n_out[:, 1], mean1=st[:, 0], mean2=st[:, 1], z=st[:, 2], p=st[:, 3])


# ---------------------------------------------------------------------------------------
# K7
# ---------------------------------------------------------------------------------------
def kruskal_rows(ps, groups, row_begin=0, row_end=None, out=None):
    """Kruskal-Wallis H test per row across the column groups ``groups`` (a list of k host column-index
    lists) of a float32 / float64 CUDA PS matrix (sd_kruskal_rows; fully asynchronous):
    scipy.stats.kruskal(*groups, nan_policy='omit') on the non-NaN cells, with NaN H and p where a group
    has no defined cell or every defined cell is tied.  Returns a dict of CUDA views n (int32 [J, k]),
    mean (float64 [J, k]), H and p (float64 [J]); only rows [row_begin, row_end) are written.
    ``out`` = (int32 [J, >= k], float64 [J, >= k], float64 [J, >= 2]) gives the buffers behind those
    views.  The lists are checked here: 2 <= k <= 256, each non-empty, integers in [0, S) without
    repeats, the lists disjoint, at most 16,384 columns in all."""
    require_cuda()
    if ps.dtype not in (torch.float32, torch.float64) or not ps.is_cuda or ps.dim() != 2:
        raise TypeError("kruskal_rows: ps must be a 2-D float32 / float64 CUDA tensor")
    J, S = ps.shape
    if J and S and ps.stride(1) != 1:
        raise ValueError("kruskal_rows: ps must be row-major")
    k = len(groups)
    if not 2 <= k <= native.SD_KRUSKAL_MAX_GROUPS:
        raise ValueError(f"kruskal_rows: {k} groups; 2 to {native.SD_KRUSKAL_MAX_GROUPS} are supported")
    host = []
    for g, cols in enumerate(groups):
        h = np.asarray(cols.cpu() if isinstance(cols, torch.Tensor) else cols)
        if h.ndim != 1 or h.size == 0 or not np.issubdtype(h.dtype, np.integer):
            raise ValueError(f"kruskal_rows: group {g} must be a non-empty list of column indices")
        if h.min() < 0 or h.max() >= S:
            raise ValueError(f"kruskal_rows: group {g} has a column outside [0, {S})")
        host.append(h.astype(np.int64))
    cols = np.concatenate(host)
    if cols.size > native.SD_RANKSUM_MAX_SAMPLES:
        raise ValueError(f"kruskal_rows: {cols.size} columns in all; at most {native.SD_RANKSUM_MAX_SAMPLES}")
    if np.unique(cols).size != cols.size:
        raise ValueError("kruskal_rows: a column is listed twice")
    dev = ps.device
    # group by group, so that the lanes of a warp mostly share a label
    group_of = np.repeat(np.arange(k, dtype=np.int32), [len(h) for h in host])
    d_cols, d_group = _i32(cols, dev), _i32(group_of, dev)
    row_end = J if row_end is None else row_end
    if out is None:
        out = (torch.empty((J, k), dtype=torch.int32, device=dev), torch.empty((J, k), dtype=torch.float64, device=dev),
               torch.empty((J, 2), dtype=torch.float64, device=dev))
    n_out, mean, st = out
    if (n_out.dtype != torch.int32 or mean.dtype != torch.float64 or st.dtype != torch.float64
            or any(t.dim() != 2 or t.device != dev or t.shape[0] != J or t.stride(1) != 1 for t in out)
            or n_out.shape[1] < k or mean.shape[1] < k or st.shape[1] < 2):
        raise TypeError("kruskal_rows: out must be (int32 [J, >= k], float64 [J, >= k], float64 [J, >= 2]) "
                        "on the PS device")
    kind = native.SD_RANKSUM_F32 if ps.dtype == torch.float32 else native.SD_RANKSUM_F64
    with torch.cuda.device(dev):
        native.call("sd_kruskal_rows", J, S, native.ptr(ps), ps.stride(0), kind, k, cols.size, native.ptr(d_cols),
                    native.ptr(d_group), row_begin, row_end, native.ptr(n_out), n_out.stride(0), native.ptr(mean),
                    mean.stride(0), native.ptr(st), st.stride(0), _sp())
    return dict(n=n_out[:, :k], mean=mean[:, :k], H=st[:, 0], p=st[:, 1])


# ---------------------------------------------------------------------------------------
# K8
# ---------------------------------------------------------------------------------------
def signedrank_rows(ps, cols1, cols2, row_begin=0, row_end=None, out=None):
    """Wilcoxon signed-rank test per row between matched column pairs (cols1[i], cols2[i]) of a float32 /
    float64 CUDA PS matrix (sd_signedrank_rows; fully asynchronous): scipy.stats.wilcoxon(x, y,
    nan_policy='omit') with the differences taken in the matrix's precision.  Returns a dict of [J] CUDA
    views n, c, method (int32: complete pairs, ranked differences, 0 untested / 1 exact / 2 normal
    approximation) and mean1, mean2, W, p (float64); only rows [row_begin, row_end) are written.
    ``out`` = (int32 [J, >= 3], float64 [J, >= 4]) gives the buffers behind those views.  The lists are
    checked here: the same non-zero length up to 8,192, integers in [0, S), no column listed twice in
    either list or across both."""
    require_cuda()
    if ps.dtype not in (torch.float32, torch.float64) or not ps.is_cuda or ps.dim() != 2:
        raise TypeError("signedrank_rows: ps must be a 2-D float32 / float64 CUDA tensor")
    J, S = ps.shape
    if J and S and ps.stride(1) != 1:
        raise ValueError("signedrank_rows: ps must be row-major")
    host = []
    for name, cols in (("cols1", cols1), ("cols2", cols2)):
        h = np.asarray(cols.cpu() if isinstance(cols, torch.Tensor) else cols)
        if h.ndim != 1 or h.size == 0 or not np.issubdtype(h.dtype, np.integer):
            raise ValueError(f"signedrank_rows: {name} must be a non-empty list of column indices")
        if h.min() < 0 or h.max() >= S:
            raise ValueError(f"signedrank_rows: {name} has a column outside [0, {S})")
        host.append(h)
    if host[0].size != host[1].size:
        raise ValueError(f"signedrank_rows: cols1 has {host[0].size} columns, cols2 {host[1].size}; pairs need both")
    if host[0].size > native.SD_SIGNEDRANK_MAX_PAIRS:
        raise ValueError(f"signedrank_rows: {host[0].size} pairs; at most {native.SD_SIGNEDRANK_MAX_PAIRS}")
    if np.unique(np.concatenate(host)).size != 2 * host[0].size:
        raise ValueError("signedrank_rows: a column is listed twice")
    dev = ps.device
    c1, c2 = _i32(host[0], dev), _i32(host[1], dev)
    row_end = J if row_end is None else row_end
    if out is None:
        out = (torch.empty((J, 3), dtype=torch.int32, device=dev), torch.empty((J, 4), dtype=torch.float64, device=dev))
    n_out, st = out
    if (n_out.dtype != torch.int32 or st.dtype != torch.float64
            or any(t.dim() != 2 or t.device != dev or t.shape[0] != J or t.stride(1) != 1 for t in out)
            or n_out.shape[1] < 3 or st.shape[1] < 4):
        raise TypeError("signedrank_rows: out must be (int32 [J, >= 3], float64 [J, >= 4]) on the PS device")
    kind = native.SD_RANKSUM_F32 if ps.dtype == torch.float32 else native.SD_RANKSUM_F64
    with torch.cuda.device(dev):
        native.call("sd_signedrank_rows", J, S, native.ptr(ps), ps.stride(0), kind, c1.numel(), native.ptr(c1),
                    native.ptr(c2), row_begin, row_end, native.ptr(n_out), n_out.stride(0), native.ptr(st),
                    st.stride(0), _sp())
    return dict(n=n_out[:, 0], c=n_out[:, 1], method=n_out[:, 2], mean1=st[:, 0], mean2=st[:, 1], W=st[:, 2],
                p=st[:, 3])


# ---------------------------------------------------------------------------------------
# K9
# ---------------------------------------------------------------------------------------
def friedman_rows(ps, blocks, row_begin=0, row_end=None, out=None):
    """Friedman test per row across the conditions of a float32 / float64 CUDA PS matrix
    (sd_friedman_rows; fully asynchronous): ``blocks`` is a host int array [n_blocks, k], row b the columns
    of subject b under conditions 0 .. k - 1.  scipy.stats.friedmanchisquare(*conditions,
    nan_policy='omit'): a block with a NaN cell is dropped, Q and p are NaN where no block is complete or
    every complete block is tied throughout.  Returns a dict of CUDA views n (int32 [J]: complete blocks),
    mean (float64 [J, k]: condition means over those blocks), Q and p (float64 [J]); only rows
    [row_begin, row_end) are written.  ``out`` = (int32 [J], float64 [J, >= k], float64 [J, >= 2]) gives
    the buffers behind those views.  The array is checked here: 2-D integer, 3 <= k <= 256, n_blocks >= 1,
    n_blocks * k <= 16,384, every column in [0, S) and none listed twice."""
    require_cuda()
    if ps.dtype not in (torch.float32, torch.float64) or not ps.is_cuda or ps.dim() != 2:
        raise TypeError("friedman_rows: ps must be a 2-D float32 / float64 CUDA tensor")
    J, S = ps.shape
    if J and S and ps.stride(1) != 1:
        raise ValueError("friedman_rows: ps must be row-major")
    h = np.asarray(blocks.cpu() if isinstance(blocks, torch.Tensor) else blocks)
    if h.ndim != 2 or not np.issubdtype(h.dtype, np.integer):
        raise ValueError("friedman_rows: blocks must be a 2-D integer array [n_blocks, k] of column indices")
    nb, k = h.shape
    if not 3 <= k <= native.SD_FRIEDMAN_MAX_CONDITIONS:
        raise ValueError(f"friedman_rows: {k} conditions; 3 to {native.SD_FRIEDMAN_MAX_CONDITIONS} are supported")
    if nb < 1:
        raise ValueError("friedman_rows: no blocks")
    if nb * k > native.SD_RANKSUM_MAX_SAMPLES:
        raise ValueError(f"friedman_rows: {nb} blocks x {k} conditions = {nb * k} cells; "
                         f"at most {native.SD_RANKSUM_MAX_SAMPLES}")
    if h.min() < 0 or h.max() >= S:
        raise ValueError(f"friedman_rows: a column outside [0, {S})")
    if np.unique(h).size != h.size:
        raise ValueError("friedman_rows: a column is listed twice")
    dev = ps.device
    # condition-major: the lanes of a warp hold consecutive subjects of one condition
    d_cols = _i32(np.ascontiguousarray(h.T).reshape(-1), dev)
    row_end = J if row_end is None else row_end
    if out is None:
        out = (torch.empty(J, dtype=torch.int32, device=dev), torch.empty((J, k), dtype=torch.float64, device=dev),
               torch.empty((J, 2), dtype=torch.float64, device=dev))
    n_out, mean, st = out
    if (n_out.dtype != torch.int32 or mean.dtype != torch.float64 or st.dtype != torch.float64
            or n_out.dim() != 1 or n_out.device != dev or n_out.shape[0] != J or (J and n_out.stride(0) != 1)
            or any(t.dim() != 2 or t.device != dev or t.shape[0] != J or t.stride(1) != 1 for t in (mean, st))
            or mean.shape[1] < k or st.shape[1] < 2):
        raise TypeError("friedman_rows: out must be (int32 [J], float64 [J, >= k], float64 [J, >= 2]) on the PS device")
    kind = native.SD_RANKSUM_F32 if ps.dtype == torch.float32 else native.SD_RANKSUM_F64
    with torch.cuda.device(dev):
        native.call("sd_friedman_rows", J, S, native.ptr(ps), ps.stride(0), kind, k, nb, native.ptr(d_cols),
                    row_begin, row_end, native.ptr(n_out), native.ptr(mean), mean.stride(0), native.ptr(st),
                    st.stride(0), _sp())
    return dict(n=n_out, mean=mean[:, :k], Q=st[:, 0], p=st[:, 1])


# ---------------------------------------------------------------------------------------
# K4
# ---------------------------------------------------------------------------------------
def ir_ratio(median, counts, row_ptr=None, col_idx=None, row_begin=0, row_end=None):
    require_cuda()
    J, S = counts.shape
    dev = counts.device
    median = median.to(device=dev, dtype=torch.float64).contiguous()
    rp = None if row_ptr is None else _i32(row_ptr, dev)
    ci = None if col_idx is None else _i32(col_idx, dev)
    out = torch.empty((J, S), dtype=torch.float64, device=dev)
    row_end = J if row_end is None else row_end
    with torch.cuda.device(dev):
        native.call("sd_ir_ratio", J, S, native.ptr(median), median.stride(0), native.ptr(counts), counts.stride(0),
                    native.ptr(rp), native.ptr(ci), native.ptr(out), out.stride(0), row_begin, row_end, _sp())
    return out


def rsd5(cov5):
    require_cuda()
    cov5 = cov5.to(dtype=torch.float64).contiguous()
    n = cov5.numel() // 5
    out = torch.empty(cov5.shape[:-1], dtype=torch.float64, device=cov5.device)
    with torch.cuda.device(cov5.device):
        native.call("sd_rsd5", n, native.ptr(cov5), native.ptr(out), _sp())
    return out


# ---------------------------------------------------------------------------------------
# synthetic inputs + probes
# ---------------------------------------------------------------------------------------
def synth_counts(seed, row0, n_rows, n_cols, p=0.02, logical_cols=None, device=None, out=None):
    from . import synth
    dev = _dev(device)
    if out is None:
        out = torch.empty((n_rows, n_cols), dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        native.call("sd_synth_counts", seed, row0, n_rows, n_cols, n_cols if logical_cols is None else logical_cols,
                    synth.geometric_scale(p), native.ptr(out), out.stride(0), _sp())
    return out


def probe_fp64(device=None):
    dev = _dev(device)
    g = ctypes.c_double()
    with torch.cuda.device(dev):
        native.call("sd_probe_fp64", ctypes.byref(g), _sp())
    return g.value


def probe_copy(nbytes=1 << 30, device=None):
    dev = _dev(device)
    g = ctypes.c_double()
    with torch.cuda.device(dev):
        native.call("sd_probe_copy", nbytes, ctypes.byref(g), _sp())
    return g.value
