"""The faiss surface evo-ssearch's hot path uses, backed by ``libevs.so`` on a B200.

Mirrors (names, argument meaning, error behaviour) the five symbols ``oldapp.py`` touches::

    faiss.IndexFlatIP(d)              oldapp.py:87      -> IndexFlatIP(d)
    index.add(x)                      oldapp.py:88      -> IndexFlatIP.add
    index.search(x, k) -> (D, I)      oldapp.py:2005, :2112 -> IndexFlatIP.search
    faiss.write_index(index, fname)   oldapp.py:98      -> write_index
    faiss.read_index(fname)           oldapp.py:117     -> read_index

so ``import evs as faiss`` leaves the application code unchanged.  Behaviour follows faiss's Python
wrappers (``faiss/python/class_wrappers.py`` ``replacement_add`` / ``replacement_search``): inputs are
made C-contiguous float32, a dimension mismatch or ``k <= 0`` is an ``AssertionError``, library failures
are ``RuntimeError``; results are ``D float32[nq,k]`` descending and ``I int64[nq,k]``, unfilled slots
``(-FLT_MAX, -1)``.

Beyond the reference (SURVEY.md section 8f rank 2): ``add`` and ``search`` also take CUDA ``torch``
tensors and then stay on the device (no ``.cpu().numpy()`` bounce, no host synchronisation).
"""
from __future__ import annotations

import ctypes
import os
from typing import Optional, Tuple

import numpy as np

from . import _lib
from ._lib import EVS_BF16, EVS_F16, EVS_F32, EVS_STORE_BF16_F32, EVS_STORE_F32, check, host_ptr, lib

METRIC_INNER_PRODUCT = 0
METRIC_L2 = 1

_STORAGE = {"f32": EVS_STORE_F32, "fp32": EVS_STORE_F32, "float32": EVS_STORE_F32,
            "bf16": EVS_STORE_BF16_F32, "bfloat16": EVS_STORE_BF16_F32}


def default_device() -> int:
    """CUDA ordinal used when none is given: ``EVS_DEVICE``, else ``LOCAL_RANK`` (torchrun), else 0."""
    for var in ("EVS_DEVICE", "LOCAL_RANK"):
        v = os.environ.get(var)
        if v not in (None, ""):
            return int(v)
    return 0


def default_storage() -> str:
    return os.environ.get("EVS_STORAGE", "f32")


def _is_torch_cuda(x) -> bool:
    return type(x).__module__.startswith("torch") and getattr(x, "is_cuda", False)


def _torch_dtype_code(t) -> int:
    import torch
    return {torch.float32: EVS_F32, torch.float16: EVS_F16, torch.bfloat16: EVS_BF16}[t.dtype]


class IndexFlatIP:
    """Exact inner-product index resident in the HBM of one B200 (faiss ``IndexFlatIP`` drop-in)."""

    def __init__(self, d: int, *, device: Optional[int] = None, storage: Optional[str] = None, _handle=None):
        self._h = ctypes.c_void_p()
        if _handle is not None:
            self._h = _handle
        else:
            storage = default_storage() if storage is None else storage
            if storage not in _STORAGE:
                raise ValueError(f"storage must be one of {sorted(_STORAGE)}")
            dev = default_device() if device is None else int(device)
            check(lib().evs_index_create(int(d), dev, _STORAGE[storage], ctypes.byref(self._h)))
        v = ctypes.c_int(0)
        check(lib().evs_index_d(self._h, ctypes.byref(v)))
        self.d = v.value
        check(lib().evs_index_device(self._h, ctypes.byref(v)))
        self.device = v.value
        check(lib().evs_index_storage(self._h, ctypes.byref(v)))
        self.storage = "bf16" if v.value == EVS_STORE_BF16_F32 else "f32"
        self.is_trained = True
        self.metric_type = METRIC_INNER_PRODUCT
        self.verbose = False

    # -- lifetime ---------------------------------------------------------------------------
    def __del__(self):
        h, self._h = getattr(self, "_h", None), None
        if h:
            try:
                lib().evs_index_free(h)
            except Exception:
                pass

    @property
    def ntotal(self) -> int:
        n = ctypes.c_int64(0)
        check(lib().evs_index_ntotal(self._h, ctypes.byref(n)))
        return n.value

    @property
    def id_base(self) -> int:
        n = ctypes.c_int64(0)
        check(lib().evs_index_id_base(self._h, ctypes.byref(n)))
        return n.value

    @id_base.setter
    def id_base(self, base: int) -> None:
        check(lib().evs_index_set_id_base(self._h, int(base)))

    def reserve(self, nrows: int) -> None:
        check(lib().evs_index_reserve(self._h, int(nrows)))

    def set_storage(self, storage: str) -> None:
        """Switch the scan precision in place: ``"bf16"`` derives the bf16 scan copy of an fp32-storage index (large
        query batches then run the bf16 tensor-core scan instead of tf32 from the fp32 rows), ``"f32"`` drops it."""
        if storage not in _STORAGE:
            raise ValueError(f"storage must be one of {sorted(_STORAGE)}")
        check(lib().evs_index_set_storage(self._h, _STORAGE[storage]))
        self.storage = "bf16" if _STORAGE[storage] == EVS_STORE_BF16_F32 else "f32"

    @property
    def max_row_norm(self) -> float:
        """Largest row norm (it scales the certification bound of the searches)."""
        v = ctypes.c_float(0)
        check(lib().evs_index_max_row_norm(self._h, ctypes.byref(v)))
        return v.value

    def guard_stats(self):
        """``(reruns, uncertified)``: queries finalised again from the device-side exact re-run, and results that
        stayed uncertified, since the index was created."""
        r, u = ctypes.c_int64(0), ctypes.c_int64(0)
        check(lib().evs_index_guard_stats(self._h, ctypes.byref(r), ctypes.byref(u)))
        return r.value, u.value

    def shadow_stats(self):
        """``(wide_searches, emax, last_candidates)``: single-query searches of the int8 scan copy whose window held more
        than 256 candidates, the largest ``|x - s c|_2`` of a row of the copy (-1 without a copy), and how many
        candidates (the window C) the last search of the copy re-scored exactly."""
        w, e, c = ctypes.c_int64(0), ctypes.c_float(0), ctypes.c_int64(0)
        check(lib().evs_index_shadow_stats(self._h, ctypes.byref(w), ctypes.byref(e), ctypes.byref(c)))
        return w.value, e.value, c.value

    def large_k_stats(self):
        """``(searches, last_candidates)``: searches with k > 112 (option ``max_k``) on this index, and how many rows the
        last one re-scored exactly (its largest candidate set over the queries)."""
        s, c = ctypes.c_int64(0), ctypes.c_int64(0)
        check(lib().evs_index_large_k_stats(self._h, ctypes.byref(s), ctypes.byref(c)))
        return s.value, c.value

    def coalesce_stats(self):
        """``(groups, grouped_queries, i8_batch_passes)``: groups of two or more concurrent single-query ``search`` calls
        served as one search and the queries they held (a caller that found the index idle moves neither), and the passes
        of the exact batch search of the int8 copy (batches of 2..4 queries, any entry point)."""
        g, q, p = ctypes.c_int64(0), ctypes.c_int64(0), ctypes.c_int64(0)
        check(lib().evs_index_coalesce_stats(self._h, ctypes.byref(g), ctypes.byref(q), ctypes.byref(p)))
        return g.value, q.value, p.value

    def scan_clocks(self) -> np.ndarray:
        """Diagnostics (option ``scan_clock``): ``uint64[nctas, 2]`` start / end-of-scan-loop times (ns) of the CTAs of
        the last fused single-query scan."""
        n = ctypes.c_int64(0)
        check(lib().evs_index_scan_clocks(self._h, None, 0, ctypes.byref(n)))
        out = np.zeros((n.value + 12, 2), np.uint64)
        if n.value:
            check(lib().evs_index_scan_clocks(self._h, out.ctypes.data_as(ctypes.c_void_p), n.value + 12, ctypes.byref(n)))
        # the last CTA: [ticket taken, finalise (+ merge) done, buffers sorted, list merged + stored, scan loop left] and the
        # finalise's phases [head blocks loaded, survivors, ranked, re-scored, results written, ...] (16 slots; slots 8-13:
        # the int8 window pass, evs_scan.cuh)
        self.last_cta_stamps = out[n.value:n.value + 4].reshape(-1)
        self.finalize_stamps = out[n.value + 4:n.value + 12].reshape(-1)
        return out[:n.value]

    def reset(self) -> None:
        """faiss ``Index.reset``: drop all vectors."""
        base = self.id_base
        new = IndexFlatIP(self.d, device=self.device, storage=self.storage)
        new.id_base = base
        old, self._h, new._h = self._h, new._h, None
        lib().evs_index_free(old)

    # -- add ----------------------------------------------------------------------------------
    def add(self, x) -> None:
        """``index.add(embeddings_array)`` (oldapp.py:88).  ``x``: ``(n, d)`` array-like or CUDA tensor."""
        if _is_torch_cuda(x):
            import torch
            assert x.dim() == 2
            n, d = x.shape
            assert d == self.d
            assert x.device.index == self.device, "tensor is on another device than the index"
            if x.dtype not in (torch.float32, torch.float16, torch.bfloat16):
                x = x.float()
            x = x.contiguous()
            st = torch.cuda.current_stream(x.device).cuda_stream
            check(lib().evs_index_add_dev(self._h, n, ctypes.c_void_p(x.data_ptr()), _torch_dtype_code(x),
                                          ctypes.c_void_p(st)))
            return
        x = np.asarray(x)
        n, d = x.shape
        assert d == self.d
        x = np.ascontiguousarray(x, dtype="float32")
        check(lib().evs_index_add(self._h, n, x.ctypes.data_as(ctypes.c_void_p)))

    def add_rows_from(self, src: "IndexFlatIP", rows) -> None:
        """Append rows ``rows`` (ids into ``src``) of another index on the same device, device to device."""
        rows = np.ascontiguousarray(np.asarray(rows, dtype=np.int64))
        assert rows.ndim == 1 and src.d == self.d
        check(lib().evs_index_add_rows_from(self._h, src._h, rows.shape[0], rows.ctypes.data_as(ctypes.c_void_p)))

    def add_synthetic(self, n: int, seed: int, normalize: bool = True) -> None:
        """Append ``n`` counter-based synthetic rows generated on the device (bench / tests)."""
        check(lib().evs_index_add_synth(self._h, int(n), int(seed), int(bool(normalize))))

    # -- search -------------------------------------------------------------------------------
    def search(self, x, k: int, *, params=None, D=None, I=None):
        """``index.search(q.reshape(1, -1), k)`` (oldapp.py:2005, :2112) -> ``(D, I)``."""
        assert params is None, "search params are not supported by a flat index"
        if _is_torch_cuda(x):
            return self._search_torch(x, k, D, I)
        x = np.asarray(x)
        n, d = x.shape
        x = np.ascontiguousarray(x, dtype="float32")
        assert d == self.d
        assert k > 0
        if D is None:
            D = np.empty((n, k), dtype=np.float32)
        else:
            assert D.shape == (n, k) and D.dtype == np.float32 and D.flags.c_contiguous
        if I is None:
            I = np.empty((n, k), dtype=np.int64)
        else:
            assert I.shape == (n, k) and I.dtype == np.int64 and I.flags.c_contiguous
        check(lib().evs_index_search(self._h, n, host_ptr(x), int(k), host_ptr(D), host_ptr(I)))
        return D, I

    def _search_torch(self, x, k: int, D=None, I=None):
        import torch
        assert x.dim() == 2
        n, d = x.shape
        assert d == self.d
        assert k > 0
        assert x.device.index == self.device, "tensor is on another device than the index"
        x = x.to(torch.float32).contiguous()
        if D is None:
            D = torch.empty((n, k), dtype=torch.float32, device=x.device)
        if I is None:
            I = torch.empty((n, k), dtype=torch.int64, device=x.device)
        assert D.is_contiguous() and I.is_contiguous() and D.shape == (n, k) and I.shape == (n, k)
        st = torch.cuda.current_stream(x.device).cuda_stream
        check(lib().evs_index_search_dev(self._h, n, ctypes.c_void_p(x.data_ptr()), int(k),
                                         ctypes.c_void_p(D.data_ptr()), ctypes.c_void_p(I.data_ptr()),
                                         ctypes.c_void_p(st)))
        return D, I

    def search_partial(self, x, k: int):
        """Row-sharded search, stage 1 (CUDA tensors only): this shard's k best as
        ``(scores float64[nq,k], ids int64[nq,k])`` with global ids (``id_base`` added)."""
        import torch
        assert _is_torch_cuda(x) and x.dim() == 2 and x.shape[1] == self.d and k > 0
        x = x.to(torch.float32).contiguous()
        n = x.shape[0]
        S = torch.empty((n, k), dtype=torch.float64, device=x.device)
        I = torch.empty((n, k), dtype=torch.int64, device=x.device)
        st = torch.cuda.current_stream(x.device).cuda_stream
        check(lib().evs_index_search_partial_dev(self._h, n, ctypes.c_void_p(x.data_ptr()), int(k),
                                                 ctypes.c_void_p(S.data_ptr()), ctypes.c_void_p(I.data_ptr()),
                                                 ctypes.c_void_p(st)))
        return S, I

    def search_exchange(self, exchange: "PeerExchange", x, k: int):
        """Row-sharded search in one call (CUDA tensors only): scan this shard, store its k best into every
        rank's exchange slot over NVLink, wait for all shards' partials and merge -> final ``(D, I)``.
        Collective: every rank calls it in the same order with the same ``nq`` and ``k``."""
        import torch
        assert _is_torch_cuda(x) and x.dim() == 2 and x.shape[1] == self.d and k > 0
        x = x.to(torch.float32).contiguous()
        n = x.shape[0]
        D = torch.empty((n, k), dtype=torch.float32, device=x.device)
        I = torch.empty((n, k), dtype=torch.int64, device=x.device)
        st = torch.cuda.current_stream(x.device).cuda_stream
        check(lib().evs_index_search_exchange_dev(self._h, exchange._h, n, ctypes.c_void_p(x.data_ptr()), int(k),
                                                  ctypes.c_void_p(D.data_ptr()), ctypes.c_void_p(I.data_ptr()),
                                                  ctypes.c_void_p(st)))
        return D, I

    def search_exchange_host(self, exchange: "PeerExchange", x, k: int):
        """``search_exchange`` for numpy queries: staging, copies and the one synchronisation are done by the library
        (``evs_index_search_exchange``).  Collective, like ``search_exchange``."""
        x = np.ascontiguousarray(np.asarray(x), dtype="float32")
        n, d = x.shape
        assert d == self.d and k > 0
        D = np.empty((n, k), dtype=np.float32)
        I = np.empty((n, k), dtype=np.int64)
        check(lib().evs_index_search_exchange(self._h, exchange._h, n, host_ptr(x), int(k), host_ptr(D), host_ptr(I)))
        return D, I

    def last_margins(self, nq: int) -> np.ndarray:
        """Safety margin per query of the last search (see ``evs_index_last_margins``)."""
        out = np.empty(nq, np.float32)
        check(lib().evs_index_last_margins(self._h, nq, out.ctypes.data_as(ctypes.c_void_p)))
        return out

    def time_scan(self, xq_cuda, k: int, iters: int = 20) -> float:
        """Mean device time (ms) of the scan stage alone, CUDA events on the index's stream."""
        import torch
        assert _is_torch_cuda(xq_cuda) and xq_cuda.dtype == torch.float32 and xq_cuda.is_contiguous()
        torch.cuda.synchronize(xq_cuda.device)
        ms = ctypes.c_float(0)
        check(lib().evs_index_time_scan(self._h, xq_cuda.shape[0], ctypes.c_void_p(xq_cuda.data_ptr()), int(k),
                                        int(iters), ctypes.byref(ms)))
        return ms.value

    def tc_max_queries(self) -> int:
        """Queries one tensor-core pass serves for this index (0 = dimension not supported)."""
        v = ctypes.c_int(0)
        check(lib().evs_index_tc_max_queries(self._h, ctypes.byref(v)))
        return v.value

    def tc_x3_max_queries(self) -> int:
        """Queries one 3xTF32 pass serves for this index (0: bf16 storage, option off, or dimension not supported)."""
        v = ctypes.c_int(0)
        check(lib().evs_index_tc_x3_max_queries(self._h, ctypes.byref(v)))
        return v.value

    def tc_scores(self, xq_cuda):
        """Diagnostics: raw tensor-core scan scores, ``float32[ntotal, nq]`` CUDA tensor."""
        import torch
        assert _is_torch_cuda(xq_cuda) and xq_cuda.dtype == torch.float32 and xq_cuda.is_contiguous()
        nq = xq_cuda.shape[0]
        got = ctypes.c_int(0)
        st = torch.cuda.current_stream(xq_cuda.device).cuda_stream
        check(lib().evs_index_tc_scores_dev(self._h, nq, ctypes.c_void_p(xq_cuda.data_ptr()), None, ctypes.byref(got),
                                            ctypes.c_void_p(st)))  # pitch query
        pitch = got.value
        out = torch.empty((self.ntotal, pitch), dtype=torch.float32, device=xq_cuda.device)
        check(lib().evs_index_tc_scores_dev(self._h, nq, ctypes.c_void_p(xq_cuda.data_ptr()), ctypes.c_void_p(out.data_ptr()),
                                            ctypes.byref(got), ctypes.c_void_p(st)))
        assert got.value == pitch
        return out[:, :nq]

    def scan_profile(self):
        """(searches recorded, summed scan ms) since the last call; needs ``set_option("profile_scans", 1)``."""
        n, ms = ctypes.c_int64(0), ctypes.c_double(0)
        check(lib().evs_index_scan_profile(self._h, ctypes.byref(n), ctypes.byref(ms)))
        return n.value, ms.value

    # -- reconstruct ----------------------------------------------------------------------------
    def reconstruct_n(self, n0: int = 0, ni: int = -1) -> np.ndarray:
        if ni == -1:
            ni = self.ntotal - n0
        out = np.empty((ni, self.d), np.float32)
        check(lib().evs_index_get_rows(self._h, int(n0), int(ni), out.ctypes.data_as(ctypes.c_void_p)))
        return out

    def reconstruct(self, key: int) -> np.ndarray:
        return self.reconstruct_n(int(key), 1)[0]


class PeerExchange:
    """Symmetric peer-mapped buffer for the shard-partial exchange (``evs_exchange_*``): replaces the
    all-gather + merge of a row-sharded search by NVLink stores issued from the finalise kernel and a
    flag-waiting merge kernel.  One per rank; ``connect`` takes the 64-byte handles of all ranks in
    rank order (exchanged by the caller, e.g. ``torch.distributed.all_gather``)."""

    def __init__(self, device: int, rank: int, world: int, max_nq: int = 1024, max_k: int = 48):
        self._h = ctypes.c_void_p()
        self.rank, self.world, self.max_nq, self.max_k = int(rank), int(world), int(max_nq), int(max_k)
        check(lib().evs_exchange_create(int(device), self.rank, self.world, self.max_nq, self.max_k, ctypes.byref(self._h)))

    def __del__(self):
        h, self._h = getattr(self, "_h", None), None
        if h:
            try:
                lib().evs_exchange_free(h)
            except Exception:
                pass

    def handle(self) -> bytes:
        buf = ctypes.create_string_buffer(_lib.EVS_IPC_HANDLE_BYTES)
        check(lib().evs_exchange_handle(self._h, buf, _lib.EVS_IPC_HANDLE_BYTES))
        return buf.raw

    def connect(self, handles) -> None:
        """``handles``: the ``world`` handles in rank order (bytes objects or one concatenated bytes)."""
        blob = handles if isinstance(handles, (bytes, bytearray)) else b"".join(bytes(h) for h in handles)
        assert len(blob) == self.world * _lib.EVS_IPC_HANDLE_BYTES
        check(lib().evs_exchange_connect(self._h, ctypes.c_char_p(bytes(blob)), len(blob)))

    def status(self):
        """``(timed_out, searches)``: whether any merge gave up waiting for a rank, and the search count."""
        t, n = ctypes.c_int(0), ctypes.c_int64(0)
        check(lib().evs_exchange_status(self._h, ctypes.byref(t), ctypes.byref(n)))
        return bool(t.value), n.value


def write_index(index: IndexFlatIP, fname: str) -> None:
    """``faiss.write_index(index, path)`` (oldapp.py:98): 45-byte flat header + fp32 payload."""
    check(lib().evs_index_write(index._h, os.fsencode(str(fname))))


def read_index(fname: str, *, device: Optional[int] = None, storage: Optional[str] = None) -> IndexFlatIP:
    """``faiss.read_index(path)`` (oldapp.py:117): file -> pinned staging -> HBM, resident index."""
    storage = default_storage() if storage is None else storage
    dev = default_device() if device is None else int(device)
    h = ctypes.c_void_p()
    check(lib().evs_index_read(os.fsencode(str(fname)), dev, _STORAGE[storage], ctypes.byref(h)))
    return IndexFlatIP(0, _handle=h)


def read_index_rows(fname: str, row_lo: int, row_hi: int, *, device: Optional[int] = None,
                    storage: Optional[str] = None) -> Tuple[IndexFlatIP, int]:
    """The shard loader: rows ``[row_lo, row_hi)`` of an ``index.faiss`` (only that byte range of the file is read)
    -> ``(index with id_base = row_lo, rows in the file)``."""
    storage = default_storage() if storage is None else storage
    dev = default_device() if device is None else int(device)
    h, n = ctypes.c_void_p(), ctypes.c_int64(0)
    check(lib().evs_index_read_rows(os.fsencode(str(fname)), dev, _STORAGE[storage], int(row_lo), int(row_hi),
                                    ctypes.byref(h), ctypes.byref(n)))
    return IndexFlatIP(0, _handle=h), n.value


def index_file_info(fname: str) -> Tuple[int, int]:
    """``(d, ntotal)`` from the 45-byte header of an ``index.faiss``."""
    d, n = ctypes.c_int(0), ctypes.c_int64(0)
    check(lib().evs_index_file_info(os.fsencode(str(fname)), ctypes.byref(d), ctypes.byref(n)))
    return d.value, n.value


def normalize_L2(x) -> None:
    """``faiss.normalize_L2(x)`` / ``x /= x.norm(dim=-1, keepdim=True)`` (oldapp.py:35/43/51), in place.

    ``x``: ``(n, d)`` float32 numpy array (staged through the device) or a CUDA tensor of dtype
    float32 / float16 / bfloat16 (normalised where it lies).  No epsilon: a zero row becomes NaN.
    """
    if _is_torch_cuda(x):
        import torch
        assert x.dim() == 2 and x.is_contiguous()
        st = torch.cuda.current_stream(x.device).cuda_stream
        check(lib().evs_l2_normalize_dev(x.device.index, ctypes.c_void_p(x.data_ptr()), x.shape[0], x.shape[1],
                                         _torch_dtype_code(x), ctypes.c_void_p(st)))
        return
    assert isinstance(x, np.ndarray) and x.dtype == np.float32 and x.ndim == 2 and x.flags.c_contiguous
    check(lib().evs_l2_normalize(default_device(), host_ptr(x), x.shape[0], x.shape[1]))


def merge_partials(scores, ids, k: int):
    """Row-sharded search, stage 2: ``scores float64[G,nq,k]``, ``ids int64[G,nq,k]`` CUDA tensors
    (the all-gathered shard partials) -> final ``(D float32[nq,k], I int64[nq,k])`` on the same device.
    The two may be strided views of one gathered buffer as long as each ``[nq,k]`` block is dense and
    both use the same part stride."""
    import torch
    assert scores.is_cuda and ids.is_cuda and scores.dtype == torch.float64 and ids.dtype == torch.int64
    assert scores.shape == ids.shape and scores.dim() == 3
    G, nq, kk = scores.shape
    assert kk == k
    assert scores.stride()[1:] == (k, 1) and ids.stride()[1:] == (k, 1) and scores.stride(0) == ids.stride(0)
    D = torch.empty((nq, k), dtype=torch.float32, device=scores.device)
    I = torch.empty((nq, k), dtype=torch.int64, device=scores.device)
    st = torch.cuda.current_stream(scores.device).cuda_stream
    check(lib().evs_merge_partials_dev(scores.device.index, G, nq, k, ctypes.c_void_p(scores.data_ptr()),
                                       ctypes.c_void_p(ids.data_ptr()), scores.stride(0) if G > 1 else 0,
                                       ctypes.c_void_p(D.data_ptr()),
                                       ctypes.c_void_p(I.data_ptr()), ctypes.c_void_p(st)))
    return D, I
