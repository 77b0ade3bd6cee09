"""Index lifecycle and search entry points of the application, kept by name.

Mirrors ``oldapp.py``::

    create_index(folder)                         oldapp.py:54-90   (+ batched indexing, config.BATCH_SIZE)
    update_index(folder)                         -- incremental re-index from metadata.pkl (SURVEY.md 8(f) rank 4)
    save_index(index, paths, metadata, folder)   oldapp.py:92-106
    load_index(folder)                           oldapp.py:108-135
    search (text) handler body                   oldapp.py:1985-2045  -> search_text
    search_by_image handler body                 oldapp.py:2065-2152  -> search_image

with the same ``<folder>/.clip_index/{index.faiss, paths.pkl, metadata.pkl}`` files.  What changes is the
engine underneath (``IndexFlatIP`` on the GPU) and that ``load_index`` keeps indexes RESIDENT: the
reference re-reads the whole ``index.faiss`` on every request (oldapp.py:1993, :2084); here a loaded
index stays in HBM, keyed by the file's (path, mtime, size) and reloaded only when that changes.

The CLIP encoder is out of scope (north_star: "unchanged CLIP ViT encoder"); callers pass any object
with the reference's three embedding functions (``get_image_embedding``, ``get_image_embedding_from_pil``,
``get_text_embedding``; oldapp.py:30-52).  HTTP, thumbnails and JSON stay in the application.
"""
from __future__ import annotations

import os
import pickle
import threading
from collections import OrderedDict
from pathlib import Path
from typing import Any, List, Optional, Tuple

import numpy as np

from . import _lib
from .config import config
from .index import IndexFlatIP, read_index, write_index

# Resident indexes: an LRU keyed by the resolved path of index.faiss, bounded by a byte budget (HBM held by the cached
# indexes on this GPU; EVS_CACHE_BYTES, default 120 GiB of the B200's 180 GB).  An entry is valid while the
# (mtime_ns, size) of index.faiss, paths.pkl AND metadata.pkl are unchanged -- save_index writes the three files one
# after the other, so index.faiss alone would pin "new vectors, old paths" if another process loaded in between.
_cache_lock = threading.Lock()
_cache: "OrderedDict[str, tuple]" = OrderedDict()  # key -> (signature, index, paths, metadata, bytes)
CACHE_BUDGET_BYTES = int(os.environ.get("EVS_CACHE_BYTES", str(120 << 30)))
load_stats = {"loads": 0, "bytes": 0, "seconds": 0.0, "evictions": 0}  # what the loader did (bench / tests)


def _index_bytes(index) -> int:
    local = getattr(index, "local", index)  # a sharded index holds only its block on this GPU
    # fp32 rows; the bf16 rows of bf16 storage; the int8 scan copy (one byte per element, one fp32 scale per row) that
    # bf16 storage always keeps and an fp32 index built with the option "scan_shadow" on keeps
    bf16 = getattr(index, "storage", "f32") == "bf16"
    copy = bf16 or (hasattr(local, "shadow_stats") and local.shadow_stats()[1] >= 0)
    n, d = int(local.ntotal), index.d
    return n * d * (4 + (2 if bf16 else 0) + (1 if copy else 0)) + (4 * n if copy else 0)


def _signature(index_path: Path):
    sig = []
    for name in ("index.faiss", "paths.pkl", "metadata.pkl"):
        try:
            st = os.stat(index_path / name)
            sig.append((st.st_mtime_ns, st.st_size))
        except OSError:
            sig.append(None)
    return tuple(sig)


def _cache_put(key: str, sig, index, paths, meta) -> None:
    nbytes = _index_bytes(index)
    with _cache_lock:
        _cache.pop(key, None)
        _cache[key] = (sig, index, paths, meta, nbytes)
        total = sum(e[4] for e in _cache.values())
        while total > CACHE_BUDGET_BYTES and len(_cache) > 1:  # least recently used first; never the entry just added
            _, old = _cache.popitem(last=False)
            total -= old[4]
            load_stats["evictions"] += 1


def _want_sharded(sharded: Optional[bool]) -> bool:
    if sharded is not None:
        return bool(sharded)
    env = os.environ.get("EVS_SHARDED", "auto").lower()
    if env in ("0", "no", "false"):
        return False
    try:
        import torch.distributed as dist
        return dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1
    except Exception:  # noqa: BLE001
        return False


def _walk(folder_path: Path) -> List[Path]:
    """The reference's walk: one non-recursive glob per supported extension (oldapp.py:64-65)."""
    out: List[Path] = []
    for ext in config.SUPPORTED_EXTENSIONS:
        out.extend(folder_path.glob(f"*{ext}"))
    return out


def _is_cuda_tensor(x) -> bool:
    return type(x).__module__.startswith("torch") and getattr(x, "is_cuda", False)


def _embed_files(files: List[Path], encoder, batch_size: int, index: Optional[IndexFlatIP]):
    """Embed ``files`` and append the embeddings to ``index`` (created on first use) in order.

    Two encoder protocols:
      * the reference's ``get_image_embedding(path) -> (d,)`` (already normalised, oldapp.py:30-37), called
        per image and stacked ``BATCH_SIZE`` at a time before one ``add`` -- ``np.array(...).astype('float32')``
        as oldapp.py:86;
      * optional ``encode_images(paths) -> (m, d)`` raw (un-normalised) features as a numpy array or a CUDA
        tensor of dtype float32/float16/bfloat16, i.e. one batched CLIP forward (SURVEY.md 8(f) rank 3: the
        reference's ``config.BATCH_SIZE`` is dead code).  The batch is L2-normalised by the library's kernel
        where it lies (oldapp.py:35 done for ``m`` rows at once) and appended without leaving the device.  A
        batch that fails is retried image by image so that one unreadable file only drops itself.
    Returns ``(index, ok_files)``; files whose embedding failed are printed and skipped like the reference.
    """
    from .index import normalize_L2
    ok: List[Path] = []
    batched = getattr(encoder, "encode_images", None)
    for b0 in range(0, len(files), batch_size):
        chunk = files[b0:b0 + batch_size]
        feats = None
        if batched is not None:
            try:
                feats = batched([str(p) for p in chunk])
                if feats.shape[0] != len(chunk):
                    raise ValueError("encode_images returned a different number of rows")
            except Exception as e:  # noqa: BLE001
                print(f"Error processing batch of {len(chunk)} images ({e}); retrying one by one")
                feats = None
        if feats is not None:
            if _is_cuda_tensor(feats):
                feats = feats.contiguous()
            else:
                feats = np.ascontiguousarray(np.asarray(feats), dtype="float32")
            normalize_L2(feats)
            good = chunk
        else:
            rows, good = [], []
            for img_path in chunk:
                try:
                    rows.append(encoder.get_image_embedding(img_path))
                    good.append(img_path)
                except Exception as e:  # noqa: BLE001 - the reference prints and continues
                    print(f"Error processing {img_path}: {e}")
            if not rows:
                continue
            feats = np.array(rows).astype("float32")
        if index is None:
            index = IndexFlatIP(int(feats.shape[1]))
        index.add(feats)
        ok.extend(good)
    return index, ok


def _file_meta(img_path: Path) -> dict:
    stat = img_path.stat()
    return {"path": str(img_path), "mtime": stat.st_mtime, "size": stat.st_size}


def create_index(folder_path, encoder, batch_size: Optional[int] = None
                 ) -> Tuple[Optional[IndexFlatIP], Optional[List[str]], Optional[List[dict]]]:
    """Embed every supported image directly inside ``folder_path`` and build the index (oldapp.py:54-90).

    Same walk as the reference: one non-recursive glob per extension, per-image failures are printed
    and skipped, ``(None, None, None)`` when nothing could be embedded.  Embeddings are appended
    ``batch_size`` (default ``config.BATCH_SIZE``) rows at a time; see ``_embed_files`` for the two encoder
    protocols.  With the reference's per-image protocol the index rows are exactly
    ``np.array(embeddings).astype('float32')`` (oldapp.py:86).
    """
    folder_path = Path(folder_path)
    batch_size = max(1, int(batch_size or config.BATCH_SIZE))
    index, ok = _embed_files(_walk(folder_path), encoder, batch_size, None)
    if index is None or not ok:
        return None, None, None
    return index, [str(p) for p in ok], [_file_meta(p) for p in ok]


def update_index(folder_path, encoder, batch_size: Optional[int] = None):
    """Incremental re-index (SURVEY.md 8(f) rank 4): re-use the stored embedding of every file whose
    ``(path, mtime, size)`` still matches ``metadata.pkl`` (oldapp.py:71-78 writes exactly these), embed only
    new or changed files, drop deleted ones.  Kept rows never leave the GPU (``evs_index_add_rows_from``).

    Returns ``(index, image_paths, image_metadata, stats)`` in the order a fresh ``create_index`` would
    produce, so the two are interchangeable; the caller saves with ``save_index`` as after ``create_index``.
    Falls back to ``create_index`` when the folder has no usable index or no metadata.
    """
    folder_path = Path(folder_path)
    batch_size = max(1, int(batch_size or config.BATCH_SIZE))
    old_index, old_paths, old_meta = load_index(folder_path)
    files = _walk(folder_path)
    stats = {"kept": 0, "embedded": 0, "removed": 0, "failed": 0}
    if old_index is None or not old_meta or len(old_meta) != len(old_paths) or old_index.ntotal != len(old_paths):
        index, paths, meta = create_index(folder_path, encoder, batch_size)
        stats["embedded"] = 0 if paths is None else len(paths)
        stats["failed"] = len(files) - stats["embedded"]
        return index, paths, meta, stats
    known = {m["path"]: (row, m.get("mtime"), m.get("size")) for row, m in enumerate(old_meta)}
    plan = []   # per file in walk order: ("keep", old row, meta) or ("new", position among the files to embed, None)
    todo: List[Path] = []
    for img_path in files:
        hit = known.get(str(img_path))
        try:
            meta = _file_meta(img_path)
        except OSError as e:
            print(f"Error processing {img_path}: {e}")
            stats["failed"] += 1
            continue
        if hit is not None and hit[1] == meta["mtime"] and hit[2] == meta["size"]:
            plan.append(("keep", hit[0], meta))
        else:
            plan.append(("new", len(todo), meta))
            todo.append(img_path)
    fresh, ok = _embed_files(todo, encoder, batch_size, None)
    ok_pos = {str(p): i for i, p in enumerate(ok)}  # row of each successfully embedded file in `fresh`
    stats["failed"] += len(todo) - len(ok)
    # pool = [kept rows of the old index][fresh rows]; the final index is one gather of the pool in walk order
    kept_rows = [row for kind, row, _ in plan if kind == "keep"]
    d = old_index.d
    pool = IndexFlatIP(d, device=old_index.device, storage="f32")
    if kept_rows:
        pool.add_rows_from(old_index, kept_rows)
    if fresh is not None and fresh.ntotal:
        pool.add_rows_from(fresh, np.arange(fresh.ntotal))
    perm, paths, metas = [], [], []
    nkept = 0
    for kind, ref, meta in plan:
        if kind == "keep":
            perm.append(nkept)
            nkept += 1
        else:
            pos = ok_pos.get(str(todo[ref]))
            if pos is None:
                continue  # embedding failed: skipped like create_index does
            perm.append(len(kept_rows) + pos)
        paths.append(meta["path"])
        metas.append(meta)
    stats["kept"] = len(kept_rows)
    stats["embedded"] = len(ok)
    stats["removed"] = len(old_paths) - len(kept_rows) - sum(1 for p in todo if str(p) in known)
    if not perm:
        return None, None, None, stats
    index = IndexFlatIP(d, device=old_index.device, storage=old_index.storage)
    index.add_rows_from(pool, perm)
    return index, paths, metas, stats


def save_index(index: IndexFlatIP, image_paths, image_metadata, folder_path) -> None:
    """Write ``index.faiss``, ``paths.pkl``, ``metadata.pkl`` under ``<folder>/.clip_index`` (oldapp.py:92-106)."""
    index_path = Path(folder_path) / config.INDEX_FOLDER_NAME
    index_path.mkdir(exist_ok=True)
    write_index(index, str(index_path / "index.faiss"))
    with open(index_path / "paths.pkl", "wb") as f:
        pickle.dump(image_paths, f)
    with open(index_path / "metadata.pkl", "wb") as f:
        pickle.dump(image_metadata, f)
    # the index just written is the resident one for this folder
    key = str((index_path / "index.faiss").resolve())
    _cache_put(key, _signature(index_path), index, list(image_paths), image_metadata)


def _read_resident(fname: Path, sharded: bool):
    """index.faiss -> HBM.  Sharded: every rank reads only its own row block of the file (collective call)."""
    import time
    t0 = time.perf_counter()
    if sharded:
        from .sharded import ShardedIndexFlatIP
        index = ShardedIndexFlatIP.read_index(str(fname), exchange=os.environ.get("EVS_EXCHANGE", "peer"))
    else:
        index = read_index(str(fname))
    load_stats["loads"] += 1
    load_stats["bytes"] += int(getattr(index, "local", index).ntotal) * index.d * 4
    load_stats["seconds"] += time.perf_counter() - t0
    return index


def load_index(folder_path, sharded: Optional[bool] = None):
    """``(index, image_paths, image_metadata)`` or ``(None, None, None)`` (oldapp.py:108-135).

    Any failure -- missing folder, corrupt file, unreadable pickle -- yields the ``None`` triple, as the
    reference's blanket ``except`` does.  A hit in the resident cache costs three ``stat`` calls.

    ``sharded`` (default: automatic -- true when ``torch.distributed`` is initialised with more than one rank; env
    ``EVS_SHARDED=0`` forces it off): the index is row-sharded over the ranks' GPUs, each rank streaming only its own
    block of ``index.faiss`` into its HBM, and the returned object is a ``ShardedIndexFlatIP`` with the same
    ``search(x, k)``.  Then ``load_index`` and the searches are collective calls.
    """
    index_path = Path(folder_path) / config.INDEX_FOLDER_NAME
    if not index_path.exists():
        return None, None, None
    try:
        fname = index_path / "index.faiss"
        key = str(fname.resolve())
        sig = _signature(index_path)
        if sig[0] is None:
            return None, None, None
        use_shards = _want_sharded(sharded)
        with _cache_lock:
            hit = _cache.get(key)
            if hit is not None and hit[0] == sig and hasattr(hit[1], "local") == use_shards:
                _cache.move_to_end(key)
                return hit[1], hit[2], hit[3]
        try:
            index = _read_resident(fname, use_shards)
        except _lib.EvsError as e:
            if e.code != _lib.EVS_ENOMEM:
                raise
            evict_index()  # HBM is full of other folders' indexes: drop them and try once more
            index = _read_resident(fname, use_shards)
        with open(index_path / "paths.pkl", "rb") as f:
            image_paths = pickle.load(f)
        image_metadata = None
        metadata_file = index_path / "metadata.pkl"
        if metadata_file.exists():
            try:
                with open(metadata_file, "rb") as f:
                    image_metadata = pickle.load(f)
            except Exception:  # noqa: BLE001 - backwards compatible, as the reference
                image_metadata = None
        _cache_put(key, sig, index, image_paths, image_metadata)
        return index, image_paths, image_metadata
    except Exception:  # noqa: BLE001 - the reference swallows everything here
        return None, None, None


def evict_index(folder_path=None) -> None:
    """Drop one folder's resident index (or all of them) and free its HBM."""
    with _cache_lock:
        if folder_path is None:
            load_stats["evictions"] += len(_cache)
            _cache.clear()
        else:
            key = str((Path(folder_path) / config.INDEX_FOLDER_NAME / "index.faiss").resolve())
            _cache.pop(key, None)


def clamp_limit(limit: Any) -> int:
    """The handlers' limit rule (oldapp.py:1985-1990, :2065-2070): int in [MIN, MAX] else DEFAULT."""
    try:
        limit = int(limit)
        if limit < config.MIN_RESULTS or limit > config.MAX_RESULTS:
            limit = config.DEFAULT_RESULTS
    except (ValueError, TypeError):
        limit = config.DEFAULT_RESULTS
    return limit


def _collect(index, image_paths, image_metadata, embedding, limit, sort_by) -> List[dict]:
    """Search + the handlers' post-processing (oldapp.py:2002-2045) minus thumbnails."""
    k = min(limit, len(image_paths))
    if k == 0:
        return []
    similarities, indices = index.search(np.asarray(embedding).reshape(1, -1), k)
    results = []
    for idx, sim in zip(indices[0], similarities[0]):
        if idx >= 0 and idx < len(image_paths):
            img_path = image_paths[idx]
            metadata_info = {}
            if image_metadata and idx < len(image_metadata):
                meta = image_metadata[idx]
                metadata_info = {"mtime": meta.get("mtime", 0), "size": meta.get("size", 0)}
            results.append({"path": img_path, "filename": os.path.basename(img_path), "similarity": float(sim),
                            "metadata": metadata_info})
    if sort_by == "time" and image_metadata:
        results.sort(key=lambda x: x["metadata"].get("mtime", 0), reverse=True)
    return results


def search_text(folder, query: str, encoder, limit=10, sort_by: str = "similarity") -> Optional[List[dict]]:
    """Body of ``POST /search`` (oldapp.py:1972-2053).  ``None`` = folder not indexed."""
    limit = clamp_limit(limit)
    index, image_paths, image_metadata = load_index(folder)
    if index is None:
        return None
    return _collect(index, image_paths, image_metadata, encoder.get_text_embedding(query), limit, sort_by)


def search_image(folder, image, encoder, limit=12, sort_by: str = "similarity") -> Optional[List[dict]]:
    """Body of ``POST /search_by_image`` (oldapp.py:2055-2157).  ``image`` is a path or a PIL image."""
    limit = clamp_limit(limit)
    index, image_paths, image_metadata = load_index(folder)
    if index is None:
        return None
    if isinstance(image, (str, os.PathLike)):
        emb = encoder.get_image_embedding(image)
    else:
        emb = encoder.get_image_embedding_from_pil(image)
    return _collect(index, image_paths, image_metadata, emb, limit, sort_by)
