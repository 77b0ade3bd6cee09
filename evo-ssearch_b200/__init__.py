"""evo-ssearch_b200 -- B200-native (sm_100a) exact inner-product top-k search for evo-ssearch.

Drop-in for the reference's similarity-search hot path only (SURVEY.md section 8): the faiss symbols
``oldapp.py`` uses (``IndexFlatIP``, ``add``, ``search``, ``write_index``, ``read_index``), the index lifecycle
functions (``create_index``, ``save_index``, ``load_index``) and the search entry points, over the same
``.clip_index`` files.  All arithmetic runs in hand-written CUDA kernels behind the C ABI of
``libevs.so`` (``include/evs.h``); there is no CPU fallback.

Importable as ``evo_ssearch_b200`` (shim at the repo root) or, faiss-style, ``import evs as faiss``.
"""
import os as _os

from ._lib import EvsError, device_count, get_option, kernel_launches, set_option  # noqa: F401
from .config import Config, config  # noqa: F401
from .index import (METRIC_INNER_PRODUCT, METRIC_L2, IndexFlatIP, PeerExchange, merge_partials,  # noqa: F401
                    normalize_L2, read_index, write_index)
from .lifecycle import (clamp_limit, create_index, evict_index, load_index, save_index, search_image,  # noqa: F401
                        search_text, update_index)
from .sharded import ShardedIndexFlatIP, shard_bounds  # noqa: F401

# ``EVS_MAX_K`` raises the largest k a search accepts (option "max_k", up to 2048; default 112), read once at import like
# ``EVS_STORAGE`` and ``EVS_DEVICE``: an application that lets its users ask for more results (``EVOSSEARCH_MAX_RESULTS``)
# sets it beside that limit.
if _os.environ.get("EVS_MAX_K"):
    set_option("max_k", int(_os.environ["EVS_MAX_K"]))

__all__ = [
    "IndexFlatIP", "PeerExchange", "read_index", "write_index", "normalize_L2", "merge_partials", "METRIC_INNER_PRODUCT", "METRIC_L2",
    "create_index", "update_index", "save_index", "load_index", "evict_index", "search_text", "search_image", "clamp_limit",
    "ShardedIndexFlatIP", "shard_bounds", "config", "Config", "EvsError", "device_count", "set_option",
    "get_option", "kernel_launches",
]
