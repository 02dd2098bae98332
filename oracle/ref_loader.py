"""TEST INFRASTRUCTURE -- loaders for the real reference (never imported by the product).

``reference_ext(kind)``      the UNMODIFIED reference segment tree compiled by build_ref.py into
                             oracle/_ref/{cpu,cuda}/_torchrl.so (travels to the GPU box).
``reference_functionals()``  the reference's Python value functionals imported by path under a
                             ten-line ``tensordict`` shim, from the torchrl source checkout named by
                             $RLB_REFERENCE_ROOT (None when it is not set).
"""
from __future__ import annotations

import importlib.util
import os
import sys
import types
from pathlib import Path

_REF_DIR = Path(__file__).resolve().parent / "_ref"
_EXT = {}
_FUNCS = None


def reference_ext(kind: str = "cpu"):
    """Returns the compiled reference module (SumSegmentTreeFp32, ... [CudaSumSegmentTreeFp32, ...]) or None."""
    if kind in _EXT:
        return _EXT[kind]
    so = _REF_DIR / kind / "_torchrl.so"
    if not so.exists():
        try:
            from .build_ref import build

            build(with_cuda=(kind == "cuda"))
        except Exception:
            _EXT[kind] = None
            return None
    import torch  # noqa: F401  (libtorch symbols must be loaded first)

    name = "_torchrl"
    # both variants register the pybind module `_torchrl`; only one can live in a process
    if name in sys.modules and getattr(sys.modules[name], "__file__", None) != str(so):
        other = sys.modules[name]
        _EXT[kind] = other if (kind == "cpu" or hasattr(other, "CudaSumSegmentTreeFp32")) else None
        return _EXT[kind]
    spec = importlib.util.spec_from_file_location(name, so)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    sys.modules[name] = mod
    _EXT[kind] = mod
    return mod


def reference_trees(kind: str = "cpu"):
    """tree_factory for OraclePrioritizedSampler backed by the compiled reference trees."""
    ext = reference_ext(kind)
    if ext is None:
        return None
    return lambda size, is_min: (ext.MinSegmentTreeFp32 if is_min else ext.SumSegmentTreeFp32)(size)


def reference_root() -> Path | None:
    """The reference's source checkout: $RLB_REFERENCE_ROOT, or None when it is not set."""
    root = os.environ.get("RLB_REFERENCE_ROOT")
    return Path(root) if root else None


def reference_functionals(root: str | None = None):
    """Import torchrl/objectives/value/{utils,functional}.py by path (SURVEY.md Appendix A.2)."""
    global _FUNCS
    if _FUNCS is not None:
        return _FUNCS
    root = root or reference_root()
    if root is None:
        return None
    base = Path(root) / "torchrl" / "objectives" / "value"
    if not base.exists():
        return None
    td = sys.modules.setdefault("tensordict", types.ModuleType("tensordict"))
    tdu = sys.modules.setdefault("tensordict.utils", types.ModuleType("tensordict.utils"))
    if not hasattr(td, "TensorDictBase") or not hasattr(tdu, "expand_right"):

        class TensorDictBase:  # isinstance() target only
            pass

        def expand_right(t, shape):
            while t.ndim < len(shape):
                t = t.unsqueeze(-1)
            return t.expand(shape)

        td.TensorDictBase, tdu.expand_right, td.utils = TensorDictBase, expand_right, tdu
    for n in ("torchrl", "torchrl.objectives", "torchrl.objectives.value"):
        if n not in sys.modules:
            m = types.ModuleType(n)
            m.__path__ = []
            sys.modules[n] = m

    def _load(name, path):
        spec = importlib.util.spec_from_file_location(name, path)
        m = importlib.util.module_from_spec(spec)
        sys.modules[name] = m
        spec.loader.exec_module(m)
        return m

    _load("torchrl.objectives.value.utils", base / "utils.py")
    _FUNCS = _load("torchrl.objectives.value.functional", base / "functional.py")
    return _FUNCS


# ----------------------------------------------------------------------------------------------------------
# the reference's samplers module, UNMODIFIED, imported by path
# ----------------------------------------------------------------------------------------------------------
_SAMPLERS = None


class StubTD:
    """The few TensorDict operations torchrl/data/replay_buffers/samplers.py performs on storage contents: nested-key
    ``get`` / ``[key]``, row indexing, ``keys(include_nested=True)``.  Flat dict keyed by tuples."""

    def __init__(self, data: dict):
        self._d = {(k,) if isinstance(k, str) else tuple(k): v for k, v in data.items()}

    @staticmethod
    def _k(key):
        return (key,) if isinstance(key, str) else tuple(key)

    def keys(self, include_nested=False, leaves_only=False):
        return [k[0] if len(k) == 1 else k for k in self._d]

    def get(self, key, default=...):
        k = self._k(key)
        if k in self._d:
            return self._d[k]
        if default is ...:
            raise KeyError(key)
        return default

    def __getitem__(self, item):
        if isinstance(item, str) or (isinstance(item, tuple) and item and all(isinstance(i, str) for i in item)):
            return self.get(item)
        return StubTD({k: v[item] for k, v in self._d.items()})


def reference_samplers(root: str | None = None):
    """Import torchrl/data/replay_buffers/samplers.py by path, with stub modules for what it imports at module level
    (tensordict, pyvers, torchrl._utils, the storages module) and the COMPILED reference trees as ``torchrl._torchrl``.
    Returns a namespace with the module (``.mod``) and ``make_storage(data: dict, length, max_size, last_cursor)`` that
    builds the minimal ``TensorStorage`` the samplers need.  None when no reference checkout is given.
    """
    global _SAMPLERS
    if _SAMPLERS is not None:
        return _SAMPLERS
    root = root or reference_root()
    if root is None:
        return None
    path = Path(root) / "torchrl" / "data" / "replay_buffers" / "samplers.py"
    if not path.exists():
        return None
    import logging

    import torch

    def mod(name, **attrs):
        m = sys.modules.get(name)
        if m is None:
            m = types.ModuleType(name)
            m.__path__ = []
            sys.modules[name] = m
        for k, v in attrs.items():
            if not hasattr(m, k):
                setattr(m, k, v)
        return m

    def implement_for(*a, **k):          # pyvers: version-gated overloads; the last definition wins, as at import
        return lambda fn: fn

    def _replace_last(key, new):         # torchrl/_utils.py: replace the last element of a (nested) key
        return new if isinstance(key, str) else (*key[:-1], new)

    class Storage:                       # isinstance() targets + the attributes the samplers read
        ndim = 1

    class StorageEnsemble(Storage):
        pass

    class TensorStorage(Storage):
        """``columns`` > 0: an ndim=2 storage whose leaves are [max_size, columns, ...] (time along dim 0); ``length`` and
        ``max_size`` then count ROWS, as ``_len_along_dim0`` does in the reference (storages.py:828-863)."""

        def __init__(self, data: dict, length: int, max_size: int, last_cursor=None, columns: int = 0):
            self._storage = StubTD(data)
            self._rows, self._max_rows, self._last_cursor = int(length), int(max_size), last_cursor
            self._columns = int(columns)
            self.ndim = 2 if columns else 1
            self.max_size = self._max_rows * max(1, self._columns)
            self._len = self._rows * max(1, self._columns)
            self.device = next(iter(data.values())).device

        def __len__(self):
            return self._len

        @property
        def _is_full(self):
            return self._len == self.max_size

        @property
        def _total_shape(self):
            return torch.Size([self._max_rows] + ([self._columns] if self._columns else []))

        @property
        def _len_along_dim0(self):
            return self._rows

        @property
        def shape(self):          # truncated to the fill level, as TensorStorage.shape (storages.py:856-863)
            return torch.Size([self._max_rows if self._is_full else self._rows] + ([self._columns] if self._columns else []))

        def __getitem__(self, index):
            if isinstance(index, slice) and index == slice(None):
                return StubTD({k: v[: self._rows] for k, v in self._storage._d.items()})
            if isinstance(index, tuple) and len(index) == 1:
                index = index[0]
            return self._storage[index]

    mod("pyvers", implement_for=implement_for)
    td = mod("tensordict", is_tensor_collection=lambda x: isinstance(x, StubTD), MemoryMappedTensor=type("MMT", (), {}),
             TensorDict=StubTD)
    tdu = mod("tensordict.utils", NestedKey=object)
    td.utils = tdu
    for n in ("torchrl", "torchrl.data", "torchrl.data.replay_buffers"):
        mod(n)
    mod("torchrl._extension", EXTENSION_WARNING="")
    mod("torchrl._utils", _replace_last=_replace_last, logger=logging.getLogger("torchrl"), rl_warnings=lambda: False)
    mod("torchrl.data.replay_buffers.storages", Storage=Storage, StorageEnsemble=StorageEnsemble,
        TensorStorage=TensorStorage)
    mod("torchrl.data.replay_buffers.utils", _auto_device=lambda: torch.device("cpu"),
        _is_int=lambda i: isinstance(i, int) or (isinstance(i, torch.Tensor) and i.ndim == 0 and not i.is_floating_point()),
        unravel_index=lambda index, shape: torch.unravel_index(index, shape))
    ext = reference_ext("cpu")
    if ext is not None:
        sys.modules["torchrl._torchrl"] = ext
    spec = importlib.util.spec_from_file_location("torchrl.data.replay_buffers.samplers", path)
    m = importlib.util.module_from_spec(spec)
    sys.modules["torchrl.data.replay_buffers.samplers"] = m
    spec.loader.exec_module(m)
    _SAMPLERS = types.SimpleNamespace(mod=m, make_storage=TensorStorage, StubTD=StubTD)
    return _SAMPLERS
