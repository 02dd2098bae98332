"""Recorded conversations with the reference implementation, so that the parity tests run without it.

Every test that compares against the reference talks to it through a ``Ref`` handle (the ``ref_cpu``, ``ref_cuda``,
``ref_funcs`` and ``ref_samplers`` fixtures).  With ``RLB_RECORD_TAPES=DIR`` set, the handle forwards each operation --
attribute read or write, call, item read or write -- to the live reference and appends it to a tape: what was asked (a
SHA-256 digest of the arguments) and what came back (plain values in full; reference objects as new handles; a raised
exception by type and message).  Without it the handle plays the committed tape back
(``tests/golden/ref_tapes/<module>/<test function>.npz``, one per test function): every operation must match the recorded one, argument digest included, and returns what the reference returned.
A test whose inputs drift from the recording fails instead of comparing against stale answers.

``run(handle, fn, *args)`` records ``fn(<live reference>, *args)`` as one operation, for helpers that need the live
objects themselves (e.g. to intercept the random draws the reference makes).
"""
from __future__ import annotations

import builtins
import hashlib
import json
import os
from pathlib import Path

import numpy as np
import torch

TAPES = Path(__file__).resolve().parent / "golden" / "ref_tapes"


def record_dir() -> Path | None:
    d = os.environ.get("RLB_RECORD_TAPES")
    return Path(d) if d else None


def tape_file(directory: Path, module: str, function: str) -> Path:
    return directory / module / f"{function}.npz"


# --------------------------------------------------------------------------------------------- argument digests
def _feed(h, x) -> None:
    if isinstance(x, Ref):
        h.update(b"R" + str(x._id).encode())
    elif isinstance(x, torch.Tensor):
        a = x.detach().cpu().contiguous()
        h.update(f"T{a.dtype}{tuple(a.shape)}".encode())
        h.update(a.numpy().tobytes())
    elif isinstance(x, (np.ndarray, np.generic)):
        a = np.ascontiguousarray(x)
        h.update(f"A{a.dtype.str}{a.shape}".encode() + a.tobytes())
    elif x is None or isinstance(x, (bool, int, float, str, range, slice, torch.dtype, torch.device, torch.Size)):
        h.update(f"{type(x).__name__}:{x!r}".encode())
    elif isinstance(x, (tuple, list)):
        h.update(f"{type(x).__name__}{len(x)}(".encode())
        for y in x:
            _feed(h, y)
        h.update(b")")
    elif isinstance(x, dict):
        h.update(f"D{len(x)}(".encode())
        for k, v in x.items():
            _feed(h, k)
            _feed(h, v)
        h.update(b")")
    elif isinstance(x, torch.Generator):
        h.update(f"G{x.device}".encode())
        _feed(h, x.get_state())
    else:
        raise TypeError(f"cannot digest an argument of type {type(x).__name__}")


def digest(*args, **kwargs) -> str:
    h = hashlib.sha256()
    _feed(h, args)
    _feed(h, kwargs)
    return h.hexdigest()[:16]


# --------------------------------------------------------------------------------------------- tapes
class Tape:
    """The operations of one test, in order.  ``events is None`` records; otherwise plays back."""

    def __init__(self, name: str, events: list | None = None, blob: bytes = b"", layouts: dict | None = None):
        self.name = name
        self.recording = events is None
        self.events = [] if events is None else events
        self.blob = bytearray(blob)   # every stored array, packed end to end
        self.layouts = {} if layouts is None else layouts     # array key -> where and how it is stored
        self.pos = 0
        self.live = {}          # handle id -> live object (recording)
        self.n_obj = 0
        self._last = {}         # (dtype, shape) -> key of the last array stored with that layout

    # -- values ---------------------------------------------------------------------------------------------------
    def _pack(self, a: np.ndarray) -> dict:
        """Append an array to the blob: booleans as bits, integers in the narrowest type that holds them."""
        spec = {"dt": a.dtype.str, "sh": list(a.shape), "at": len(self.blob)}
        if a.dtype == bool:
            a, spec["bits"] = np.packbits(a.reshape(-1)), True
        elif a.dtype.kind in "iu" and a.size:
            for t in (np.int8, np.int16, np.int32):
                if np.iinfo(t).min <= a.min() and a.max() <= np.iinfo(t).max:
                    a, spec["as"] = a.astype(t), np.dtype(t).str
                    break
        self.blob += np.ascontiguousarray(a).tobytes()
        return spec

    def _unpack(self, spec: dict) -> np.ndarray:
        dt, shape, at = np.dtype(spec["dt"]), tuple(spec["sh"]), spec["at"]
        n = int(np.prod(shape, dtype=np.int64))
        if spec.get("bits"):
            raw = np.frombuffer(self.blob, np.uint8, (n + 7) // 8, at)
            return np.unpackbits(raw, count=n).astype(bool).reshape(shape)
        st = np.dtype(spec.get("as", dt))
        return np.frombuffer(self.blob, st, n, at).astype(dt).reshape(shape)

    def _store(self, a: np.ndarray) -> dict:
        """Store a copy.  A large array that differs from the previous one of its layout in few places is stored as
        the positions and values that differ (reference trees read back repeatedly after small write-backs)."""
        a = np.ascontiguousarray(a)
        key = str(len(self.layouts))
        layout = (a.dtype.str, a.shape)
        base = self._last.get(layout)
        self._last[layout] = key
        if base is not None and a.size >= 1024:
            flat, prev = a.reshape(-1), self._load({"a": base}).reshape(-1)
            u = np.uint8 if a.dtype == bool else f"u{a.itemsize}"
            pos = np.flatnonzero(flat.view(u) != prev.view(u))
            if pos.size * 4 < a.size:
                self.layouts[key] = {"base": base, "p": self._pack(pos), "v": self._pack(flat[pos])}
                return {"a": key}
        self.layouts[key] = self._pack(a)
        return {"a": key}

    def _load(self, ref: dict) -> np.ndarray:
        spec = self.layouts[ref["a"]]
        if "base" not in spec:
            return self._unpack(spec)
        a = self._load({"a": spec["base"]}).copy()
        a.reshape(-1)[self._unpack(spec["p"])] = self._unpack(spec["v"])
        return a

    def encode(self, v):
        if v is None or isinstance(v, (bool, int, float, str)):
            return {"v": v}
        if isinstance(v, torch.Tensor):
            return {"t": self._store(v.detach().cpu().numpy()), "dev": str(v.device)}
        if isinstance(v, np.ndarray):
            return {"n": self._store(v)}
        if isinstance(v, np.generic):
            return {"s": self._store(np.asarray(v))}
        if isinstance(v, torch.Size):
            return {"size": list(v)}
        if isinstance(v, (tuple, list)):
            return {type(v).__name__: [self.encode(x) for x in v]}
        if isinstance(v, dict):
            return {"dict": [[self.encode(k), self.encode(x)] for k, x in v.items()]}
        raise TypeError(f"{type(v).__name__} is not a plain value")

    def decode(self, e):
        if "v" in e:
            return e["v"]
        if "t" in e:
            return torch.from_numpy(self._load(e["t"]).copy()).to(e["dev"])
        if "n" in e:
            return self._load(e["n"]).copy()
        if "s" in e:
            return self._load(e["s"])[()]
        if "size" in e:
            return torch.Size(e["size"])
        if "tuple" in e:
            return tuple(self.decode(x) for x in e["tuple"])
        if "list" in e:
            return [self.decode(x) for x in e["list"]]
        if "dict" in e:
            return {_hashable(self.decode(k)): self.decode(x) for k, x in e["dict"]}
        raise ValueError(f"malformed tape entry {e}")

    # -- operations -----------------------------------------------------------------------------------------------
    def op(self, kind: str, target: Ref, name: str, live_fn, args=(), kwargs=None):
        kwargs = kwargs or {}
        d = digest(*args, **kwargs)
        if self.recording:
            try:
                out = live_fn(*_unwrap(args), **_unwrap(kwargs))
            except Exception as err:  # noqa: BLE001  -- the reference's own error is part of its behaviour
                self.events.append([kind, target._id, name, d, {"raise": [type(err).__name__, str(err)]}])
                raise
            try:
                enc = self.encode(out)
                ret = out
            except TypeError:
                self.n_obj += 1
                enc = {"obj": self.n_obj}
                self.live[self.n_obj] = out
                ret = Ref(self, self.n_obj)
            self.events.append([kind, target._id, name, d, enc])
            return ret
        if self.pos >= len(self.events):
            raise AssertionError(f"{self.name}: {kind} {name!r} goes past the end of the recorded reference tape")
        want = self.events[self.pos]
        self.pos += 1
        if want[:4] != [kind, target._id, name, d]:
            raise AssertionError(f"{self.name}: reference tape out of step at operation {self.pos}: the test now does "
                                 f"{[kind, target._id, name, d]}, the recording has {want[:4]} (inputs changed? "
                                 f"re-record with RLB_RECORD_TAPES, see tests/golden/README.md)")
        enc = want[4]
        if "raise" in enc:
            exc = getattr(builtins, enc["raise"][0], None)
            if not (isinstance(exc, type) and issubclass(exc, Exception)):
                exc = RuntimeError
            raise exc(enc["raise"][1])
        if "obj" in enc:
            return Ref(self, enc["obj"])
        return self.decode(enc)

    # -- files ----------------------------------------------------------------------------------------------------
    def dump(self) -> dict:
        return {f"{self.name}|blob": np.frombuffer(bytes(self.blob), np.uint8),
                f"{self.name}|events": np.array(json.dumps({"events": self.events, "layouts": self.layouts}))}


def _hashable(k):
    return tuple(k) if isinstance(k, list) else k


def recorder(name: str) -> Tape:
    return Tape(name)


def player(module: str, function: str, name: str) -> Tape:
    f = tape_file(TAPES, module, function)
    if not f.exists():
        raise AssertionError(f"{f.name} missing: record it with RLB_RECORD_TAPES (see tests/golden/README.md)")
    z = np.load(f)
    key = f"{name}|events"
    if key not in z.files:
        raise AssertionError(f"{name} has no recorded reference tape in {f.name} (see tests/golden/README.md)")
    meta = json.loads(str(z[key]))
    return Tape(name, meta["events"], z[f"{name}|blob"].tobytes(), meta["layouts"])


def save(directory: Path, module: str, function: str, tapes: list[Tape]) -> Path:
    """Write (or update: the tapes of other parameter sets in the file are kept) the tape file of one test function."""
    f = tape_file(directory, module, function)
    f.parent.mkdir(parents=True, exist_ok=True)
    names = {t.name for t in tapes}
    out = {}
    if f.exists():
        z = np.load(f)
        out = {k: z[k] for k in z.files if k.split("|")[0] not in names}
    for t in tapes:
        out.update(t.dump())
    np.savez_compressed(f, **out)
    return f


# --------------------------------------------------------------------------------------------- handles
class Ref:
    """A reference object as a test sees it: live behind a recording tape, or its recorded answers on playback."""

    __slots__ = ("_tape", "_id")

    def __init__(self, tape: Tape, ident):
        object.__setattr__(self, "_tape", tape)
        object.__setattr__(self, "_id", ident)

    def _live(self):
        return self._tape.live[self._id]

    def __getattr__(self, name):
        if name.startswith("__") and name.endswith("__"):
            raise AttributeError(name)
        return self._tape.op("get", self, name, lambda: getattr(self._live(), name))

    def __setattr__(self, name, value):
        self._tape.op("set", self, name, lambda v: setattr(self._live(), name, v), (value,))

    def __call__(self, *args, **kwargs):
        return self._tape.op("call", self, "", lambda *a, **k: self._live()(*a, **k), args, kwargs)

    def __getitem__(self, item):
        return self._tape.op("getitem", self, "", lambda i: self._live()[i], (item,))

    def __setitem__(self, item, value):
        def put(i, v):
            self._live()[i] = v

        self._tape.op("setitem", self, "", put, (item, value))

    def __repr__(self):
        return f"<reference object {self._id} of {self._tape.name}>"


def root(tape: Tape, ident: str, live=None) -> Ref:
    if tape.recording:
        tape.live[ident] = live
    return Ref(tape, ident)


def run(handle: Ref, fn, *args, **kwargs):
    """``fn(<the live object behind handle>, *args, **kwargs)`` recorded as one operation."""
    tape = handle._tape
    return tape.op("run", handle, fn.__qualname__, lambda *a, **k: fn(handle._live(), *a, **k), args, kwargs)


def _unwrap(x):
    if isinstance(x, Ref):
        return x._live()
    if isinstance(x, tuple):
        return tuple(_unwrap(y) for y in x)
    if isinstance(x, list):
        return [_unwrap(y) for y in x]
    if isinstance(x, dict):
        return {k: _unwrap(v) for k, v in x.items()}
    return x
