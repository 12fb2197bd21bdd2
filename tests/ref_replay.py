"""The compiled reference's answers, recorded once and replayed everywhere else.

The tests that pin this project to nanopolish call its unmodified sources compiled into oracle/_ref/libnpref.so (oracle/Makefile),
which can only be built where those sources are.  Every call such a test makes to the compiled reference is recorded here, per test,
under tests/golden/ref_calls/: the method, a digest of its arguments and what it returned.  Everywhere else the test replays the
recording: each call must be the next recorded one with the same method and the same argument digest (the test's inputs are
seeded, so they are identical from run to run), and it receives the recorded result.  Where the compiled reference is present, the
tests call it directly (tests/conftest.py).

Record (where oracle/_ref/libnpref.so is built):  NPH_RECORD_REF=tests/golden/ref_calls python -m pytest <tests>
"""
from __future__ import annotations

import hashlib
import json
import os

import numpy as np

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_calls")


def _feed(h, x):
    """a canonical byte encoding of call arguments into the hash h"""
    if isinstance(x, (np.ndarray, np.generic)):
        a = np.ascontiguousarray(x)
        h.update(f"nd{a.dtype.str}{a.shape}:".encode()); h.update(a.tobytes())
    elif isinstance(x, (bytes, bytearray)):
        h.update(b"b%d:" % len(x)); h.update(x)
    elif isinstance(x, str):
        h.update(b"s%d:" % len(x.encode())); h.update(x.encode())
    elif isinstance(x, (list, tuple)):
        h.update(b"l%d:" % len(x))
        for y in x:
            _feed(h, y)
    elif isinstance(x, dict):
        h.update(b"d%d:" % len(x))
        for k in sorted(x):
            _feed(h, k); _feed(h, x[k])
    elif x is None or isinstance(x, (bool, int, float)):
        h.update(repr(x).encode() + b";")
    else:
        raise TypeError(f"cannot digest an argument of type {type(x).__name__}")


def _digest(name, args, kwargs):
    h = hashlib.sha256()
    _feed(h, [name, list(args), kwargs])
    return h.hexdigest()[:12]            # 48 bits tell apart the arguments of one test's calls


def _pack(x, arrays):
    """JSON-able description of a result; its arrays go to `arrays`"""
    if isinstance(x, (np.ndarray, np.generic)):
        arrays.append(np.asarray(x))
        return {"nd" if isinstance(x, np.ndarray) else "np": len(arrays) - 1}
    if isinstance(x, str):
        return {"str": x}
    if isinstance(x, bytes):
        return {"bytes": x.hex()}
    if isinstance(x, (tuple, list)):
        return {type(x).__name__: [_pack(y, arrays) for y in x]}
    if isinstance(x, frozenset):
        return {"frozenset": sorted(x)}
    if isinstance(x, dict):
        return {"dict": [[_pack(k, arrays), _pack(v, arrays)] for k, v in x.items()]}
    if x is None or isinstance(x, (bool, int, float)):
        return {"py": x}            # json writes floats with repr: they read back bit for bit
    raise TypeError(f"cannot record a result of type {type(x).__name__}")


def _unpack(d, arrays):
    (kind, v), = d.items()
    if kind == "nd":
        return arrays[v].copy()
    if kind == "np":
        return arrays[v][()]
    if kind == "bytes":
        return bytes.fromhex(v)
    if kind in ("tuple", "list"):
        return (tuple if kind == "tuple" else list)(_unpack(y, arrays) for y in v)
    if kind == "frozenset":
        return frozenset(v)
    if kind == "dict":
        return {_unpack(k, arrays): _unpack(y, arrays) for k, y in v}
    return v


class ReplayedRef:
    """Stands in for oracle.oracle_py.RefOracle inside one test (see the module docstring)."""

    def __init__(self, node, live=None, record_dir=None):
        """node: the running test; live: the compiled reference, when recording into record_dir"""
        test = node.originalname if hasattr(node, "originalname") else node.name
        self._file = f"{node.module.__name__.rsplit('.', 1)[-1]}.{test}.npz"
        self._case = node.callspec.id if hasattr(node, "callspec") else "-"
        self._live, self._record_dir = live, record_dir
        self._calls, self._arrays, self._next = [], [], 0
        self._loaded = record_dir is not None

    def _load(self):
        path = os.path.join(GOLD, self._file)
        if not os.path.exists(path):
            raise FileNotFoundError(f"{path}: no recording of the compiled reference for this test")
        with np.load(path) as z:
            self._calls = json.loads(z[self._case + "|calls"].tobytes())
            self._arrays = [z[f"{self._case}|{i}"] for i in range(len(z.files)) if f"{self._case}|{i}" in z.files]
        self._loaded = True

    def __getattr__(self, name):
        if name.startswith("_"):
            raise AttributeError(name)

        def call(*args, **kwargs):
            digest = _digest(name, args, kwargs)
            if self._record_dir is not None:
                result = getattr(self._live, name)(*args, **kwargs)
                self._calls.append({"method": name, "args": digest, "result": _pack(result, self._arrays)})
                return result
            if not self._loaded:
                self._load()
            assert self._next < len(self._calls), f"{name}: the recording of {self._file} [{self._case}] has no more calls"
            rec = self._calls[self._next]
            self._next += 1
            assert rec["method"] == name and rec["args"] == digest, \
                f"call {self._next} of {self._file} [{self._case}]: {name} with other arguments than recorded ({rec['method']})"
            return _unpack(rec["result"], self._arrays)
        return call

    def finish(self):
        """write the recording of this test case (merged into the test's file next to its other parameter sets)"""
        if self._record_dir is None or not self._calls:
            return
        os.makedirs(self._record_dir, exist_ok=True)
        path = os.path.join(self._record_dir, self._file)
        keep = {}
        if os.path.exists(path):
            with np.load(path) as z:
                keep = {k: z[k] for k in z.files if not k.startswith(self._case + "|")}
        keep[self._case + "|calls"] = np.frombuffer(json.dumps(self._calls).encode(), np.uint8)
        keep.update({f"{self._case}|{i}": a for i, a in enumerate(self._arrays)})
        np.savez_compressed(path, **keep)
