"""The reference's side of the tests that compare with the original BindsNET, stored with the tests.

Such a test asks ``stored(name, compute)`` for each value it compares against.  Normally the value comes from
``tests/golden/live/<test module>.npz``, so the comparison runs wherever the suite does.  With
``BINDSNET_B200_RECORD_REFERENCE=1`` set and the reference importable (``cases.namespace("reference")``: a checkout
of the original package named by ``BINDSNET_REFERENCE``, or an install under baseline/_ref),
``compute()`` runs the reference instead, the test compares against that, and every value the run asked for is
written back to the module's file when the process exits.  Record whole modules, for instance

    BINDSNET_REFERENCE=/path/to/bindsnet-checkout BINDSNET_B200_RECORD_REFERENCE=1 python -m pytest tests/test_srm0_live.py

since a module's file holds exactly what the recording run asked for.

Values are tensors, numpy arrays, Python scalars, strings, ``None`` and lists, tuples and dicts of them; tensors
and arrays keep their dtype and shape, floats their exact value.
"""
from __future__ import annotations

import atexit
import json
import os

import numpy as np
import torch

import cases

DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "live")
RECORDING = os.environ.get("BINDSNET_B200_RECORD_REFERENCE") == "1"
#: the live reference's namespace while recording, else None
REF = cases.namespace("reference") if RECORDING else None

_recorded = {}   # module -> {key: value}
_loaded = {}     # module -> (spec, arrays)


def _current_test():
    """(module, test id) of the running test, e.g. ("test_srm0_live", "test_srm0_window_matches_the_live_reference[None]")."""
    node = os.environ["PYTEST_CURRENT_TEST"].rsplit(" (", 1)[0]
    path, name = node.split("::", 1)
    return os.path.splitext(os.path.basename(path))[0], name


class _Buffers:
    """Arrays being stored: one flat buffer per dtype, each distinct array once (the n-gram dictionaries hold hundreds
    of tiny tensors, the monitor recordings repeat whole arrays)."""

    def __init__(self):
        self.chunks, self.size, self.seen = {}, {}, {}

    def add(self, a: np.ndarray):
        a = np.ascontiguousarray(a)
        key = (a.dtype.name, a.shape, a.tobytes())
        if key not in self.seen:
            self.seen[key] = self.size.get(a.dtype.name, 0)
            self.chunks.setdefault(a.dtype.name, []).append(a.reshape(-1))
            self.size[a.dtype.name] = self.seen[key] + a.size
        return [a.dtype.name, self.seen[key], list(a.shape)]

    def arrays(self):
        """The buffers as stored: a multi-byte buffer as its byte planes ([itemsize, n] uint8), which compress better."""
        out = {}
        for dtype, chunks in self.chunks.items():
            a = np.concatenate(chunks)
            out[dtype] = a.view(np.uint8).reshape(-1, a.itemsize).T.copy() if a.itemsize > 1 else a
        return out


def _buffers(stored: dict) -> dict:
    """Inverse of ``_Buffers.arrays``."""
    return {dtype: (a.T.copy().view(np.dtype(dtype)).reshape(-1) if a.ndim == 2 else a) for dtype, a in stored.items()}


def _pack(value, buffers: _Buffers):
    if isinstance(value, torch.Tensor):
        return {"tensor": buffers.add(value.detach().cpu().numpy())}
    if isinstance(value, np.ndarray):
        return {"array": buffers.add(value)}
    if isinstance(value, (list, tuple)):
        return {"list" if isinstance(value, list) else "tuple": [_pack(v, buffers) for v in value]}
    if isinstance(value, dict):
        return {"dict": [[_pack(k, buffers), _pack(v, buffers)] for k, v in value.items()]}
    if isinstance(value, np.generic):
        value = value.item()
    if value is None or isinstance(value, (bool, int, float, str)):
        return {"value": value}
    raise TypeError(f"cannot store a {type(value).__name__}")


def _unpack(spec, arrays):
    (kind, body), = spec.items()
    if kind in ("tensor", "array"):
        dtype, offset, shape = body
        a = arrays[dtype][offset:offset + int(np.prod(shape))].reshape(shape).copy()
        return torch.from_numpy(a) if kind == "tensor" else a
    if kind in ("list", "tuple"):
        items = [_unpack(s, arrays) for s in body]
        return items if kind == "list" else tuple(items)
    if kind == "dict":
        return {_unpack(k, arrays): _unpack(v, arrays) for k, v in body}
    return body


def _save():
    for module, values in _recorded.items():
        buffers = _Buffers()
        spec = {key: _pack(value, buffers) for key, value in values.items()}
        os.makedirs(DIR, exist_ok=True)
        np.savez_compressed(os.path.join(DIR, f"{module}.npz"), spec=np.frombuffer(json.dumps(spec).encode(), dtype=np.uint8),
                            **buffers.arrays())


if RECORDING:
    atexit.register(_save)


def stored(name: str, compute):
    """The reference's value ``name`` for the running test: ``compute()`` while recording, else the stored value."""
    module, test = _current_test()
    key = f"{test}/{name}"
    if RECORDING:
        value = compute()
        _recorded.setdefault(module, {})[key] = value
        buffers = _Buffers()
        return _unpack(_pack(value, buffers), _buffers(buffers.arrays()))   # exactly what the stored file will give back
    if module not in _loaded:
        z = np.load(os.path.join(DIR, f"{module}.npz"))
        _loaded[module] = (json.loads(bytes(z["spec"]).decode()), _buffers({k: z[k] for k in z.files if k != "spec"}))
    spec, arrays = _loaded[module]
    if key not in spec:
        raise KeyError(f"{module}: no stored reference value {key!r}; record it (see tests/golden/live.py)")
    return _unpack(spec[key], arrays)
