"""Generate the golden fixtures by running the LIVE reference (the original package, found as
``cases.namespace("reference")`` finds it) under fixed seeds:

    BINDSNET_REFERENCE=/path/to/bindsnet-checkout python tests/golden/gen_golden.py [case ...]

For every case of ``cases.py`` this writes ``tests/golden/<case>.npz`` holding the exact input
spikes (bit-packed), the final state of every layer and connection after ``network.run`` and
the per-neuron spike counts.  The reference's only random draw on the path —
``torch.multinomial`` in ``DiehlAndCookNodes.forward`` (nodes.py:1097-1105) — is replaced by the
shared tie-break hash of include/snn_b200.h (same distribution: uniform over the candidates),
so that the oracle and the kernels can reproduce the run.
"""
from __future__ import annotations

import hashlib
import json
import os
import sys
import time

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", ".."))
sys.path.insert(0, HERE)

import cases  # noqa: E402


def _fmix32(h: np.ndarray) -> np.ndarray:
    h = h.astype(np.uint64)
    h ^= h >> np.uint64(16); h = (h * np.uint64(0x85EBCA6B)) & np.uint64(0xFFFFFFFF)
    h ^= h >> np.uint64(13); h = (h * np.uint64(0xC2B2AE35)) & np.uint64(0xFFFFFFFF)
    h ^= h >> np.uint64(16)
    return h


def one_spike_winner(seed: int, t: int, layer: int, b: int, cand_js: np.ndarray) -> int:
    """arg-max of snn_one_spike_key over the candidate indices (vectorised)."""
    M = np.uint64(0xFFFFFFFF)
    h = _fmix32(np.array([(seed ^ ((0x9E3779B9 * (t + 1)) & 0xFFFFFFFF)) & 0xFFFFFFFF], dtype=np.uint64))
    h = _fmix32((h + np.uint64((0x85EBCA6B * (layer + 1)) & 0xFFFFFFFF) + np.uint64(b)) & M)
    j = cand_js.astype(np.uint64)
    h = _fmix32((h ^ ((np.uint64(0xC2B2AE35) * (j + np.uint64(1))) & M)) & M)
    key = ((h | np.uint64(0x80000000)) << np.uint64(32)) | j
    return int(cand_js[int(np.argmax(key))])


class OneSpikePatch:
    """Replaces torch.multinomial while the reference runs; tracks (t, layer, sample)."""

    def __init__(self, net, seed: int):
        self.net, self.seed = net, seed
        self.layer_ids = {id(l): i for i, l in enumerate(net.layers.values())}
        self.current = None
        self.steps = {}

    def __enter__(self):
        self._orig = torch.multinomial
        self._wrapped = []
        for layer in self.net.layers.values():
            if type(layer).__name__ == "DiehlAndCookNodes":
                orig_forward = layer.forward
                self.steps[id(layer)] = 0

                def fwd(x, _layer=layer, _orig=orig_forward):
                    self.current = _layer
                    _orig(x)
                    self.steps[id(_layer)] += 1
                    self.current = None

                layer.forward = fwd
                self._wrapped.append(layer)

        def multinomial(probs, num_samples, *a, **k):
            layer = self.current
            assert layer is not None and num_samples == 1
            B = layer.batch_size
            rows = layer.s.view(B, -1).any(1).nonzero().flatten().tolist()
            assert len(rows) == probs.shape[0]
            t = self.steps[id(layer)]
            lid = self.layer_ids[id(layer)]
            out = []
            for r, b in enumerate(rows):
                js = probs[r].nonzero().flatten().numpy()
                out.append(one_spike_winner(self.seed, t, lid, b, js))
            return torch.tensor(out, dtype=torch.long).view(-1, 1)

        torch.multinomial = multinomial
        return self

    def __exit__(self, *exc):
        torch.multinomial = self._orig
        for layer in self._wrapped:
            del layer.forward
        return False


def pack(x: torch.Tensor) -> np.ndarray:
    return np.packbits(x.numpy().astype(np.uint8).reshape(-1))


def conn_weight(conn) -> torch.Tensor:
    return conn.w if hasattr(conn, "w") and not hasattr(conn, "pipeline") else conn.pipeline[0].value


def patch_reference_conv_mstdp(ns) -> None:
    """SURVEY.md §0.8 / §8c: ``MSTDP._conv2d_connection_update`` allocates a per-sample eligibility
    ``[B, *w.shape]`` (learning.py:1958-1961) and sums ``reward * eligibility`` over dim 0 (:1973-1974), but its
    last line views the new eligibility as ``w.size()`` (:2013) — that raises for B > 1 and, for B = 1, makes
    the next step sum over the OUTPUT CHANNELS instead of the batch.  The goldens are produced by the
    reference's own code with that one view taken per sample (the source is re-executed from
    the reference's own source at run time, nothing is copied)."""
    import inspect
    import textwrap

    L = ns.learning
    if getattr(L.MSTDP, "_b200_patched", False):
        return
    src = textwrap.dedent(inspect.getsource(L.MSTDP._conv2d_connection_update))
    bad = "self.eligibility = self.eligibility.view(self.connection.w.size())"
    assert bad in src and "super().update()" in src
    src = src.replace(bad, "self.eligibility = self.eligibility.view(batch_size, *self.connection.w.size())")
    src = src.replace("super().update()", "LearningRule.update(self)")  # zero-arg super() has no __class__ cell under exec
    g = dict(vars(sys.modules[L.MSTDP.__module__]))
    exec(src, g)
    L.MSTDP._conv2d_connection_update = g["_conv2d_connection_update"]
    L.MSTDP._b200_patched = True


def generate(name: str) -> None:
    ns = cases.namespace("reference")
    patch_reference_conv_mstdp(ns)
    torch.manual_seed(1234)
    net, inputs, kw, T = cases.CASES[name](ns)
    w0 = {f"{s}->{t}": conn_weight(c).detach().clone() for (s, t), c in net.connections.items()}
    for lname, layer in net.layers.items():
        net.add_monitor(ns.monitors.Monitor(layer, ["s"], time=T), f"mon_{lname}")
    t0 = time.time()
    with OneSpikePatch(net, cases.ONE_SPIKE_SEED):
        net.run(inputs={k: v.clone() for k, v in inputs.items()}, time=T, **kw)
    wall = time.time() - t0

    out = {}
    meta = {"case": name, "T": T, "seed": cases.ONE_SPIKE_SEED, "ref_wall_s": wall,
            "torch": torch.__version__, "threads": torch.get_num_threads(), "layers": {}, "conns": {}, "inputs": {}}
    for k, v in inputs.items():
        if v.dtype.is_floating_point and not bool(((v == 0) | (v == 1)).all()):
            out[f"inf/{k}"] = v.float().numpy()   # analog input current: stored as is
        else:
            out[f"in/{k}"] = pack(v)
        meta["inputs"][k] = list(v.shape)
    for lname, layer in net.layers.items():
        B = layer.s.shape[0]
        raster = net.monitors[f"mon_{lname}"].get("s").reshape(T, B, -1)
        out[f"L/{lname}/count"] = raster.sum(dim=(0, 1)).to(torch.int32).numpy()
        out[f"L/{lname}/count_b"] = raster.sum(dim=(0, 2)).to(torch.int32).numpy()
        out[f"L/{lname}/s"] = np.asarray(layer.s.reshape(B, -1).to(torch.uint8).numpy())
        for var in ("v", "refrac_count", "x", "theta", "summed", "i"):
            val = getattr(layer, var, None)
            if isinstance(val, torch.Tensor) and val.numel() > 0:
                out[f"L/{lname}/{var}"] = val.detach().reshape(-1 if var == "theta" else (B, -1)).float().numpy() \
                    if var != "theta" else val.detach().float().reshape(-1).numpy()
        meta["layers"][lname] = {"n": layer.n, "B": B, "spikes": int(raster.sum())}
    for (s, t), conn in net.connections.items():
        key = f"{s}->{t}"
        w = conn_weight(conn).detach().float()
        meta["conns"][key] = {
            "shape": list(w.shape),
            "w0_sha256": hashlib.sha256(w0[key].numpy().tobytes()).hexdigest(),
            "w_sha256": hashlib.sha256(w.numpy().tobytes()).hexdigest(),
            "w_sum": float(w.double().sum()), "w_sqsum": float((w.double() ** 2).sum()),
        }
        if name in cases.LARGE:
            out[f"C/{key}/w_rows8"] = w[::8].numpy()
            out[f"C/{key}/w_colsum"] = w.double().sum(0).numpy()
        else:
            out[f"C/{key}/w"] = w.numpy()
    out["meta"] = np.frombuffer(json.dumps(meta).encode(), dtype=np.uint8)
    path = os.path.join(HERE, f"{name}.npz")
    np.savez_compressed(path, **out)
    spikes = {k: v["spikes"] for k, v in meta["layers"].items()}
    print(f"{name}: reference wall {wall:.2f}s, spikes {spikes}, {os.path.getsize(path) / 1e6:.2f} MB")


if __name__ == "__main__":
    names = sys.argv[1:] or list(cases.CASES)
    for n in names:
        generate(n)
