"""Randomised parity: small networks drawn from a seeded generator (layer kinds, rules, reductions, options, batch
sizes) run through the reference and through our host API on the oracle; both must agree within the north_star's
tolerances (final spikes equal, weights 1e-4 relative, state fp32 tolerance, spike counts equal).  The golden fixtures
pin hand-picked cases; this walks the option space between them.  The reference's results are stored under
tests/golden/live (see tests/golden/live.py).  CPU only."""
import hashlib
import os
import sys

import numpy as np
import pytest
import torch

import cases
import helpers
from live import REF, stored

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))

NODE_KINDS = ["LIFNodes", "IFNodes", "BoostedLIFNodes", "CurrentLIFNodes", "AdaptiveLIFNodes", "DiehlAndCookNodes", "McCullochPitts"]
RULES = ["PostPre", "WeightDependentPostPre", "Hebbian", "NoOp"]


def _draw(seed: int) -> dict:
    """One random network description (plain numbers and names only, so that both namespaces build the same thing)."""
    r = np.random.RandomState(seed)
    n_in, n_hid = int(r.randint(20, 90)), int(r.randint(8, 70))
    spec = dict(seed=seed, B=int(r.randint(1, 6)), T=int(r.randint(40, 110)), n_in=n_in, n_hid=n_hid,
                p_in=float(r.uniform(0.05, 0.3)), additive=bool(r.randint(2)), sum_input=bool(r.randint(2)),
                kind=NODE_KINDS[r.randint(len(NODE_KINDS))], rule=RULES[r.randint(len(RULES))],
                mean=bool(r.randint(2)), norm=(float(r.uniform(5.0, 25.0)) if r.randint(2) else None),
                decay=(float(r.uniform(1e-4, 5e-3)) if r.randint(3) == 0 else 0.0), bias=bool(r.randint(2)),
                nu=(float(r.uniform(5e-4, 5e-3)), float(r.uniform(2e-3, 4e-2))), second=bool(r.randint(2)),
                n_out=int(r.randint(6, 30)), lbound=bool(r.randint(2)))
    return spec


def _layer(ns, spec):
    k, n = spec["kind"], spec["n_hid"]
    common = dict(n=n, traces=True, traces_additive=spec["additive"], sum_input=spec["sum_input"])
    lb = -68.0 if spec["lbound"] else None
    if k == "LIFNodes":
        return ns.nodes.LIFNodes(thresh=-58.0, rest=-65.0, reset=-63.0, refrac=2, tc_decay=40.0, lbound=lb, **common)
    if k == "IFNodes":
        return ns.nodes.IFNodes(thresh=-57.0, reset=-64.0, refrac=3, lbound=lb, **common)
    if k == "BoostedLIFNodes":
        return ns.nodes.BoostedLIFNodes(thresh=6.0, refrac=2, tc_decay=30.0, **common)
    if k == "CurrentLIFNodes":
        return ns.nodes.CurrentLIFNodes(thresh=-57.0, rest=-65.0, reset=-63.0, refrac=2, tc_decay=40.0, tc_i_decay=3.0, lbound=lb, **common)
    if k == "AdaptiveLIFNodes":
        return ns.nodes.AdaptiveLIFNodes(thresh=-58.0, rest=-65.0, reset=-62.0, refrac=2, tc_decay=50.0, theta_plus=0.3,
                                         tc_theta_decay=150.0, lbound=lb, **common)
    if k == "DiehlAndCookNodes":   # one_spike off: no random draw on the path
        return ns.nodes.DiehlAndCookNodes(thresh=-58.0, rest=-65.0, reset=-62.0, refrac=2, tc_decay=50.0, theta_plus=0.3,
                                          tc_theta_decay=150.0, lbound=lb, one_spike=False, **common)
    return ns.nodes.McCullochPitts(thresh=4.0, **common)


def _build(ns, spec):
    g = torch.Generator().manual_seed(1000 + spec["seed"])
    net = ns.Network(dt=1.0, batch_size=spec["B"])
    X = ns.nodes.Input(n=spec["n_in"], traces=True, traces_additive=spec["additive"])
    Y = _layer(ns, spec)
    scale = {"BoostedLIFNodes": 1.5, "McCullochPitts": 1.2}.get(spec["kind"], 1.6)
    w = scale * torch.rand(spec["n_in"], spec["n_hid"], generator=g)
    kw = dict(w=w, update_rule=getattr(ns.learning, spec["rule"]), nu=spec["nu"], reduction=(torch.mean if spec["mean"] else torch.sum),
              wmin=0.0, wmax=2.0, weight_decay=spec["decay"])
    if spec["norm"] is not None:
        kw["norm"] = spec["norm"]
    if spec["bias"]:
        kw["b"] = 0.4 * torch.rand(spec["n_hid"], generator=g) - 0.1
    net.add_layer(X, "X"); net.add_layer(Y, "Y")
    net.add_connection(ns.topology.Connection(source=X, target=Y, **kw), "X", "Y")
    if spec["second"]:
        Z = ns.nodes.LIFNodes(n=spec["n_out"], traces=True, thresh=-59.0, rest=-65.0, reset=-64.0, refrac=1, tc_decay=30.0)
        w2 = 2.5 * torch.rand(spec["n_hid"], spec["n_out"], generator=g)
        net.add_layer(Z, "Z")
        net.add_connection(ns.topology.Connection(source=Y, target=Z, w=w2, update_rule=ns.learning.PostPre, nu=(1e-3, 1e-2),
                                                  reduction=torch.sum, wmin=0.0, wmax=3.0), "Y", "Z")
    x = torch.bernoulli(spec["p_in"] * torch.ones(spec["T"], spec["B"], spec["n_in"]), generator=g).byte()
    return net, x


def _snapshot(net):
    out = {}
    for name, layer in net.layers.items():
        B = layer.s.shape[0]
        out[f"{name}/s"] = layer.s.reshape(B, -1).to(torch.uint8).numpy().copy()
        for var in ("v", "refrac_count", "x", "theta", "summed", "i"):
            val = getattr(layer, var, None)
            if isinstance(val, torch.Tensor) and val.numel() and val.dtype.is_floating_point:
                out[f"{name}/{var}"] = val.detach().float().reshape(-1).numpy().copy()
    for (s, t), c in net.connections.items():
        out[f"{s}->{t}/w"] = c.w.detach().float().numpy().copy()
    return out


def _digest(x: torch.Tensor) -> str:
    return f"{x.dtype} {tuple(x.shape)} " + hashlib.sha256(x.contiguous().numpy().tobytes()).hexdigest()


@pytest.mark.parametrize("seed", list(range(24)))
def test_random_network_oracle_matches_live_reference(seed):
    from bindsnet_b200.network.monitors import Monitor
    from oracle.oracle import OracleBackend

    spec = _draw(seed)

    def reference():
        ref, x = _build(REF, spec)
        rmon = {n: REF.monitors.Monitor(l, ["s"], time=spec["T"]) for n, l in ref.layers.items()}
        for n, m in rmon.items():
            ref.add_monitor(m, n)
        ref.run(inputs={"X": x.clone()}, time=spec["T"])
        counts = {n: m.get("s").reshape(spec["T"], spec["B"], -1).sum(0).numpy() for n, m in rmon.items()}
        return _digest(x), counts, _snapshot(ref)

    x_digest, ref_counts, a = stored("window", reference)
    ours, x2 = _build(cases.namespace("b200"), spec)
    assert _digest(x2) == x_digest            # same input raster, drawn from the same seeded generator
    for n, l in ours.layers.items():
        ours.add_monitor(Monitor(l, ["s"], time=spec["T"]), n)
    with OracleBackend() as ob:
        ours.run(inputs={"X": x2}, time=spec["T"])
        assert ob.err == 0

    b = _snapshot(ours)
    assert a.keys() == b.keys(), (sorted(a), sorted(b))
    what = f"seed {seed} {spec['kind']} {spec['rule']} B={spec['B']}"
    for n, ca in ref_counts.items():   # spike counts per neuron over the window, exactly
        cb = ours.monitors[n].get("s").reshape(spec["T"], spec["B"], -1).sum(0).cpu().numpy()
        assert np.array_equal(ca, cb), f"{what}: spike counts of {n} differ"
    for k in a:
        if k.endswith("/s"):
            assert np.array_equal(a[k], b[k]), f"{what}: {k} differs"
        elif k.endswith("/w"):
            err = np.abs(a[k] - b[k]).max() / max(np.abs(a[k]).max(), 1e-12)
            assert err <= 1e-4, f"{what}: {k} max rel err {err:.3e}"
        else:
            bad = np.abs(a[k] - b[k]) > 1e-4 + 1e-5 * np.abs(a[k])
            assert not bad.any(), f"{what}: {k} max |d| {np.abs(a[k] - b[k]).max():.3e}"
    if seed == 0:
        assert sum(int(v.sum()) for k, v in a.items() if k.endswith("Y/s")) >= 0


@pytest.mark.parametrize("seed", [1, 4, 9, 12, 16, 19])
def test_random_network_oracle_dense_equals_sparse(seed):
    """The oracle's costed dense restatement (zeros multiplied like the reference does) and its zero-skipping mode agree
    bit for bit on the random networks too."""
    from oracle.oracle import OracleBackend

    spec = _draw(seed)
    ns = cases.namespace("b200")
    outs = []
    for dense in (0, 1):
        net, x = _build(ns, spec)
        helpers.add_spike_monitors(net, spec["T"])
        with OracleBackend(dense=dense) as ob:
            net.run(inputs={"X": x}, time=spec["T"])
            assert ob.err == 0
        outs.append((helpers.snapshot(net), helpers.spike_counts(net, spec["T"])))
    helpers.assert_bit_identical(outs[0][0], outs[1][0], f"seed {seed} state")
    helpers.assert_bit_identical(outs[0][1], outs[1][1], f"seed {seed} spike counts")
