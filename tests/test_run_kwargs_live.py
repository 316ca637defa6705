"""Run kwargs of ``Network.run`` that no golden fixture covers, through the reference (its results stored under
tests/golden/live) and through our host API on the oracle, plus the kernels' CUDA sources on the emulation of tests/emu:

* ``a_plus`` / ``a_minus`` as dicts keyed by connection (network.py:359-377, 440-461): each connection's MSTDP sees its
  own entry, a connection without one the rule's defaults (learning.py:1552-1553);
* ``clamp`` / ``unclamp`` as per-step INDEX tensors ``[T, k]`` (network.py:416-429), not only bool masks.

CPU only."""
import os
import sys

import numpy as np
import pytest
import torch

import cases
import helpers
from live import REF, stored

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "emu"))

T, B = 50, 2


def _two_mstdp(ns):
    g = torch.Generator().manual_seed(77)
    net = ns.Network(dt=1.0, batch_size=B)
    X = ns.nodes.Input(n=40, traces=True)
    Y = ns.nodes.LIFNodes(n=14, traces=True, thresh=-61.0, refrac=1)
    Z = ns.nodes.LIFNodes(n=9, traces=True, thresh=-60.0, refrac=2)
    for l, n in ((X, "X"), (Y, "Y"), (Z, "Z")):
        net.add_layer(l, n)
    common = dict(update_rule=ns.learning.MSTDP, reduction=torch.sum, wmin=-1.0, wmax=2.5, tc_plus=15.0, tc_minus=25.0)
    net.add_connection(ns.topology.Connection(source=X, target=Y, w=1.4 * torch.rand(40, 14, generator=g), nu=3e-2, **common), "X", "Y")
    net.add_connection(ns.topology.Connection(source=Y, target=Z, w=2.4 * torch.rand(14, 9, generator=g), nu=5e-2, **common), "Y", "Z")
    x = torch.bernoulli(0.15 * torch.ones(T, B, 40), generator=g).byte()
    return net, x


def _clamped(ns):
    g = torch.Generator().manual_seed(78)
    net = ns.Network(dt=1.0, batch_size=B)
    X = ns.nodes.Input(n=40, traces=True)
    Y = ns.nodes.LIFNodes(n=14, traces=True, thresh=-58.0, refrac=1)
    net.add_layer(X, "X"); net.add_layer(Y, "Y")
    net.add_connection(ns.topology.Connection(source=X, target=Y, w=0.9 * torch.rand(40, 14, generator=g), update_rule=ns.learning.PostPre,
                                              nu=(1e-3, 1e-2), reduction=torch.sum, wmin=0.0, wmax=1.0), "X", "Y")
    x = torch.bernoulli(0.12 * torch.ones(T, B, 40), generator=g).byte()
    clamp = torch.randint(0, 14, (T, 2), generator=g)           # two neurons forced to spike each step (repeats allowed)
    unclamp = torch.randint(0, 14, (T, 3), generator=g)         # three forbidden each step
    static = torch.tensor([0, 13])                              # 1-D index form on the input layer
    return net, x, {"clamp": {"Y": clamp}, "unclamp": {"Y": unclamp, "X": static}}


def _compare(a, ours, what):
    b = helpers.snapshot(ours)
    assert a.keys() == b.keys()
    for k in a:
        if k.endswith("/s"):
            assert np.array_equal(a[k], b[k]), f"{what}: {k} differs"
        else:
            tol = (2e-6 + 1e-4 * np.abs(a[k])) if k.endswith("/w") else (1e-4 + 1e-5 * np.abs(a[k]))
            assert not (np.abs(a[k].astype(np.float64) - b[k]) > tol).any(), f"{what}: {k} max |d| {np.abs(a[k] - b[k]).max():.3e}"


KW = {"reward": 0.6, "a_plus": {("X", "Y"): 0.7, ("Y", "Z"): 1.4}, "a_minus": {("Y", "Z"): -0.5}}


def test_per_connection_a_plus_a_minus_match_the_live_reference():
    from oracle.oracle import OracleBackend

    def reference():
        ref, x = _two_mstdp(REF)
        ref.run(inputs={"X": x.clone()}, time=T, **{k: (dict(v) if isinstance(v, dict) else v) for k, v in KW.items()})
        return helpers.snapshot(ref)

    ref = stored("state", reference)
    ours, x2 = _two_mstdp(cases.namespace("b200"))
    with OracleBackend() as ob:
        ours.run(inputs={"X": x2}, time=T, **KW)
        assert ob.err == 0
    _compare(ref, ours, "a_plus / a_minus dicts")
    # the dict entries were used: scalar kwargs end elsewhere
    flat, x3 = _two_mstdp(cases.namespace("b200"))
    with OracleBackend():
        flat.run(inputs={"X": x3}, time=T, reward=0.6, a_plus=0.7)
    assert not torch.equal(flat.connections[("Y", "Z")].w, ours.connections[("Y", "Z")].w)


def test_per_step_index_clamps_match_the_live_reference():
    from oracle.oracle import OracleBackend

    def reference():
        ref, x, kw = _clamped(REF)
        rm = REF.monitors.Monitor(ref.layers["Y"], ["s"], time=T); ref.add_monitor(rm, "Y")
        ref.run(inputs={"X": x.clone()}, time=T, **kw)
        return helpers.snapshot(ref), rm.get("s").reshape(T, B, -1).sum(dim=(0, 1)).numpy()

    ref, ca = stored("state", reference)
    ours, x2, kw2 = _clamped(cases.namespace("b200"))
    helpers.add_spike_monitors(ours, T)
    with OracleBackend() as ob:
        ours.run(inputs={"X": x2}, time=T, **kw2)
        assert ob.err == 0
    _compare(ref, ours, "index clamps")
    assert np.array_equal(ca, helpers.spike_counts(ours, T)["L/Y/count"])
    assert ca.sum() >= T      # the clamps fired


@pytest.mark.parametrize("which", ["dicts", "clamps"])
def test_the_same_runs_on_the_emulated_kernels_bit_exact_vs_oracle(which):
    import emu
    from oracle.oracle import OracleBackend

    ns = cases.namespace("b200")

    def once(backend):
        if which == "dicts":
            net, x = _two_mstdp(ns); kw = KW
        else:
            net, x, kw = _clamped(ns)
        helpers.add_spike_monitors(net, T)
        with backend() as be:
            net.run(inputs={"X": x}, time=T, **kw)
        assert be.err == 0
        return helpers.snapshot(net), helpers.spike_counts(net, T)

    s_emu, c_emu = once(emu.EmuBackend)
    s_cpu, c_cpu = once(OracleBackend)
    helpers.assert_bit_identical(s_emu, s_cpu, f"{which} state (emulated kernel)")
    helpers.assert_bit_identical(c_emu, c_cpu, f"{which} spike counts (emulated kernel)")
