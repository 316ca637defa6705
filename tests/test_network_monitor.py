"""``monitors.NetworkMonitor`` (reference: monitors.py:127-329): per-step recordings of every layer's and connection's
state variables — growing (``time=None``) and rolling (``time=T``) — equal the reference's on the same run (spikes
exactly, voltages and weights within the north_star's tolerances; the reference's recordings are stored under
tests/golden/live); the same run on the kernels' CUDA sources (emulation of tests/emu) equals the oracle bit for bit;
``save`` writes the reference's npz keys.  CPU only."""
import os
import sys

import numpy as np
import pytest
import torch

import cases
from live import REF, stored

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "emu"))

T, B = 30, 2


def _net(ns):
    g = torch.Generator().manual_seed(91)
    net = ns.Network(dt=1.0, batch_size=B)
    X = ns.nodes.Input(n=30, traces=True)
    Y = ns.nodes.LIFNodes(n=12, traces=True, thresh=-60.0, refrac=1)
    net.add_layer(X, "X"); net.add_layer(Y, "Y")
    net.add_connection(ns.topology.Connection(source=X, target=Y, w=1.1 * torch.rand(30, 12, generator=g), update_rule=ns.learning.PostPre,
                                              nu=(1e-3, 1e-2), reduction=torch.sum, wmin=0.0, wmax=1.2, norm=9.0), "X", "Y")
    x = torch.bernoulli(0.2 * torch.ones(T, B, 30), generator=g).byte()
    return net, x


def _record(ns, time, backend=None):
    net, x = _net(ns)
    mon = ns.monitors.NetworkMonitor(net, time=time)
    net.add_monitor(mon, "all")
    if backend is None:
        net.run(inputs={"X": x}, time=T)
    else:
        with backend() as be:
            net.run(inputs={"X": x}, time=T)
        assert be.err == 0
    return mon


@pytest.mark.parametrize("time", [None, T, 7])
def test_network_monitor_matches_the_live_reference(time):
    from oracle.oracle import OracleBackend

    ref = stored("recording", lambda: _record(REF, time).get())
    ours = _record(cases.namespace("b200"), time, OracleBackend).get()
    assert list(ref) == list(ours) == ["X", "Y", ("X", "Y")]
    for key in ref:
        assert sorted(ref[key]) == sorted(ours[key]), key
        for v in ref[key]:
            a, b = ref[key][v], ours[key][v].cpu()
            assert a.shape == b.shape and a.dtype == b.dtype, (key, v, a.shape, b.shape, a.dtype, b.dtype)
            assert a.shape[0] == (T if time is None else time)
            if v == "s":
                assert torch.equal(a, b), (key, v)
            else:
                tol = 2e-6 + 1e-4 * a.abs() if v == "w" else 1e-4 + 1e-5 * a.abs()
                assert not ((a - b).abs() > tol).any(), (key, v, float((a - b).abs().max()))
    assert ref["Y"]["s"].sum() > 0 and not torch.equal(ref[("X", "Y")]["w"][0], ref[("X", "Y")]["w"][-1])


def test_network_monitor_on_the_emulated_kernel_bit_exact_vs_oracle(tmp_path):
    import emu
    from oracle.oracle import OracleBackend

    ns = cases.namespace("b200")
    a, b = _record(ns, None, emu.EmuBackend), _record(ns, None, OracleBackend)
    for key in a.get():
        for v in a.get()[key]:
            assert torch.equal(a.get()[key][v], b.get()[key][v]), (key, v)
    # save / reset (monitors.py:258-329)
    path = os.path.join(tmp_path, "rec", "all.npz")
    a.save(path)
    z = np.load(path)
    assert sorted(z.files) == ["X-Y_w", "X_s", "Y_s", "Y_v"]
    assert np.array_equal(z["Y_s"], a.get()["Y"]["s"].numpy())
    a.reset_state_variables()
    assert a.get()["Y"]["s"].numel() == 0
    rolling = ns.monitors.NetworkMonitor(a.network, layers=["Y"], connections=[], state_vars=("s", "theta"), time=5)
    assert list(rolling.get()) == ["Y"] and list(rolling.get()["Y"]) == ["s"] and rolling.get()["Y"]["s"].shape == (5, B, 12)


def test_get_inputs_matches_the_live_reference():
    """``Network._get_inputs`` (network.py:211-250) as a host call: per-target sums of ``compute`` over the connections."""
    from oracle.oracle import OracleBackend

    def build(ns):
        net, _ = _net(ns)
        g = torch.Generator().manual_seed(5)
        Z = ns.nodes.LIFNodes(n=12, traces=True)
        net.add_layer(Z, "Z")
        net.add_connection(ns.topology.Connection(source=Z, target=net.layers["Y"], w=torch.rand(12, 12, generator=g) - 0.5,
                                                  b=0.1 * torch.rand(12, generator=g)), "Z", "Y")
        net.add_connection(ns.topology.Connection(source=net.layers["Y"], target=Z, w=torch.rand(12, 12, generator=g)), "Y", "Z")
        for name, p in (("X", 0.3), ("Y", 0.4), ("Z", 0.5)):
            net.layers[name].s = torch.bernoulli(p * torch.ones(B, net.layers[name].n), generator=g).bool()
        return net

    a = stored("inputs", lambda: build(REF)._get_inputs())
    ours = build(cases.namespace("b200"))
    with OracleBackend():
        b = ours._get_inputs()
        only = ours._get_inputs(["Z"])
    assert sorted(a) == sorted(b) == ["Y", "Z"] and list(only) == ["Z"]
    for k in a:
        assert a[k].shape == b[k].shape and torch.allclose(a[k], b[k], rtol=1e-5, atol=1e-6), k
    assert torch.equal(only["Z"], b["Z"]) and float(a["Y"].abs().sum()) > 0
