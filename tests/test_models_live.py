"""``models.IncreasingInhibitionNetwork`` (reference: models.py:349-454) and ``models.LocallyConnectedNetwork``
(:457-584): same wiring as the reference (static weights equal to the bit, same layer / connection parameters), and
a learning window through the reference — ``torch.multinomial`` replaced by the shared tie-break hash, like the
goldens — equals ours on the oracle (the reference's side stored under tests/golden/live); the kernels' CUDA sources on
the emulation of tests/emu agree with the oracle bit for bit.  CPU only."""
import os
import sys

import numpy as np
import pytest
import torch

import cases
import helpers
from live import REF, stored

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "emu"))
sys.path.insert(0, os.path.join(HERE, "golden"))

T, B, SEED = 60, 3, 515


def _batch(which):
    return B if which == "increasing" else 1   # the reference's LocalConnection.compute views a_post as target.shape (topology.py:1453)


def _make(ns, which):
    g = torch.Generator().manual_seed(31)
    if which == "increasing":
        net = ns.models.IncreasingInhibitionNetwork(n_input=64, n_neurons=25, start_inhib=0.5, max_inhib=-30.0, nu=(1e-3, 1e-2),
                                                    reduction=torch.sum, norm=12.0, theta_plus=0.3, inpt_shape=(1, 8, 8))
        w = 0.45 * torch.rand(64, 25, generator=g)
    else:
        net = ns.models.LocallyConnectedNetwork(n_inpt=64, input_shape=[8, 8], kernel_size=4, stride=2, n_filters=3, inh=20.0,
                                                nu=(1e-3, 1e-2), reduction=torch.sum, theta_plus=0.3, norm=0.35)
        c = net.connections[("X", "Y")]
        w = torch.where(c.mask, torch.zeros(()), 0.9 * torch.rand(64, 27, generator=g))
    with torch.no_grad():
        net.connections[("X", "Y")].w.copy_(w)
    shape = (1, 8, 8) if which == "increasing" else (64,)
    x = torch.bernoulli(0.2 * torch.ones(T, _batch(which), *shape), generator=g).byte()
    return net, x


@pytest.mark.parametrize("which", ["increasing", "local"])
def test_wiring_equals_the_live_reference(which):
    params = ("thresh", "rest", "reset", "refrac", "tc_decay", "tc_trace", "theta_plus", "tc_theta_decay")

    def reference():
        ref, _ = _make(REF, which)
        a = ref.connections[("X", "Y")]
        out = {"layers": list(ref.layers), "connections": list(ref.connections), "Y->Y/w": ref.connections[("Y", "Y")].w,
               "Y": {name: float(getattr(ref.layers["Y"], name)) for name in params},
               "X->Y": (float(a.wmin), float(a.wmax), float(a.norm)), "nu": [float(v) for v in a.update_rule.nu]}
        if which == "local":
            out["mask"], out["locations"] = a.mask, a.locations
        else:
            out["n_sqrt"] = ref.n_sqrt
        return out

    ref = stored("wiring", reference)
    ours, _ = _make(cases.namespace("b200"), which)
    assert ref["layers"] == list(ours.layers) and ref["connections"] == list(ours.connections)
    assert torch.equal(ref["Y->Y/w"], ours.connections[("Y", "Y")].w)
    for name in params:
        assert ref["Y"][name] == float(getattr(ours.layers["Y"], name)), name
    b = ours.connections[("X", "Y")]
    assert ref["X->Y"] == (float(b.wmin), float(b.wmax), float(b.norm))
    assert ref["nu"] == [float(v) for v in b.update_rule.nu]
    if which == "local":
        assert torch.equal(ref["mask"], b.mask) and torch.equal(ref["locations"], b.locations)
        # a freshly drawn weight matrix lives inside the same receptive fields, within the same bounds
        fresh = cases.namespace("b200").models.LocallyConnectedNetwork(64, [8, 8], 4, 2, 3).connections[("X", "Y")]
        assert torch.equal(fresh.w == 0, b.mask) and float(fresh.w.max()) <= 1.0
    else:
        assert ours.n_sqrt == ref["n_sqrt"] == 5


@pytest.mark.parametrize("which", ["increasing", "local"])
def test_learning_window_matches_the_live_reference(which):
    from gen_golden import OneSpikePatch
    from oracle.oracle import OracleBackend

    def reference():
        ref, x = _make(REF, which)
        rmon = REF.monitors.Monitor(ref.layers["Y"], ["s"], time=T); ref.add_monitor(rmon, "Y")
        with OneSpikePatch(ref, SEED):
            ref.run(inputs={"X": x.clone()}, time=T)
        return rmon.get("s").reshape(T, _batch(which), -1).sum(dim=(0, 1)).numpy(), helpers.snapshot(ref)

    counts, a = stored("window", reference)
    ours, x2 = _make(cases.namespace("b200"), which)
    helpers.add_spike_monitors(ours, T)
    with OracleBackend() as ob:
        ours.run(inputs={"X": x2}, time=T, one_spike_seed=SEED)
        assert ob.err == 0
    assert counts.sum() > 10, "the window produced no activity: nothing tested"
    assert np.array_equal(counts, helpers.spike_counts(ours, T)["L/Y/count"])
    b = helpers.snapshot(ours)
    assert a.keys() == b.keys()
    for k in a:
        if k.endswith("/s"):
            assert np.array_equal(a[k], b[k]), k
        else:
            tol = (2e-6 + 1e-4 * np.abs(a[k])) if k.endswith("/w") else (1e-4 + 1e-5 * np.abs(a[k]))
            assert not (np.abs(a[k].astype(np.float64) - b[k]) > tol).any(), f"{which}: {k} max |d| {np.abs(a[k] - b[k]).max():.3e}"


@pytest.mark.parametrize("which", ["increasing", "local"])
def test_learning_window_on_the_emulated_kernel_bit_exact_vs_oracle(which):
    import emu
    from oracle.oracle import OracleBackend

    out = []
    for backend in (emu.EmuBackend, OracleBackend):
        net, x = _make(cases.namespace("b200"), which)
        helpers.add_spike_monitors(net, T)
        with backend() as be:
            net.run(inputs={"X": x}, time=T, one_spike_seed=SEED)
        assert be.err == 0
        out.append((helpers.snapshot(net), helpers.spike_counts(net, T)))
    helpers.assert_bit_identical(out[0][0], out[1][0], f"{which} state (emulated kernel)")
    helpers.assert_bit_identical(out[0][1], out[1][1], f"{which} spike counts (emulated kernel)")
