"""``SRM0Nodes`` (reference: nodes.py:1555-1701) on the scripted tier: with torch's generator seeded alike, a learning
window of ``Input -> SRM0Nodes`` (PostPre, normalize) equals the reference's — same spikes, voltages and weights
within the north_star's tolerances (the built-in pieces run on the oracle backend here).  Also here, on the same tier:
``learning.Rmax`` (the rule made for SRM0 targets) and ``IzhikevichNodes``.  The reference's results are stored under
tests/golden/live (see tests/golden/live.py).  CPU only."""
import numpy as np
import pytest
import torch

import cases
import helpers
from live import REF, stored

T, B = 80, 3


def _net(ns, lbound=None):
    g = torch.Generator().manual_seed(61)
    net = ns.Network(dt=1.0, batch_size=B)
    X = ns.nodes.Input(n=40, traces=True)
    Y = ns.nodes.SRM0Nodes(n=15, traces=True, thresh=-55.0, rest=-70.0, reset=-72.0, refrac=3, tc_decay=12.0, eps_0=1.5,
                           rho_0=0.8, d_thresh=4.0, lbound=lbound, sum_input=True)
    net.add_layer(X, "X"); net.add_layer(Y, "Y")
    net.add_connection(ns.topology.Connection(source=X, target=Y, w=2.5 * torch.rand(40, 15, generator=g), update_rule=ns.learning.PostPre,
                                              nu=(1e-3, 1e-2), reduction=torch.sum, wmin=0.0, wmax=3.0, norm=40.0), "X", "Y")
    x = torch.bernoulli(0.25 * torch.ones(T, B, 40), generator=g).byte()
    return net, x


@pytest.mark.parametrize("lbound", [None, -71.0])
def test_srm0_window_matches_the_live_reference(lbound):
    from oracle.oracle import OracleBackend

    def reference():
        ref, x = _net(REF, lbound)
        rm = REF.monitors.Monitor(ref.layers["Y"], ["s", "v"], time=T); ref.add_monitor(rm, "Y")
        torch.manual_seed(2024)
        ref.run(inputs={"X": x.clone()}, time=T)
        return rm.get("s"), rm.get("v"), helpers.snapshot(ref)

    rs, rv, a = stored("window", reference)
    ours, x2 = _net(cases.namespace("b200"), lbound)
    assert ours._scripted_required()
    om = cases.namespace("b200").monitors.Monitor(ours.layers["Y"], ["s", "v"], time=T); ours.add_monitor(om, "Y")
    torch.manual_seed(2024)
    with OracleBackend() as ob:
        ours.run(inputs={"X": x2}, time=T)
        assert ob.err == 0
    assert torch.equal(rs, om.get("s")) and int(rs.sum()) > 20
    assert torch.allclose(rv, om.get("v"), rtol=1e-5, atol=1e-4)
    b = helpers.snapshot(ours)
    assert a.keys() == b.keys()
    for k in a:
        if k.endswith("/s"):
            assert np.array_equal(a[k], b[k]), k
        else:
            tol = (2e-6 + 1e-4 * np.abs(a[k])) if k.endswith("/w") else (1e-4 + 1e-5 * np.abs(a[k]))
            assert not (np.abs(a[k].astype(np.float64) - b[k]) > tol).any(), f"{k} max |d| {np.abs(a[k] - b[k]).max():.3e}"
    # reset_state_variables (nodes.py:1675-1682)
    ours.reset_state_variables()
    assert float(ours.layers["Y"].v.min()) == float(ours.layers["Y"].v.max()) == -70.0 and float(ours.layers["Y"].refrac_count.abs().sum()) == 0


def test_rmax_on_srm0_matches_the_live_reference():
    """``learning.Rmax`` (learning.py:2858-2960): eligibility trace per synapse, reward-scaled update — batch size 1,
    additive input traces, an SRM0 target; three windows with different rewards against the live reference."""
    from oracle.oracle import OracleBackend

    def build(ns):
        g = torch.Generator().manual_seed(62)
        net = ns.Network(dt=1.0, batch_size=1)
        X = ns.nodes.Input(n=30, traces=True, traces_additive=True)
        Y = ns.nodes.SRM0Nodes(n=10, traces=True, thresh=-56.0, refrac=2, tc_decay=15.0, rho_0=0.7, d_thresh=4.0)
        net.add_layer(X, "X"); net.add_layer(Y, "Y")
        net.add_connection(ns.topology.Connection(source=X, target=Y, w=2.0 * torch.rand(30, 10, generator=g), update_rule=ns.learning.Rmax,
                                                  nu=2e-2, wmin=0.0, wmax=3.0, weight_decay=1e-3, tc_c=4.0, tc_e_trace=20.0), "X", "Y")
        xs = [torch.bernoulli(0.3 * torch.ones(50, 1, 30), generator=g).byte() for _ in range(3)]
        return net, xs

    def reference():
        ref, xs = build(REF)
        torch.manual_seed(99)
        for r, x in zip((1.0, -0.5, 0.8), xs):
            ref.run(inputs={"X": x.clone()}, time=50, reward=r)
        Y, c = ref.layers["Y"], ref.connections[("X", "Y")]
        return Y.s, Y.v, c.w.detach(), c.update_rule.eligibility_trace

    rs, rv, wa, ea = stored("windows", reference)
    ours, xs2 = build(cases.namespace("b200"))
    assert ours._scripted_required()
    torch.manual_seed(99)
    with OracleBackend() as ob:
        for r, x in zip((1.0, -0.5, 0.8), xs2):
            ours.run(inputs={"X": x}, time=50, reward=r)
        assert ob.err == 0
    assert torch.equal(rs, ours.layers["Y"].s)
    assert torch.allclose(rv, ours.layers["Y"].v, rtol=1e-5, atol=1e-4)
    wb = ours.connections[("X", "Y")].w.detach()
    assert not ((wa - wb).abs() > 2e-6 + 1e-4 * wa.abs()).any(), float((wa - wb).abs().max())
    eb = ours.connections[("X", "Y")].update_rule.eligibility_trace
    assert torch.allclose(ea, eb, rtol=1e-4, atol=1e-5) and float(eb.abs().sum()) > 0


@pytest.mark.parametrize("excitatory", [1, 0, 0.75])
def test_izhikevich_nodes_match_the_live_reference(excitatory):
    """``IzhikevichNodes`` (nodes.py:1147-1316): a seeded construction gives the reference's per-neuron parameters and
    lateral matrix; a PostPre window through the scripted tier equals the live reference's."""
    from oracle.oracle import OracleBackend

    def build(ns):
        torch.manual_seed(321)
        net = ns.Network(dt=1.0, batch_size=2)
        X = ns.nodes.Input(n=30, traces=True)
        Y = ns.nodes.IzhikevichNodes(n=12, traces=True, excitatory=excitatory, thresh=30.0, lbound=-80.0, sum_input=True)
        net.add_layer(X, "X"); net.add_layer(Y, "Y")
        g = torch.Generator().manual_seed(63)
        net.add_connection(ns.topology.Connection(source=X, target=Y, w=6.0 * torch.rand(30, 12, generator=g), update_rule=ns.learning.PostPre,
                                                  nu=(1e-3, 1e-2), reduction=torch.sum, wmin=0.0, wmax=8.0), "X", "Y")
        return net, torch.bernoulli(0.3 * torch.ones(70, 2, 30), generator=g).byte()

    params = ("r", "a", "b", "c", "d", "S", "excitatory", "u")
    state = ("v", "u", "x", "summed")

    def reference():
        ref, x = build(REF)
        built = {name: getattr(ref.layers["Y"], name).clone() for name in params}
        rm = REF.monitors.Monitor(ref.layers["Y"], ["s"], time=70); ref.add_monitor(rm, "Y")
        ref.run(inputs={"X": x.clone()}, time=70)
        return built, rm.get("s"), {name: getattr(ref.layers["Y"], name) for name in state}, ref.connections[("X", "Y")].w.detach()

    built, rs, after, wa = stored("window", reference)
    ours, x2 = build(cases.namespace("b200"))
    for name in params:
        assert torch.equal(built[name], getattr(ours.layers["Y"], name)), name
    om = cases.namespace("b200").monitors.Monitor(ours.layers["Y"], ["s"], time=70); ours.add_monitor(om, "Y")
    assert ours._scripted_required()
    with OracleBackend() as ob:
        ours.run(inputs={"X": x2}, time=70)
        assert ob.err == 0
    assert torch.equal(rs, om.get("s")) and int(om.get("s").sum()) > 10
    for name in state:
        assert torch.allclose(after[name], getattr(ours.layers["Y"], name), rtol=1e-4, atol=1e-3), name
    wb = ours.connections[("X", "Y")].w.detach()
    assert not ((wa - wb).abs() > 2e-6 + 1e-4 * wa.abs()).any(), float((wa - wb).abs().max())
