"""Host-side logic (plan building, reference API quirks) exercised on CPU through the oracle
backend — mirrors what the reference's own tests check (test/network/test_network.py,
test_monitors.py, test_nodes.py, test/models/test_models.py) plus the run() semantics."""
import os

import numpy as np
import pytest
import torch

from bindsnet_b200 import _abi, _backend
from bindsnet_b200.learning import NoOp, PostPre, WeightDependentPostPre, MSTDP, MSTDPET
from bindsnet_b200.models import DiehlAndCook2015, DiehlAndCook2015v2, TwoLayerNetwork
from bindsnet_b200.network import Network, load
from bindsnet_b200.network.monitors import Monitor
from bindsnet_b200.network.nodes import DiehlAndCookNodes, IFNodes, Input, LIFNodes
from bindsnet_b200.network.topology import Connection, Conv1dConnection, Conv2dConnection, MulticompartmentConnection
from bindsnet_b200.network.topology_features import Weight
from oracle.oracle import OracleBackend


def test_model_wiring_matches_reference_tests():
    # test/models/test_models.py:6-67
    net = TwoLayerNetwork(n_inpt=50, n_neurons=32)
    assert isinstance(net.layers["X"], Input) and isinstance(net.layers["Y"], LIFNodes)
    assert net.connections[("X", "Y")].w.shape == (50, 32)
    dc = DiehlAndCook2015(n_inpt=50, n_neurons=20, exc=22.5, inh=17.5)
    assert isinstance(dc.layers["Ae"], DiehlAndCookNodes) and isinstance(dc.layers["Ai"], LIFNodes)
    assert set(dc.connections) == {("X", "Ae"), ("Ae", "Ai"), ("Ai", "Ae")}
    assert torch.equal(dc.connections[("Ae", "Ai")].w, 22.5 * torch.eye(20))
    assert isinstance(dc.connections[("X", "Ae")], MulticompartmentConnection)
    v2 = DiehlAndCook2015v2(n_inpt=50, n_neurons=20)
    assert set(v2.connections) == {("X", "Y"), ("Y", "Y")}


def test_nodes_initial_state_like_reference():
    # test/network/test_nodes.py:17-59
    for cls in (LIFNodes, DiehlAndCookNodes):
        l = cls(n=100, traces=True)
        l.compute_decays(1.0); l.set_batch_size(3)
        assert l.s.shape == (3, 100) and not l.s.any()
        assert torch.all(l.v == l.rest) and torch.all(l.x == 0) and torch.all(l.refrac_count == 0)
    # decays are exp(-dt/tc) evaluated in fp32 like nodes.py:129-131,546-548
    l = LIFNodes(n=4, tc_decay=100.0)
    l.compute_decays(1.0)
    assert float(l.decay) == float(torch.exp(-torch.tensor(1.0) / torch.tensor(100.0)))


def test_unsupported_reference_features_fail_loudly():
    from bindsnet_b200.network.nodes import CSRMNodes, IzhikevichNodes

    assert IFNodes(n=10).kind is not None          # implemented since round 2 (SURVEY.md §8f rank 4)
    assert IzhikevichNodes(n=10).kind is None      # host class on the scripted tier (tests/test_srm0_live.py)
    with pytest.raises(NotImplementedError):
        CSRMNodes(n=10)
    with pytest.raises(NotImplementedError):
        Conv1dConnection(None, None, 3)
    X, Y = Input(n=4, traces=True), LIFNodes(n=4, traces=True)
    from bindsnet_b200.learning import Rmax
    with pytest.raises(AssertionError):            # learning.py:2899-2904: additive input traces and an SRM0Nodes target
        Connection(X, Y, update_rule=Rmax)
    # MSTDPET is implemented for dense connections at batch size 1 (the only one the reference's flattened traces allow)
    netb = Network(dt=1.0, batch_size=2)
    Xb, Yb = Input(n=4, traces=True), LIFNodes(n=4, traces=True)
    netb.add_layer(Xb, "X"); netb.add_layer(Yb, "Y")
    netb.add_connection(Connection(Xb, Yb, update_rule=MSTDPET, nu=1e-2, wmin=-1.0, wmax=1.0), "X", "Y")
    with OracleBackend():
        with pytest.raises(NotImplementedError):
            netb.run({"X": torch.zeros(3, 2, 4)}, time=3, reward=1.0)
    # MSTDP is implemented (SURVEY.md §8a A11/A12); its reward is mandatory like in the reference
    net = Network(dt=1.0, batch_size=1)
    net.add_layer(X, "X"); net.add_layer(Y, "Y")
    net.add_connection(Connection(X, Y, update_rule=MSTDP, nu=1e-2, wmin=-1.0, wmax=1.0), "X", "Y")
    with OracleBackend():
        with pytest.raises(KeyError):
            net.run({"X": torch.zeros(3, 1, 4)}, time=3)
    with pytest.raises(NotImplementedError):
        Connection(X, Y, w_dtype=torch.float16)
    net = TwoLayerNetwork(n_inpt=8, n_neurons=4)
    with OracleBackend():   # masks (network.py:279-280): implemented for dense connections — all weights masked -> all zero
        net.run({"X": torch.ones(3, 1, 8, dtype=torch.uint8)}, time=3, masks={("X", "Y"): torch.ones(8, 4, dtype=torch.bool)})
    assert float(net.connections[("X", "Y")].w.abs().sum()) == 0.0
    with pytest.raises(ValueError):
        net.run({"X": torch.zeros(3, 1, 8)}, time=3, masks={("X", "Y"): torch.ones(4, 8, dtype=torch.bool)})   # wrong shape
    with pytest.raises(AssertionError):
        net.run([torch.zeros(3, 1, 8)], time=3)


def test_batch_size_inference_resets_state_and_monitor_shapes():
    # network.py:329-353; test/network/test_monitors.py:8-84
    net = TwoLayerNetwork(n_inpt=30, n_neurons=12, reduction=torch.sum)
    net.add_monitor(Monitor(net.layers["Y"], ["s", "v"], time=20), "Y")
    net.add_monitor(Monitor(net.layers["X"], ["s"], time=20), "X")
    g = torch.Generator().manual_seed(0)
    with OracleBackend():
        net.run({"X": torch.bernoulli(0.3 * torch.ones(20, 30), generator=g)}, time=20)  # [T, n] -> batch 1
        assert net.batch_size == 1 and net.monitors["Y"].get("s").shape == (20, 1, 12)
        assert net.monitors["Y"].get("v").shape == (20, 1, 12) and net.monitors["X"].get("s").shape == (20, 1, 30)
        net.layers["Y"].v.fill_(-55.0)
        net.run({"X": torch.bernoulli(0.3 * torch.ones(20, 5, 30), generator=g).byte()}, time=20)  # batch 5
        assert net.batch_size == 5 and net.layers["Y"].v.shape == (5, 12)
        assert net.monitors["Y"].get("s").shape == (20, 5, 12)
        # X's monitor returns exactly the input spikes
        x = torch.bernoulli(0.3 * torch.ones(20, 5, 30), generator=g).byte()
        net.run({"X": x}, time=20)
        assert torch.equal(net.monitors["X"].get("s"), x.bool())


def test_stepwise_fallback_equals_fused_window():
    """A monitor on a variable the kernels do not record (x) makes run() fall back to one-step
    windows; the result must equal the fused window bit for bit (same tie-break stream)."""
    def build():
        torch.manual_seed(1)
        return DiehlAndCook2015(n_inpt=64, n_neurons=24, batch_size=3, inpt_shape=(1, 8, 8), inh=60.0)
    g = torch.Generator().manual_seed(2)
    x = torch.bernoulli(0.15 * torch.ones(40, 3, 1, 8, 8), generator=g).byte()
    a, b = build(), build()
    b.add_monitor(Monitor(b.layers["Ae"], ["x", "s"], time=40), "trace")
    with OracleBackend():
        a.run({"X": x}, time=40, one_spike_seed=9)
        b.run({"X": x}, time=40, one_spike_seed=9)
    for name in ("Ae", "Ai"):
        assert torch.equal(a.layers[name].v, b.layers[name].v) and torch.equal(a.layers[name].s, b.layers[name].s)
    assert torch.equal(a.connections[("X", "Ae")].w, b.connections[("X", "Ae")].w)
    assert b.monitors["trace"].get("x").shape == (40, 3, 24)


def test_learning_off_freezes_weights_and_theta():
    net = DiehlAndCook2015(n_inpt=64, n_neurons=16, batch_size=2, inpt_shape=(1, 8, 8))
    net.train(False)
    w0 = net.connections[("X", "Ae")].w.detach().clone()
    net.layers["Ae"].theta.fill_(0.5)
    with OracleBackend():
        net.run({"X": torch.ones(30, 2, 1, 8, 8, dtype=torch.uint8)}, time=30)
    # no STDP; the end-of-run normalize still runs, learning or not (network.py:464-465)
    assert torch.allclose(net.connections[("X", "Ae")].w, w0 * (78.4 / w0.sum(0)), rtol=1e-5)
    assert torch.all(net.layers["Ae"].theta == 0.5)


def test_reset_state_variables_keeps_theta_and_w():
    # nodes.py:1113-1120: theta is not reset
    net = DiehlAndCook2015(n_inpt=64, n_neurons=16, batch_size=2, inpt_shape=(1, 8, 8), inh=60.0)
    with OracleBackend():
        net.run({"X": torch.ones(40, 2, 1, 8, 8, dtype=torch.uint8)}, time=40)
    theta = net.layers["Ae"].theta.clone(); w = net.connections[("X", "Ae")].w.detach().clone()
    assert theta.abs().sum() > 0
    net.reset_state_variables()
    assert torch.equal(net.layers["Ae"].theta, theta) and torch.equal(net.connections[("X", "Ae")].w, w)
    assert torch.all(net.layers["Ae"].v == -65.0) and not net.layers["Ae"].s.any() and torch.all(net.layers["X"].x == 0)


def test_save_load_clone_round_trip(tmp_path):
    # test/network/test_network.py:15-68
    net = DiehlAndCook2015(n_inpt=16, n_neurons=8, batch_size=1, inpt_shape=(1, 4, 4))
    net.add_monitor(Monitor(net.layers["Ae"], ["s"], time=5), "m")
    p = tmp_path / "net.pt"
    net.save(str(p))
    net2 = load(str(p), learning=False)
    assert net2.dt == net.dt and net2.learning is False
    assert list(net2.layers) == list(net.layers) and list(net2.connections) == list(net.connections)
    assert torch.equal(net2.connections[("X", "Ae")].w, net.connections[("X", "Ae")].w)
    net3 = net.clone()
    assert list(net3.monitors) == ["m"]


def test_squeeze_reduction_pitfall_is_reported():
    # SURVEY.md §0.9: TwoLayerNetwork builds its rule with reduction=squeeze (batch_size==1 at construction)
    net = TwoLayerNetwork(n_inpt=10, n_neurons=4)
    with OracleBackend():
        net.run({"X": torch.zeros(3, 1, 10, dtype=torch.uint8)}, time=3)   # batch 1: fine
        with pytest.raises(RuntimeError, match="squeeze"):
            net.run({"X": torch.zeros(3, 2, 10, dtype=torch.uint8)}, time=3)


def test_structure_hints_detected_for_static_matrices():
    from bindsnet_b200.network import _plan

    net = DiehlAndCook2015(n_inpt=16, n_neurons=8, batch_size=2, inpt_shape=(1, 4, 4), exc=22.5, inh=120.0)
    plan, _ = _plan.build_net(net, 2, {}, {}, {}, {}, {})
    kinds = [(plan.conns[i].structure, plan.conns[i].structure_val) for i in range(3)]
    assert kinds[0][0] == _abi.SNN_W_DENSE
    assert kinds[1] == (_abi.SNN_W_DIAG, 22.5) and kinds[2] == (_abi.SNN_W_OFFDIAG, -120.0)
    with torch.no_grad():
        net.connections[("Ai", "Ae")].w[0, 1] = -1.0            # in-place edit bumps Tensor._version
    plan, _ = _plan.build_net(net, 2, {}, {}, {}, {}, {})
    assert plan.conns[2].structure == _abi.SNN_W_DENSE


def test_nonbinary_input_flag_from_oracle_backend():
    net = TwoLayerNetwork(n_inpt=6, n_neurons=3)
    x = torch.zeros(4, 1, 6, dtype=torch.uint8); x[1, 0, 2] = 5
    with OracleBackend() as ob:
        net.run({"X": x}, time=4)
    assert ob.err & _abi.SNN_ERR_NONBINARY


def test_spike_counter_equals_raster_sum():
    """SpikeCounter (in-kernel counts, no raster) == Monitor raster summed over time."""
    from bindsnet_b200.network.monitors import SpikeCounter

    torch.manual_seed(4)
    net = DiehlAndCook2015(n_inpt=64, n_neurons=24, batch_size=3, inpt_shape=(1, 8, 8), inh=60.0)
    net.add_monitor(Monitor(net.layers["Ae"], ["s"], time=50), "raster")
    net.add_monitor(SpikeCounter(net.layers["Ae"]), "count")
    net.add_monitor(SpikeCounter(net.layers["Ai"]), "count_i")
    g = torch.Generator().manual_seed(5)
    with OracleBackend():
        for _ in range(2):  # counts restart every window
            x = torch.bernoulli(0.2 * torch.ones(50, 3, 1, 8, 8), generator=g).byte()
            net.run({"X": x}, time=50, one_spike_seed=1)
            raster = net.monitors["raster"].get("s")
            assert torch.equal(net.monitors["count"].get("s"), raster.sum(0).to(torch.int32))
            assert net.monitors["count"].get("s").shape == (3, 24) and raster.sum() > 0
            assert net.monitors["count_i"].get("s").sum() > 0


def test_async_readback_ring_order_and_overflow():
    """pipeline.AsyncReadback hands results back in submission order, one window behind."""
    from bindsnet_b200.pipeline import AsyncReadback

    rb = AsyncReadback(depth=2)
    seen = []
    for k in range(5):
        rb.push(torch.full((3, 4), k, dtype=torch.int32))
        if len(rb) == rb.depth:
            seen.append(int(rb.pop()[0, 0]))
    while len(rb):
        seen.append(int(rb.pop()[0, 0]))
    assert seen == [0, 1, 2, 3, 4]
    rb.push(torch.zeros(2)); rb.push(torch.zeros(2))
    with pytest.raises(RuntimeError):
        rb.push(torch.zeros(2))


def test_conv2d_connection_constructor_and_window_like_reference_tests():
    """test/network/test_connections.py (Conv2dConnection cases): constructor geometry checks, default
    weights inside [wmin, wmax], zero bias, and a short run through the window path."""
    from bindsnet_b200.network.nodes import Input as In

    X = In(shape=[2, 9, 9], traces=True)
    H = LIFNodes(shape=[3, 5, 5], traces=True)
    c = Conv2dConnection(X, H, kernel_size=3, stride=2, padding=1, wmin=-0.5, wmax=0.5)
    assert tuple(c.w.shape) == (3, 2, 3, 3) and tuple(c.b.shape) == (3,) and not c.b.any()
    assert float(c.w.min()) >= -0.5 and float(c.w.max()) <= 0.5
    with pytest.raises(AssertionError):
        Conv2dConnection(X, LIFNodes(shape=[3, 4, 4]), kernel_size=3, stride=2, padding=1)   # wrong target size
    from bindsnet_b200._backend import BackendError
    with pytest.raises(BackendError):
        c.compute(torch.zeros(1, 2, 9, 9))                                                    # CPU tensors: no CPU fallback
    g0 = torch.Generator().manual_seed(3)
    s0 = torch.bernoulli(0.3 * torch.ones(4, 2, 9, 9), generator=g0).byte()
    cn = Conv2dConnection(X, H, kernel_size=3, stride=2, padding=1, wmin=-0.5, wmax=0.5, norm=0.7,
                          b=torch.tensor([0.1, -0.2, 0.3]))
    with OracleBackend():  # standalone operators (topology.py:799-815, 824-837) against torch
        out = cn.compute(s0)
        ref = torch.nn.functional.conv2d(s0.float(), cn.w, cn.b, stride=2, padding=1)
        assert out.shape == ref.shape and torch.allclose(out, ref, atol=1e-5)
        w0 = cn.w.clone()
        cn.normalize()
        expect = w0 * (0.7 / w0.sum(dim=(2, 3), keepdim=True))
        assert torch.allclose(cn.w, expect, rtol=1e-5, atol=1e-6)
    net = Network(dt=1.0, batch_size=2)
    net.add_layer(X, "X"); net.add_layer(H, "H")
    net.add_connection(c, "X", "H")
    net.add_monitor(Monitor(H, ["s", "v"], time=12), "H")
    g = torch.Generator().manual_seed(5)
    with OracleBackend():
        net.run({"X": torch.bernoulli(0.3 * torch.ones(12, 2, 2, 9, 9), generator=g).byte()}, time=12)
    assert net.monitors["H"].get("s").shape == (12, 2, 3, 5, 5) and net.monitors["H"].get("v").shape == (12, 2, 3, 5, 5)


def test_mstdp_rule_state_and_eligibility_view():
    """learning.MSTDP keeps p_plus / p_minus like the reference and rebuilds the dense eligibility on request
    (learning.py:1519-1535, 1568-1572)."""
    X, Y = Input(n=6, traces=True), LIFNodes(n=4, traces=True, thresh=-64.0)
    net = Network(dt=1.0, batch_size=2)
    net.add_layer(X, "X"); net.add_layer(Y, "Y")
    c = Connection(X, Y, update_rule=MSTDP, nu=1e-1, reduction=torch.sum, wmin=-1.0, wmax=1.0, w=0.5 * torch.ones(6, 4))
    net.add_connection(c, "X", "Y")
    x = torch.ones(8, 2, 6, dtype=torch.uint8)
    with OracleBackend():
        net.run({"X": x}, time=8, reward=1.0)
    r = c.update_rule
    assert r.p_plus.shape == (2, 6) and r.p_minus.shape == (2, 4) and r.eligibility.shape == (2, 6, 4)
    # constant input: P+ = sum_k decay^k after 8 steps of a_plus = 1 (fp32, same order as the rule)
    p = torch.tensor(0.0)
    for _ in range(8):
        p = p * torch.exp(torch.tensor(-1.0) / r.tc_plus) + 1.0
    assert torch.allclose(r.p_plus, p.expand(2, 6))
    assert not torch.equal(c.w, 0.5 * torch.ones(6, 4))   # reward-modulated update happened


def test_local_connection_structure_matches_the_reference():
    """LocalConnection (topology.py:1304-1484): receptive-field structure (mask of the default initialisation), kernel-scaled
    norm and the bias the reference always creates — compared with the reference's (stored under tests/golden/live)."""
    from bindsnet_b200.network.topology import LocalConnection
    from live import REF, stored

    X, Y = Input(n=64, traces=True), LIFNodes(n=2 * 36, traces=True)
    c = LocalConnection(X, Y, kernel_size=3, stride=1, n_filters=2, norm=0.5, wmin=0.0, wmax=1.0)
    assert c.w.shape == (64, 72) and c.mask.shape == (64, 72) and c.b.shape == (72,)
    assert int((~c.mask).sum()) == 2 * 36 * 9                       # n_filters * conv_prod * kernel_prod weights inside the fields
    assert torch.all(c.w[c.mask] == 0) and float(c.norm) == pytest.approx(0.5 * 9)
    assert bool(((~c.mask).sum(0) == 9).all())                      # every target neuron sees exactly one 3x3 field
    def reference():
        rx, ry = REF.nodes.Input(n=64, traces=True), REF.nodes.LIFNodes(n=72, traces=True)
        rc = REF.topology.LocalConnection(rx, ry, kernel_size=3, stride=1, n_filters=2, norm=0.5, wmin=0.0, wmax=1.0)
        rc2 = REF.topology.LocalConnection(REF.nodes.Input(n=48, traces=True), REF.nodes.LIFNodes(n=27, traces=True), kernel_size=(2, 4),
                                           stride=(2, 2), n_filters=3, input_shape=(6, 8))
        return rc.mask.bool(), rc.locations, float(rc.norm), rc2.mask.bool(), rc2.locations

    mask, locations, norm, mask2, locations2 = stored("structure", reference)
    assert torch.equal(mask, c.mask.bool()) and torch.equal(locations, c.locations)
    assert norm == pytest.approx(float(c.norm))
    # rectangular input, stride 2
    X2, Y2 = Input(n=6 * 8, traces=True), LIFNodes(n=3 * 3 * 3, traces=True)
    c2 = LocalConnection(X2, Y2, kernel_size=(2, 4), stride=(2, 2), n_filters=3, input_shape=(6, 8))
    assert torch.equal(locations2, c2.locations) and torch.equal(mask2, c2.mask.bool())


def test_boosted_lif_and_mcculloch_pitts_state_like_reference():
    from bindsnet_b200.network.nodes import BoostedLIFNodes, McCullochPitts

    l = BoostedLIFNodes(n=10, traces=True)
    l.compute_decays(1.0); l.set_batch_size(2)
    assert l.v.shape == (2, 10) and torch.all(l.v == 0) and torch.all(l.refrac_count == 0)   # nodes.py:668-678
    assert float(l.thresh) == 13.0 and float(l.decay) == float(torch.exp(-torch.tensor(1.0) / torch.tensor(100.0)))
    l.v.fill_(3.0); l.reset_state_variables()
    assert torch.all(l.v == 0)                                                              # nodes.py:649-656
    m = McCullochPitts(n=7)
    m.compute_decays(1.0); m.set_batch_size(3)
    assert m.v.shape == (3, 7) and float(m.thresh) == 1.0 and m.kind == _abi.SNN_NODE_MCP
    m.v.fill_(2.0); m.reset_state_variables()
    assert torch.all(m.v == 2.0)                                                            # nodes.py:290-295: v is not reset


def test_mstdpet_state_and_eligibility_shapes():
    net = Network(dt=1.0, batch_size=1)
    X, Y = Input(n=6, traces=True), LIFNodes(n=4, traces=True, thresh=-64.0)
    net.add_layer(X, "X"); net.add_layer(Y, "Y")
    c = Connection(X, Y, w=0.8 * torch.ones(6, 4), update_rule=MSTDPET, nu=5e-2, wmin=-1.0, wmax=1.0, tc_e_trace=10.0)
    net.add_connection(c, "X", "Y")
    with OracleBackend():
        with pytest.raises(KeyError):
            net.run({"X": torch.ones(3, 1, 6, dtype=torch.uint8)}, time=3)                 # learning.py:2218: kwargs["reward"]
        net.run({"X": torch.ones(12, 1, 6, dtype=torch.uint8)}, time=12, reward=1.0)
    r = c.update_rule
    assert r.p_plus.shape == (1, 6) and r.p_minus.shape == (1, 4) and r.eligibility_trace.shape == (6, 4) and r.eligibility.shape == (6, 4)
    assert float(r.eligibility_trace.abs().sum()) > 0 and float((c.w - 0.8).abs().sum()) > 0
