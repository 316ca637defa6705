"""The drop-in boundary driven from the REFERENCE's own objects (VERDICT r1 item 9): a live ``bindsnet`` network —
``bindsnet.models.DiehlAndCook2015`` (MulticompartmentConnection + Weight + MCC PostPre) and a classic
``Connection`` + ``learning.PostPre`` network — is described through ``include/snn_b200.h`` by
``bindsnet_b200.reference_binding`` (no bindsnet_b200 host classes) and run by the oracle library on the CPU; the
result must equal what the reference's own ``Network.run`` computes on a twin network.  These tests need the original
package itself (stored results cannot stand in for its objects), so they skip unless it is importable: a checkout named
by ``BINDSNET_REFERENCE``, or the install baseline/install_ref.sh makes under baseline/_ref (never part of a checkout)."""
import os
import sys

import numpy as np
import pytest
import torch

import cases

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))

try:
    REF = cases.namespace("reference")
except Exception as e:  # pragma: no cover
    REF = None
    WHY = str(e)

pytestmark = pytest.mark.skipif(REF is None, reason="live reference not available")


def _state(net):
    out = {}
    for name, layer in net.layers.items():
        B = layer.s.shape[0]
        out[f"{name}/s"] = layer.s.reshape(B, -1).to(torch.uint8).numpy().copy()
        for var in ("v", "refrac_count", "x", "theta"):
            val = getattr(layer, var, None)
            if isinstance(val, torch.Tensor) and val.numel():
                out[f"{name}/{var}"] = val.detach().float().reshape(-1).numpy().copy()
    for (s, t), c in net.connections.items():
        w = c.pipeline[0].value if hasattr(c, "pipeline") else c.w
        out[f"{s}->{t}/w"] = w.detach().float().numpy().copy()
    return out


def _compare(a, b):
    assert a.keys() == b.keys()
    for k in a:
        if k.endswith("/s"):
            assert np.array_equal(a[k], b[k]), f"{k}: final spikes differ"
        elif k.endswith("/w"):
            err = np.abs(a[k] - b[k]).max() / max(np.abs(a[k]).max(), 1e-12)
            assert err <= 1e-4, f"{k}: max rel err {err:.3e}"          # north_star: weights within 1e-4 relative
        else:
            bad = np.abs(a[k] - b[k]) > 1e-4 + 1e-5 * np.abs(a[k])
            assert not bad.any(), f"{k}: max |d| {np.abs(a[k] - b[k]).max():.3e}"


def _twin(build):
    torch.manual_seed(11)
    a = build()
    torch.manual_seed(11)
    b = build()
    for (ka, ca), (kb, cb) in zip(a.connections.items(), b.connections.items()):
        wa = ca.pipeline[0].value if hasattr(ca, "pipeline") else ca.w
        wb = cb.pipeline[0].value if hasattr(cb, "pipeline") else cb.w
        assert torch.equal(wa, wb)
    return a, b


def _run_both(a, b, x, T):
    import gen_golden
    from bindsnet_b200 import reference_binding as rb
    from oracle import oracle

    with gen_golden.OneSpikePatch(a, cases.ONE_SPIKE_SEED):       # the reference's multinomial -> the shared tie-break hash
        a.run(inputs={"X": x.clone()}, time=T)
    rc = rb.run_window(b, {"X": x.clone()}, time=T, seed=cases.ONE_SPIKE_SEED, library=oracle.lib())
    assert rc == 0
    _compare(_state(a), _state(b))


def test_abi_filled_from_reference_diehlandcook2015_matches_reference_run():
    def build():
        return REF.models.DiehlAndCook2015(n_inpt=784, n_neurons=48, batch_size=6, inpt_shape=(1, 28, 28), dt=1.0, nu=(1e-4, 1e-2),
                                           norm=78.4, theta_plus=0.05, exc=22.5, inh=120.0)

    a, b = _twin(build)
    x = cases._poisson_inputs(REF, 80, 6, (1, 28, 28), 31)
    _run_both(a, b, x, 80)
    # second window on the same objects (state carried over, theta adapted): still in step
    x2 = cases._poisson_inputs(REF, 40, 6, (1, 28, 28), 32)
    _run_both(a, b, x2, 40)


def test_abi_filled_from_reference_connection_postpre_matches_reference_run():
    def build():
        net = REF.Network(dt=1.0, batch_size=5)
        X = REF.nodes.Input(n=100, traces=True)
        Y = REF.nodes.LIFNodes(n=60, traces=True, thresh=-55.0)
        c = REF.topology.Connection(X, Y, w=0.3 * torch.rand(100, 60), update_rule=REF.learning.PostPre, nu=(1e-3, 1e-2),
                                    reduction=torch.sum, wmin=0.0, wmax=1.0, norm=12.0)
        net.add_layer(X, "X"); net.add_layer(Y, "Y")
        net.add_connection(c, "X", "Y")
        return net

    a, b = _twin(build)
    x = cases._bernoulli_inputs(70, 5, (100,), 0.15, 8)
    _run_both(a, b, x, 70)


@pytest.mark.parametrize("kind", ["IFNodes", "CurrentLIFNodes", "AdaptiveLIFNodes", "BoostedLIFNodes", "McCullochPitts"])
def test_abi_filled_from_the_other_reference_neuron_models(kind):
    """The remaining node kinds of the ABI, each as the learned target of a reference ``Connection`` + ``PostPre``."""
    def build():
        net = REF.Network(dt=1.0, batch_size=3)
        X = REF.nodes.Input(n=70, traces=True)
        kw = dict(IFNodes=dict(thresh=-50.0, reset=-64.0, refrac=3, lbound=-66.0),
                  CurrentLIFNodes=dict(thresh=-55.0, rest=-65.0, reset=-63.0, refrac=2, tc_decay=40.0, tc_i_decay=3.0),
                  AdaptiveLIFNodes=dict(thresh=-56.0, rest=-65.0, reset=-62.0, refrac=2, tc_decay=50.0, theta_plus=0.4, tc_theta_decay=200.0),
                  BoostedLIFNodes=dict(thresh=9.0, refrac=3, tc_decay=30.0),
                  McCullochPitts=dict(thresh=7.0))[kind]
        Y = getattr(REF.nodes, kind)(n=36, traces=True, **kw)
        c = REF.topology.Connection(X, Y, w=1.2 * torch.rand(70, 36), update_rule=REF.learning.PostPre, nu=(2e-3, 2e-2),
                                    reduction=torch.sum, wmin=0.0, wmax=1.5, norm=18.0)
        net.add_layer(X, "X"); net.add_layer(Y, "Y")
        net.add_connection(c, "X", "Y")
        return net

    a, b = _twin(build)
    x = cases._bernoulli_inputs(90, 3, (70,), 0.15, 62)
    _run_both(a, b, x, 90)
    assert int(a.layers["Y"].s.sum()) >= 0 and float(a.connections[("X", "Y")].w.sum()) > 0


def test_abi_filled_from_reference_localconnection_matches_reference_run():
    """``LocalConnection`` (topology.py:1304-1484): the binding passes the connection's own mask and the plain-sum
    normalisation; batch size 1, the only one the reference's ``compute`` supports (:1455)."""
    def build():
        net = REF.Network(dt=1.0, batch_size=1)
        X = REF.nodes.Input(n=64, traces=True)
        Y = REF.nodes.LIFNodes(n=72, traces=True, thresh=-60.0, rest=-65.0, reset=-64.0, refrac=2, tc_decay=50.0)
        probe = REF.topology.LocalConnection(X, Y, kernel_size=3, stride=1, n_filters=2)
        w = 0.9 * torch.rand(64, 72) * (~probe.mask.bool()).float()
        c = REF.topology.LocalConnection(X, Y, kernel_size=3, stride=1, n_filters=2, w=w, update_rule=REF.learning.PostPre, nu=(2e-3, 2e-2),
                                         reduction=torch.sum, wmin=0.0, wmax=1.0, norm=0.35)
        net.add_layer(X, "X"); net.add_layer(Y, "Y")
        net.add_connection(c, "X", "Y")
        return net

    a, b = _twin(build)
    x = cases._bernoulli_inputs(100, 1, (64,), 0.2, 74)
    _run_both(a, b, x, 100)
