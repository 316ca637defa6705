"""Golden-vector cases: one builder per case, written against an abstract namespace ``ns`` so
that the SAME code builds the live reference network (``gen_golden.py``, ns = reference
modules) and ours (tests, ns = ``bindsnet_b200`` modules).

Each builder returns ``(network, inputs, run_kwargs)`` with every random draw taken from the
torch CPU generator seeded by the case's seed, and initial weights passed explicitly, so the
two sides start from identical state.
"""
from __future__ import annotations

from types import SimpleNamespace

import torch


def namespace(kind: str) -> SimpleNamespace:
    """``kind`` = "reference" (the original package via the stub package of SURVEY.md §8c: the checkout named by
    ``BINDSNET_REFERENCE``, else the install baseline/install_ref.sh made under baseline/_ref) or "b200" (this repo)."""
    if kind == "b200":
        import bindsnet_b200 as pkg
        from bindsnet_b200 import encoding, learning, models
        from bindsnet_b200.network import Network, monitors, nodes, topology
    else:
        import sys
        import types

        if "bindsnet" not in sys.modules:
            import os

            here = os.path.dirname(os.path.abspath(__file__))
            ref = os.path.join(os.environ.get("BINDSNET_REFERENCE", ""), "bindsnet")
            if "BINDSNET_REFERENCE" not in os.environ or not os.path.isdir(ref):
                ref = os.path.join(here, "..", "..", "baseline", "_ref", "bindsnet")
            if not os.path.isdir(ref):
                raise ImportError("the reference is neither at $BINDSNET_REFERENCE/bindsnet nor under baseline/_ref")
            pkg = types.ModuleType("bindsnet")
            pkg.__path__ = [ref]
            sys.modules["bindsnet"] = pkg
        import bindsnet.utils  # noqa: F401  (import order matters: SURVEY.md §8b)
        import bindsnet.network  # noqa: F401
        import bindsnet.learning as learning
        import bindsnet.models as models
        import bindsnet.encoding as encoding
        from bindsnet.network import Network, monitors, nodes, topology
    return SimpleNamespace(
        kind=kind, Network=Network, nodes=nodes, topology=topology, learning=learning, models=models,
        monitors=monitors, encoding=encoding,
    )


def _poisson_inputs(ns, T, B, shape, seed, active=0.19, max_rate=128.0):
    """SURVEY.md §8d synthetic input: rate image 128*U(0,1)*Bernoulli(0.19) Hz per pixel,
    Poisson-encoded with the reference's own encoder (stored in the fixture, so our side never
    regenerates it)."""
    g = torch.Generator().manual_seed(seed)
    out = []
    for _ in range(B):
        rate = max_rate * torch.rand(*shape, generator=g) * torch.bernoulli(active * torch.ones(*shape), generator=g)
        out.append(ns.encoding.poisson(datum=rate, time=T, dt=1.0))
    return torch.stack(out, dim=1).byte()


def _bernoulli_inputs(T, B, shape, p, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.bernoulli(p * torch.ones(T, B, *shape), generator=g).byte()


def _w(shape, seed, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return scale * torch.rand(*shape, generator=g)


def _set_dc_weights(net, w0):
    f = net.connections[("X", "Ae")].pipeline[0]
    with torch.no_grad():
        f.value.copy_(w0)


# ---------------------------------------------------------------------------------------------
# BASELINE.json config 1: Input(100) -> LIFNodes(100), Connection + PostPre, T=100, B=1
def c1_lif_postpre(ns, inputs=None):
    net = ns.Network(dt=1.0)
    X = ns.nodes.Input(n=100, traces=True)
    Y = ns.nodes.LIFNodes(n=100, traces=True)
    C = ns.topology.Connection(source=X, target=Y, w=_w((100, 100), 11), update_rule=ns.learning.PostPre,
                               nu=(1e-4, 1e-2), wmin=0.0, wmax=1.0)
    net.add_layer(X, "X"); net.add_layer(Y, "Y"); net.add_connection(C, "X", "Y")
    if inputs is None:
        inputs = {"X": _bernoulli_inputs(100, 1, (100,), 0.1, 12)}
    return net, inputs, {}, 100


# Same topology, batch 4, explicit sum reduction, normalisation, bias, weight decay
def lif_postpre_batch(ns, inputs=None):
    net = ns.Network(dt=1.0)
    X = ns.nodes.Input(n=80, traces=True, traces_additive=True, tc_trace=15.0, trace_scale=0.5, sum_input=True)
    Y = ns.nodes.LIFNodes(n=48, traces=True, thresh=-55.0, rest=-65.0, reset=-62.0, refrac=3, tc_decay=50.0,
                          lbound=-70.0, sum_input=True)
    C = ns.topology.Connection(source=X, target=Y, w=_w((80, 48), 21, 0.8), b=_w((48,), 22, 0.3) - 0.1,
                               update_rule=ns.learning.PostPre, nu=(2e-3, 1e-2), reduction=torch.sum,
                               weight_decay=1e-3, wmin=0.0, wmax=1.0, norm=20.0)
    net.add_layer(X, "X"); net.add_layer(Y, "Y"); net.add_connection(C, "X", "Y")
    if inputs is None:
        inputs = {"X": _bernoulli_inputs(120, 4, (80,), 0.12, 23)}
    return net, inputs, {}, 120


# Network.run(..., masks={(source, target): mask}) (network.py:279-280,449; topology.py:127-131): two connections into
# one layer, one learned + masked, one static (NoOp) + masked, plus a masked connection with learning switched off
def lif_postpre_masked(ns, inputs=None):
    net = ns.Network(dt=1.0)
    X = ns.nodes.Input(n=60, traces=True)
    Z = ns.nodes.Input(n=20, traces=True)
    Y = ns.nodes.LIFNodes(n=40, traces=True, thresh=-57.0, refrac=2)
    C1 = ns.topology.Connection(source=X, target=Y, w=_w((60, 40), 51, 0.9), update_rule=ns.learning.PostPre, nu=(2e-3, 2e-2),
                                reduction=torch.sum, wmin=0.0, wmax=1.0, norm=15.0)
    C2 = ns.topology.Connection(source=Z, target=Y, w=_w((20, 40), 52, 0.5))
    net.add_layer(X, "X"); net.add_layer(Z, "Z"); net.add_layer(Y, "Y")
    net.add_connection(C1, "X", "Y"); net.add_connection(C2, "Z", "Y")
    g = torch.Generator().manual_seed(53)
    masks = {("X", "Y"): torch.bernoulli(0.3 * torch.ones(60, 40), generator=g).bool(),
             ("Z", "Y"): torch.bernoulli(0.5 * torch.ones(20, 40), generator=g).bool()}
    if inputs is None:
        inputs = {"X": _bernoulli_inputs(90, 3, (60,), 0.15, 54), "Z": _bernoulli_inputs(90, 3, (20,), 0.2, 55)}
    return net, inputs, {"masks": masks}, 90


# the other neuron models of the generic tier (SURVEY.md §8f rank 4): IFNodes (nodes.py:308-415), CurrentLIFNodes
# (nodes.py:681-826), AdaptiveLIFNodes (nodes.py:829-978), each as the target of a learned connection
def _one_layer_model(ns, layer, w_seed, in_seed, T=90, B=3, n_in=70):
    net = ns.Network(dt=1.0)
    X = ns.nodes.Input(n=n_in, traces=True)
    C = ns.topology.Connection(source=X, target=layer, w=_w((n_in, layer.n), w_seed, 1.2), update_rule=ns.learning.PostPre,
                               nu=(2e-3, 2e-2), reduction=torch.sum, wmin=0.0, wmax=1.5, norm=18.0)
    net.add_layer(X, "X"); net.add_layer(layer, "Y"); net.add_connection(C, "X", "Y")
    return net, {"X": _bernoulli_inputs(T, B, (n_in,), 0.15, in_seed)}, {}, T


def if_postpre(ns, inputs=None):
    Y = ns.nodes.IFNodes(n=36, traces=True, sum_input=True, thresh=-50.0, reset=-64.0, refrac=3, lbound=-66.0)
    net, x, kw, T = _one_layer_model(ns, Y, 61, 62)
    return net, (inputs or x), kw, T


def clif_postpre(ns, inputs=None):
    Y = ns.nodes.CurrentLIFNodes(n=36, traces=True, thresh=-55.0, rest=-65.0, reset=-63.0, refrac=2, tc_decay=40.0, tc_i_decay=3.0)
    net, x, kw, T = _one_layer_model(ns, Y, 63, 64)
    return net, (inputs or x), kw, T


def alif_postpre(ns, inputs=None):
    Y = ns.nodes.AdaptiveLIFNodes(n=36, traces=True, thresh=-56.0, rest=-65.0, reset=-62.0, refrac=2, tc_decay=50.0, theta_plus=0.4,
                                  tc_theta_decay=200.0, lbound=-68.0)
    net, x, kw, T = _one_layer_model(ns, Y, 65, 66)
    return net, (inputs or x), kw, T


# BoostedLIFNodes (nodes.py:562-678) and McCullochPitts (nodes.py:231-305) as learned targets; the McCulloch-Pitts layer
# also drives a second population, so its spikes are exercised as a source
def boosted_postpre(ns, inputs=None):
    Y = ns.nodes.BoostedLIFNodes(n=36, traces=True, sum_input=True, thresh=9.0, refrac=3, tc_decay=30.0)
    net, x, kw, T = _one_layer_model(ns, Y, 67, 68)
    return net, (inputs or x), kw, T


def mcp_postpre(ns, inputs=None):
    Y = ns.nodes.McCullochPitts(n=36, traces=True, sum_input=True, thresh=7.0)
    net, x, kw, T = _one_layer_model(ns, Y, 69, 70)
    Z = ns.nodes.LIFNodes(n=20, traces=True, thresh=-58.0, rest=-65.0, reset=-64.0, refrac=2, tc_decay=60.0)
    C2 = ns.topology.Connection(source=Y, target=Z, w=_w((36, 20), 71, 3.0), update_rule=ns.learning.PostPre, nu=(1e-3, 1e-2),
                                reduction=torch.sum, wmin=0.0, wmax=4.0)
    net.add_layer(Z, "Z"); net.add_connection(C2, "Y", "Z")
    return net, (inputs or x), kw, T


# LocalConnection (topology.py:1304-1484): dense weights confined to receptive fields by the connection's own mask,
# plain-sum normalisation scaled by the kernel size.  Batch size 1: the reference's compute views the result as
# target.shape (topology.py:1455), which fails for larger batches
def local_postpre(ns, inputs=None):
    T, B = 120, 1
    net = ns.Network(dt=1.0)
    X = ns.nodes.Input(n=64, traces=True)
    Y = ns.nodes.LIFNodes(n=72, traces=True, thresh=-60.0, rest=-65.0, reset=-64.0, refrac=2, tc_decay=50.0)
    probe = ns.topology.LocalConnection(X, Y, kernel_size=3, stride=1, n_filters=2)      # default init: only its mask is used
    w = _w((64, 72), 73, 0.9) * (~probe.mask.bool()).float()
    C = ns.topology.LocalConnection(X, Y, kernel_size=3, stride=1, n_filters=2, w=w, update_rule=ns.learning.PostPre, nu=(2e-3, 2e-2),
                                    reduction=torch.sum, wmin=0.0, wmax=1.0, norm=0.35)
    net.add_layer(X, "X"); net.add_layer(Y, "Y"); net.add_connection(C, "X", "Y")
    return net, (inputs or {"X": _bernoulli_inputs(T, B, (64,), 0.2, 74)}), {}, T


# WeightDependentPostPre, mean reduction
def lif_wdep(ns, inputs=None):
    net = ns.Network(dt=1.0)
    X = ns.nodes.Input(n=64, traces=True)
    Y = ns.nodes.LIFNodes(n=32, traces=True, thresh=-58.0)
    C = ns.topology.Connection(source=X, target=Y, w=_w((64, 32), 31, 0.9),
                               update_rule=ns.learning.WeightDependentPostPre, nu=(1e-2, 5e-2),
                               reduction=torch.mean, wmin=0.0, wmax=1.0)
    net.add_layer(X, "X"); net.add_layer(Y, "Y"); net.add_connection(C, "X", "Y")
    if inputs is None:
        inputs = {"X": _bernoulli_inputs(100, 4, (64,), 0.15, 32)}
    return net, inputs, {}, 100


# clamp / unclamp / injects_v run-kwargs, two stacked LIF layers, NoOp connection with decay
def lif_clamps(ns, inputs=None):
    net = ns.Network(dt=1.0)
    X = ns.nodes.Input(n=40, traces=True)
    H = ns.nodes.LIFNodes(n=24, traces=True, thresh=-60.0)
    O = ns.nodes.LIFNodes(n=10, traces=True, thresh=-62.0, refrac=2)
    C1 = ns.topology.Connection(source=X, target=H, w=_w((40, 24), 41, 1.5), update_rule=ns.learning.PostPre,
                                nu=(1e-3, 1e-2), reduction=torch.sum, wmin=0.0, wmax=2.0)
    C2 = ns.topology.Connection(source=H, target=O, w=_w((24, 10), 42, 3.0) - 0.5, weight_decay=5e-3)
    net.add_layer(X, "X"); net.add_layer(H, "H"); net.add_layer(O, "O")
    net.add_connection(C1, "X", "H"); net.add_connection(C2, "H", "O")
    T = 60
    g = torch.Generator().manual_seed(43)
    kw = {
        "clamp": {"O": torch.bernoulli(0.05 * torch.ones(T, 10), generator=g).bool()},
        "unclamp": {"H": (torch.arange(24) % 5 == 0)},
        "injects_v": {"H": 0.5 * torch.rand(T, 24, generator=g), "O": 0.2 * torch.rand(10, generator=g)},
    }
    if inputs is None:
        inputs = {"X": _bernoulli_inputs(T, 3, (40,), 0.2, 44)}
    return net, inputs, kw, T


def _dc2015(ns, n, B, T, inp_seed, w_seed, one_spike, inputs, inh=120.0, poisson=False):
    net = ns.models.DiehlAndCook2015(n_inpt=784, n_neurons=n, batch_size=B, inpt_shape=(1, 28, 28), dt=1.0,
                                     nu=(1e-4, 1e-2), norm=78.4, theta_plus=0.05, exc=22.5, inh=inh)
    _set_dc_weights(net, _w((784, n), w_seed, 0.3))
    net.layers["Ae"].one_spike = one_spike
    if inputs is None:
        if poisson:
            inputs = {"X": _poisson_inputs(ns, T, B, (1, 28, 28), inp_seed)}
        else:
            inputs = {"X": _bernoulli_inputs(T, B, (1, 28, 28), 0.05, inp_seed)}
    return net, inputs, {}, T


# SURVEY.md §0.10 configuration: deterministic dynamics (one_spike off)
def dc2015_multi(ns, inputs=None):
    return _dc2015(ns, 64, 8, 120, 51, 52, False, inputs)


# default one_spike=True, tie-break via the shared hash
def dc2015_onespike(ns, inputs=None):
    return _dc2015(ns, 100, 16, 150, 61, 62, True, inputs)


# BASELINE.json config 2: n=400, B=32, T=250, Poisson 28x28
def dc2015_c2(ns, inputs=None):
    return _dc2015(ns, 400, 32, 250, 71, 72, True, inputs, poisson=True)


# metric configuration n=1600, B=128, shortened to T=40 (the live reference needs ~2 s/step)
def dc2015_metric_t40(ns, inputs=None):
    return _dc2015(ns, 1600, 128, 40, 81, 82, True, inputs, poisson=True)


# the metric configuration at its full window length: n=1600, B=128, T=250 (north_star: "final weights within 1e-4
# rel of reference under fixed seed" at 250 steps; one ~5-minute run of the live reference)
def dc2015_metric_t250(ns, inputs=None):
    return _dc2015(ns, 1600, 128, 250, 83, 84, True, inputs, poisson=True)


# classic Connection + learning.PostPre path with a recurrent inhibitory Connection
def dc2015v2(ns, inputs=None):
    net = ns.models.DiehlAndCook2015v2(n_inpt=196, n_neurons=64, inh=60.0, nu=(1e-4, 1e-2), reduction=torch.sum,
                                       norm=30.0, inpt_shape=(1, 14, 14))
    with torch.no_grad():
        net.connections[("X", "Y")].w.copy_(_w((196, 64), 91, 0.3))
    if inputs is None:
        inputs = {"X": _bernoulli_inputs(120, 4, (1, 14, 14), 0.08, 92)}
    return net, inputs, {}, 120


# learning switched off (network.train(False)): no STDP, no theta adaptation
def dc2015_eval(ns, inputs=None):
    net, inputs, kw, T = _dc2015(ns, 49, 5, 80, 101, 102, True, inputs)
    net.train(False)
    with torch.no_grad():
        g = torch.Generator().manual_seed(103)
        net.layers["Ae"].theta.copy_(2.0 * torch.rand(49, generator=g))
    return net, inputs, kw, T


# Reward-modulated STDP on a dense Connection (learning.MSTDP._connection_update, learning.py:1504-1574)
def mstdp_dense(ns, inputs=None):
    net = ns.Network(dt=1.0, batch_size=3)
    X = ns.nodes.Input(n=60, traces=True)
    Y = ns.nodes.LIFNodes(n=20, traces=True, thresh=-62.0, refrac=2)
    net.add_layer(X, "X"); net.add_layer(Y, "Y")
    C = ns.topology.Connection(source=X, target=Y, w=_w((60, 20), 111, 1.2) - 0.2, update_rule=ns.learning.MSTDP,
                               nu=5e-2, reduction=torch.sum, wmin=-1.0, wmax=1.5, tc_plus=15.0, tc_minus=25.0)
    net.add_connection(C, "X", "Y")
    if inputs is None:
        inputs = {"X": _bernoulli_inputs(80, 3, (60,), 0.12, 112)}
    return net, inputs, {"reward": 0.7, "a_plus": 0.9, "a_minus": -1.1}, 80


# MSTDPET on a dense connection (learning.py:2187-2249): eligibility trace, batch size 1 (the only one the reference's
# flattened traces support), weight decay and clamp through the base class
def mstdpet_dense(ns, inputs=None):
    net = ns.Network(dt=1.0, batch_size=1)
    X = ns.nodes.Input(n=60, traces=True)
    Y = ns.nodes.LIFNodes(n=20, traces=True, thresh=-62.0, refrac=2)
    net.add_layer(X, "X"); net.add_layer(Y, "Y")
    C = ns.topology.Connection(source=X, target=Y, w=_w((60, 20), 113, 1.2) - 0.2, update_rule=ns.learning.MSTDPET,
                               nu=8e-2, reduction=torch.sum, wmin=-1.0, wmax=1.5, tc_plus=15.0, tc_minus=25.0, tc_e_trace=12.0,
                               weight_decay=1e-3)
    net.add_connection(C, "X", "Y")
    if inputs is None:
        inputs = {"X": _bernoulli_inputs(120, 1, (60,), 0.12, 114)}
    return net, inputs, {"reward": 0.8, "a_plus": 0.9, "a_minus": -1.1}, 120


def _conv_net(ns, B, T, in_shape, out_ch, k, stride, padding, rule, seeds, n_out=6, norm=None, conv_nu=1e-2):
    """BASELINE.json config 4 in small: Input[C,H,W] -> Conv2dConnection -> LIFNodes[Co,Ho,Wo] -> Connection ->
    LIFNodes(n_out), MSTDP on both connections (or no rule), weights in [-1, 1]."""
    cin, hin, win = in_shape
    ho = (hin - k + 2 * padding) // stride + 1
    wo = (win - k + 2 * padding) // stride + 1
    net = ns.Network(dt=1.0, batch_size=B)
    X = ns.nodes.Input(shape=[cin, hin, win], traces=True)
    H = ns.nodes.LIFNodes(shape=[out_ch, ho, wo], traces=True, thresh=-63.5, refrac=2, tc_decay=60.0)
    O = ns.nodes.LIFNodes(n=n_out, traces=True, thresh=-62.0, refrac=3)
    net.add_layer(X, "X"); net.add_layer(H, "H"); net.add_layer(O, "O")
    kw = dict(update_rule=rule, nu=conv_nu, reduction=torch.sum) if rule is not None else {}
    conv = ns.topology.Conv2dConnection(source=X, target=H, kernel_size=k, stride=stride, padding=padding,
                                        w=_w((out_ch, cin, k, k), seeds[0], 1.0) - 0.2, wmin=-1.0, wmax=1.0, norm=norm, **kw)
    dense = ns.topology.Connection(source=H, target=O, w=_w((out_ch * ho * wo, n_out), seeds[1], 0.5) - 0.1,
                                   wmin=-1.0, wmax=1.0, **kw)
    net.add_connection(conv, "X", "H"); net.add_connection(dense, "H", "O")
    return net


# conv + dense MSTDP, batch 4 (per-sample eligibility: SURVEY.md §0.8 / §8c — the reference is run with
# the one-line fix of learning.py:2013 that gen_golden.py applies)
def conv_mstdp(ns, inputs=None):
    net = _conv_net(ns, 4, 60, (1, 12, 12), 4, 3, 1, 0, ns.learning.MSTDP, (121, 122))
    if inputs is None:
        inputs = {"X": _bernoulli_inputs(60, 4, (1, 12, 12), 0.1, 123)}
    return net, inputs, {"reward": 1.0}, 60


# conv geometry: two input channels, stride 2, padding 1, filter normalisation, no learning rule
def conv_stride_norm(ns, inputs=None):
    net = _conv_net(ns, 2, 40, (2, 9, 9), 3, 3, 2, 1, None, (131, 132), n_out=5, norm=1.5)
    if inputs is None:
        inputs = {"X": _bernoulli_inputs(40, 2, (2, 9, 9), 0.15, 133)}
    return net, inputs, {}, 40


# BASELINE.json config 4 at full geometry (Input[1,32,32] -conv k5 s1-> LIFNodes[16,28,28] -> Connection ->
# LIFNodes(10), MSTDP nu=1e-2 on both, w in [-1,1] drawn like the constructors do, reward 1, Bernoulli(0.1)
# input), batch 8 and 40 steps to keep the live reference and the fixture small
def conv_mstdp_c4(ns, inputs=None, B=8, T=40, in_seed=143):
    net = ns.Network(dt=1.0, batch_size=B)
    X = ns.nodes.Input(shape=[1, 32, 32], traces=True)
    H = ns.nodes.LIFNodes(shape=[16, 28, 28], traces=True)
    O = ns.nodes.LIFNodes(n=10, traces=True)
    net.add_layer(X, "X"); net.add_layer(H, "H"); net.add_layer(O, "O")
    conv = ns.topology.Conv2dConnection(source=X, target=H, kernel_size=5, stride=1, w=2.0 * _w((16, 1, 5, 5), 141) - 1.0,
                                        update_rule=ns.learning.MSTDP, nu=1e-2, reduction=torch.sum, wmin=-1.0, wmax=1.0)
    dense = ns.topology.Connection(source=H, target=O, w=2.0 * _w((16 * 28 * 28, 10), 142) - 1.0,
                                   update_rule=ns.learning.MSTDP, nu=1e-2, reduction=torch.sum, wmin=-1.0, wmax=1.0)
    net.add_connection(conv, "X", "H"); net.add_connection(dense, "H", "O")
    if inputs is None:
        inputs = {"X": _bernoulli_inputs(T, B, (1, 32, 32), 0.1, in_seed)}
    return net, inputs, {"reward": 1.0}, T


# BASELINE.json config 4 at its full batch size: B=128 (T shortened to 24; the live reference, with the per-sample
# eligibility view of SURVEY.md §0.8, runs ~1 K sample*timesteps/s)
def conv_mstdp_c4_b128(ns, inputs=None):
    return conv_mstdp_c4(ns, inputs, B=128, T=24, in_seed=145)


# Network.run(one_step=True) (network.py:383-396): feed-forward mode — every layer's input is recomputed from
# the current spikes of its sources just before its forward.  Includes a backward connection (source later in
# the insertion order: previous-step spikes) and an external current on a layer that also has incoming
# connections (the reference's dict.update drops it in this mode).
def one_step_ff(ns, inputs=None):
    net = ns.Network(dt=1.0, batch_size=3)
    X = ns.nodes.Input(n=40, traces=True)
    H = ns.nodes.LIFNodes(n=24, traces=True, thresh=-60.0)
    O = ns.nodes.LIFNodes(n=10, traces=True, thresh=-61.0, refrac=2)
    net.add_layer(X, "X"); net.add_layer(H, "H"); net.add_layer(O, "O")
    c1 = ns.topology.Connection(source=X, target=H, w=_w((40, 24), 151, 1.6), update_rule=ns.learning.PostPre,
                                nu=(1e-3, 1e-2), reduction=torch.sum, wmin=0.0, wmax=2.0)
    c2 = ns.topology.Connection(source=H, target=O, w=_w((24, 10), 152, 2.5), update_rule=ns.learning.PostPre,
                                nu=(1e-3, 1e-2), reduction=torch.sum, wmin=0.0, wmax=3.0)
    c3 = ns.topology.Connection(source=O, target=H, w=-_w((10, 24), 153, 1.5))
    net.add_connection(c1, "X", "H"); net.add_connection(c2, "H", "O"); net.add_connection(c3, "O", "H")
    T = 70
    if inputs is None:
        g = torch.Generator().manual_seed(155)
        inputs = {"X": _bernoulli_inputs(T, 3, (40,), 0.2, 154), "H": 0.8 * torch.rand(T, 3, 24, generator=g)}
    return net, inputs, {"one_step": True}, T


# MSTDP with mean reduction, weight decay and a negative reward
def mstdp_mean_decay(ns, inputs=None):
    net = ns.Network(dt=1.0, batch_size=4)
    X = ns.nodes.Input(n=30, traces=True)
    Y = ns.nodes.LIFNodes(n=12, traces=True, thresh=-62.5, refrac=1)
    net.add_layer(X, "X"); net.add_layer(Y, "Y")
    C = ns.topology.Connection(source=X, target=Y, w=_w((30, 12), 161, 1.5), update_rule=ns.learning.MSTDP,
                               nu=3e-2, reduction=torch.mean, weight_decay=2e-3, wmin=-0.5, wmax=1.6)
    net.add_connection(C, "X", "Y")
    if inputs is None:
        inputs = {"X": _bernoulli_inputs(50, 4, (30,), 0.2, 162)}
    return net, inputs, {"reward": -0.5}, 50


# strided convolution with a non-zero bias, no learning rule (dilation > 1 cannot be constructed: the reference's
# shape assertion, topology.py:752-772, ignores it)
def conv_bias_stride(ns, inputs=None):
    net = ns.Network(dt=1.0, batch_size=2)
    X = ns.nodes.Input(shape=[1, 11, 11], traces=True)
    H = ns.nodes.LIFNodes(shape=[2, 5, 5], traces=True, thresh=-63.0)
    net.add_layer(X, "X"); net.add_layer(H, "H")
    conv = ns.topology.Conv2dConnection(source=X, target=H, kernel_size=3, stride=2, padding=0,
                                        w=_w((2, 1, 3, 3), 171, 1.2) - 0.2, b=torch.tensor([0.25, -0.1]), wmin=-1.0, wmax=1.0)
    net.add_connection(conv, "X", "H")
    if inputs is None:
        inputs = {"X": _bernoulli_inputs(30, 2, (1, 11, 11), 0.15, 172)}
    return net, inputs, {}, 30


# edge sizes: one sample, one timestep; and a window without a single input spike
def dc2015_b1_t1(ns, inputs=None):
    net, inputs, kw, _ = _dc2015(ns, 36, 1, 1, 181, 182, True, inputs)
    return net, inputs, kw, 1


def dc2015_silent(ns, inputs=None):
    if inputs is None:
        inputs = {"X": torch.zeros(12, 3, 1, 28, 28, dtype=torch.uint8)}
    net, inputs, kw, _ = _dc2015(ns, 40, 3, 12, 191, 192, True, inputs)
    return net, inputs, kw, 12


# Hebbian on a dense Connection (learning.py:1110-1136): both terms positive, nu after the batch reduction; weight decay
def hebbian_dense(ns, inputs=None):
    net = ns.Network(dt=1.0)
    X = ns.nodes.Input(n=64, traces=True)
    Y = ns.nodes.LIFNodes(n=32, traces=True, thresh=-58.0, refrac=2)
    C = ns.topology.Connection(source=X, target=Y, w=_w((64, 32), 151, 0.6), update_rule=ns.learning.Hebbian, nu=(1e-3, 4e-3),
                               reduction=torch.mean, weight_decay=2e-3, wmin=0.0, wmax=1.0)
    net.add_layer(X, "X"); net.add_layer(Y, "Y"); net.add_connection(C, "X", "Y")
    if inputs is None:
        inputs = {"X": _bernoulli_inputs(100, 4, (64,), 0.15, 152)}
    return net, inputs, {}, 100


# PostPre / WeightDependentPostPre / Hebbian on a Conv2dConnection (learning.py:457-497, 920-975, 1348-1380) feeding a
# dense connection under the same rule
def conv_postpre(ns, inputs=None):
    net = _conv_net(ns, 3, 50, (1, 10, 10), 3, 3, 1, 0, ns.learning.PostPre, (161, 162), conv_nu=(4e-3, 2e-2))
    if inputs is None:
        inputs = {"X": _bernoulli_inputs(50, 3, (1, 10, 10), 0.12, 163)}
    return net, inputs, {}, 50


def conv_wdep(ns, inputs=None):
    net = _conv_net(ns, 2, 50, (2, 9, 9), 3, 3, 2, 1, ns.learning.WeightDependentPostPre, (171, 172), n_out=5, conv_nu=(1e-2, 3e-2))
    if inputs is None:
        inputs = {"X": _bernoulli_inputs(50, 2, (2, 9, 9), 0.15, 173)}
    return net, inputs, {}, 50


def conv_hebbian(ns, inputs=None):
    net = _conv_net(ns, 3, 50, (1, 10, 10), 4, 3, 1, 1, ns.learning.Hebbian, (181, 182), conv_nu=(1e-3, 2e-3))
    if inputs is None:
        inputs = {"X": _bernoulli_inputs(50, 3, (1, 10, 10), 0.12, 183)}
    return net, inputs, {}, 50


CASES = {
    "c1_lif_postpre": c1_lif_postpre,
    "lif_postpre_batch": lif_postpre_batch,
    "lif_wdep": lif_wdep,
    "lif_postpre_masked": lif_postpre_masked,
    "if_postpre": if_postpre,
    "clif_postpre": clif_postpre,
    "alif_postpre": alif_postpre,
    "boosted_postpre": boosted_postpre,
    "local_postpre": local_postpre,
    "mstdpet_dense": mstdpet_dense,
    "mcp_postpre": mcp_postpre,
    "lif_clamps": lif_clamps,
    "dc2015_multi": dc2015_multi,
    "dc2015_onespike": dc2015_onespike,
    "dc2015v2": dc2015v2,
    "dc2015_eval": dc2015_eval,
    "dc2015_c2": dc2015_c2,
    "dc2015_metric_t40": dc2015_metric_t40,
    "dc2015_metric_t250": dc2015_metric_t250,
    "mstdp_dense": mstdp_dense,
    "conv_mstdp": conv_mstdp,
    "conv_stride_norm": conv_stride_norm,
    "conv_mstdp_c4": conv_mstdp_c4,
    "conv_mstdp_c4_b128": conv_mstdp_c4_b128,
    "one_step_ff": one_step_ff,
    "mstdp_mean_decay": mstdp_mean_decay,
    "conv_bias_stride": conv_bias_stride,
    "dc2015_b1_t1": dc2015_b1_t1,
    "dc2015_silent": dc2015_silent,
    "hebbian_dense": hebbian_dense,
    "conv_postpre": conv_postpre,
    "conv_wdep": conv_wdep,
    "conv_hebbian": conv_hebbian,
}

#: cases whose fixture stores subsampled weights only (full tensors would be several MB)
LARGE = {"dc2015_metric_t40", "dc2015_metric_t250", "conv_mstdp_c4", "conv_mstdp_c4_b128"}
#: one_spike tie-break seed used by every case
ONE_SPIKE_SEED = 20260922
