"""``Network(reward_fn=...)`` (reference: network.py:114-117, 325-326; learning/reward.py): the reward a window's
MSTDP kernels are launched with is the reward_fn's ``compute`` of the run's kwargs.  Three episodes of a dense MSTDP
network with ``MovingAvgRPE`` through the reference (its results stored under tests/golden/live) and through our host
API on the oracle: same prediction state, same spikes, weights within the north_star's 1e-4.  CPU only; a GPU twin runs
the same episodes on the kernels against the oracle bit for bit
(tests/test_zz_gpu_late_additions.py)."""
import importlib

import numpy as np
import pytest
import torch

import cases
import helpers
from live import REF, stored

T, B = 60, 3
REWARDS = (0.9, -0.4, 1.3)


def _net(ns, reward_cls, rule="MSTDP", B=B):
    g = torch.Generator().manual_seed(4242)
    net = ns.Network(dt=1.0, batch_size=B, reward_fn=reward_cls)
    X = ns.nodes.Input(n=50, traces=True)
    Y = ns.nodes.LIFNodes(n=16, traces=True, thresh=-62.0, refrac=2)
    net.add_layer(X, "X"); net.add_layer(Y, "Y")
    w = 1.3 * torch.rand(50, 16, generator=g) - 0.2
    net.add_connection(ns.topology.Connection(source=X, target=Y, w=w, update_rule=getattr(ns.learning, rule), nu=4e-2,
                                              reduction=torch.sum, wmin=-1.0, wmax=1.5, tc_plus=15.0, tc_minus=25.0), "X", "Y")
    xs = [torch.bernoulli(0.12 * torch.ones(T, B, 50), generator=g).byte() for _ in REWARDS]
    return net, xs


def _episodes(net, xs, run):
    seen = []
    for r, x in zip(REWARDS, xs):
        run(net, x, r)
        net.reward_fn.update(accumulated_reward=torch.tensor(r * T), steps=T, ema_window=4.0)
        seen.append((float(net.reward_fn.reward_predict), float(net.reward_fn.reward_predict_episode)))
    return seen


def _plain_run(net, x, r):
    net.run(inputs={"X": x}, time=T, reward=r, a_plus=0.9, a_minus=-1.1)


def test_reward_fn_matches_live_reference():
    from bindsnet_b200.learning.reward import MovingAvgRPE
    from oracle.oracle import OracleBackend

    def reference():
        ref, xs = _net(REF, importlib.import_module("bindsnet.learning.reward").MovingAvgRPE)
        seen = _episodes(ref, [x.clone() for x in xs], _plain_run)
        return seen, ref.layers["Y"].s, ref.connections[("X", "Y")].w.detach()

    seen_ref, s_ref, w_ref = stored("episodes", reference)

    ours, xs2 = _net(cases.namespace("b200"), MovingAvgRPE)
    assert isinstance(ours.reward_fn, MovingAvgRPE)
    with OracleBackend() as ob:
        seen = _episodes(ours, xs2, _plain_run)
        assert ob.err == 0

    assert seen == seen_ref, (seen, seen_ref)                      # same fp32 arithmetic: equal, not close
    assert seen[0][0] != 0.0 and len(ours.reward_fn.rewards_predict_episode) == len(REWARDS)
    assert np.array_equal(s_ref.numpy(), ours.layers["Y"].s.numpy())
    wa = w_ref.numpy()
    wb = ours.connections[("X", "Y")].w.detach().numpy()
    assert np.abs(wa - wb).max() > -1 and not (np.abs(wa - wb) > 2e-6 + 1e-4 * np.abs(wa)).any(), np.abs(wa - wb).max()
    # the reward_fn changed what was learnt: the same episodes without it end elsewhere
    plain, xs3 = _net(cases.namespace("b200"), None)
    with OracleBackend():
        for r, x in zip(REWARDS, xs3):
            _plain_run(plain, x, r)
    assert np.abs(plain.connections[("X", "Y")].w.detach().numpy() - wb).max() > 1e-3


def test_a_user_defined_reward_class_is_instantiated_and_asked_per_window():
    from bindsnet_b200.learning.reward import AbstractReward
    from oracle.oracle import OracleBackend

    calls = []

    class Halved(AbstractReward):
        def compute(self, **kwargs):
            calls.append(sorted(kwargs))
            return 0.5 * kwargs["reward"]

        def update(self, **kwargs):
            pass

    a, xs = _net(cases.namespace("b200"), Halved)
    b, _ = _net(cases.namespace("b200"), None)
    with OracleBackend():
        a.run(inputs={"X": xs[0]}, time=T, reward=0.8)
        b.run(inputs={"X": xs[0]}, time=T, reward=0.4)
    assert calls == [["reward"]]
    assert torch.equal(a.connections[("X", "Y")].w, b.connections[("X", "Y")].w)
    with pytest.raises(TypeError):
        AbstractReward()


def _kernel_vs_oracle(rule, backend, to_dev):
    """The episodes on the CUDA kernels (`backend` None: the B200; else the emulation of tests/emu) and on the oracle."""
    from bindsnet_b200.learning.reward import MovingAvgRPE
    from oracle.oracle import OracleBackend

    ns = cases.namespace("b200")
    batch = 1 if rule == "MSTDPET" else B   # the reference's flattened eligibility trace is batch-1 only (learning.py:2187-2249)
    dev, xs = _net(ns, MovingAvgRPE, rule, batch)
    if backend is None:
        dev.to("cuda")
    run = lambda n, x, r: n.run(inputs={"X": to_dev(x)}, time=T, reward=r, a_plus=0.9, a_minus=-1.1)
    if backend is None:
        seen_dev = _episodes(dev, xs, run)
        dev.check_errors()
    else:
        with backend() as eb:
            seen_dev = _episodes(dev, xs, run)
        assert eb.err == 0
    cpu, xs2 = _net(ns, MovingAvgRPE, rule, batch)
    with OracleBackend() as ob:
        seen_cpu = _episodes(cpu, xs2, _plain_run)
        assert ob.err == 0
    assert seen_dev == seen_cpu
    assert float(cpu.connections[("X", "Y")].w.abs().sum()) > 0
    helpers.assert_bit_identical(helpers.snapshot(dev), helpers.snapshot(cpu), f"{rule} with reward_fn")


@pytest.mark.parametrize("rule", ["MSTDP", "MSTDPET"])
def test_reward_fn_on_the_emulated_kernels_bit_exact_vs_oracle(rule):
    """CPU twin of the GPU test: the same episodes through the kernels' CUDA sources on the emulation of tests/emu."""
    import os
    import sys

    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "emu"))
    import emu

    _kernel_vs_oracle(rule, emu.EmuBackend, lambda x: x)
