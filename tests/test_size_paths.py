"""The size-selected code paths of the generic window kernel (csrc/snn_generic.cu + snn_phases.cuh, force_tier = 1) and
of the single operators (csrc/snn_ops.cu: Connection.compute / update / normalize, Conv2dConnection.compute / normalize),
on both sides of every threshold.

The kernels switch code paths on size: the batch (target traces staged in shared memory up to B = 768, more than eight
sample groups above B = 256, eager weight-row prefetch from B = 64, a strided sample loop in conn_compute above B = 512),
the width of a source layer (per-sample any-spike flags above 1024 neurons, a second gather group above 8192), the
number of samples with a post-synaptic event in one tile and step (16 staged slots), and the staging limits of the
convolutional gather and of the MSTDP rules.  Every case below states which of those paths it is built to reach, and a
predicate recomputed from the kernel's own constants (mirrored below, each beside the source line it copies) asserts
that it does: a later change to a threshold fails that assertion instead of silently moving a case off its path.

Window cases run bit for bit against the oracle, on the B200 (`-m gpu`) and through the emulated kernel (tests/emu).
The single operators are compared with the oracle bit for bit and, independently, with a float64 restatement of the
operation written here, within a tolerance derived from the number and size of the fp32 terms that are summed."""
import contextlib
import os
import sys
from dataclasses import dataclass
from typing import Callable, Tuple

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import cases
import helpers

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "emu"))

# ---- the kernel's thresholds -----------------------------------------------------------------------------------------
P3_MAXEV = 16                          # csrc/snn_phases.cuh:20   SNN_P3_MAXEV: staged event-sample slots per tile
CONV_STAGE_WORDS = 4096                # csrc/snn_phases.cuh:22   SNN_CONV_STAGE_WORDS
CONV_STAGE_TAPS = 4096                 # csrc/snn_phases.cuh:23   SNN_CONV_STAGE_TAPS
XT_MAX_BYTES = 96 * 1024               # csrc/snn_phases.cuh:24   SNN_XT_MAX_BYTES
TILE = 32                              # csrc/snn_common.cuh:33   SNN_TILE
GEN_WARPS = 8                          # csrc/snn_common.cuh:34-35 SNN_GEN_THREADS / 32
ACC_BYTES = 4 * GEN_WARPS * 32 * 32    # csrc/snn_phases.cuh:46   acc region (dense MSTDP staging limit, :811)
EAGER_MIN_B = 64                       # csrc/snn_phases.cuh:638  eager = B >= 64
GROUPS_PER_PASS = 8                    # csrc/snn_phases.cuh:661  for (g0 = 0; g0 < NG; g0 += 8)
GATHER_WORDS_PER_PASS = 256            # csrc/snn_phases.cuh:100  for (s0 = 0; s0 < nw_src; s0 += 256)
WIDE_SRC_WORDS = 32                    # csrc/snn_api.cu:104      wide_src: nw > 32
COMPUTE_MAX_GRID_Y = 64                # csrc/snn_ops.cu:142      conn_compute grid.y <= 64
NORM_CHUNKS = 16                       # include/snn_b200.h       SNN_NORM_CHUNKS
EPS = 2.0 ** -24                       # unit roundoff of fp32


def nw(n: int) -> int:
    return (n + 31) // 32


def xt_bytes(B: int) -> int:           # csrc/snn_phases.cuh:40-43 gen_xt_bytes
    b = 4 * 32 * B
    return b if b <= XT_MAX_BYTES else 0


def plan(layer_ns, conns, B: int, cap: int):
    """csrc/snn_generic.cu:186-216 plan_units: (nch, cs, {conn: rc}) for a grid of `cap` CTAs.  `conns` holds
    (n_src, n_tgt, kind) with kind "stdp" (row-chunked learning units), "mstdp" or "other"."""
    items = sum(nw(n) for n in layer_ns)
    nch = -(-B // (4 * GEN_WARPS))
    while nch > 1 and items * nch > 16 * cap:
        nch -= 1
    cs = -(-B // nch)
    rc = {}
    for k, (ns, nt, kind) in enumerate(conns):
        if kind == "stdp":
            rc[k] = max(1, min(-(-cap // nw(nt)), -(-nw(ns) // GEN_WARPS)))
    return -(-B // cs), cs, rc


# ---- window cases ------------------------------------------------------------------------------------------------------
def _ns():
    return cases.namespace("b200")


def _lif(ns, n):
    return ns.nodes.LIFNodes(n=n, traces=True, thresh=-60.0, rest=-65.0, reset=-64.0, refrac=1, tc_decay=30.0)


def _rule(ns, name):
    return {"PostPre": ns.learning.PostPre, "WDep": ns.learning.WeightDependentPostPre, "Hebbian": ns.learning.Hebbian}[name]


NU = {"PostPre": (2e-3, 1e-2), "WDep": (1e-2, 3e-2), "Hebbian": (1e-3, 4e-3), "MCC": (2e-3, 1e-2)}


def _learned(ns, src, tgt, w, rule, mean, decay, wmax, B):
    """A learned dense connection: Connection + rule, or (rule "MCC") MulticompartmentConnection + Weight + MCC PostPre."""
    red = torch.mean if mean else torch.sum
    if rule == "MCC":
        from bindsnet_b200.learning.MCC_learning import PostPre as MCCPostPre
        from bindsnet_b200.network.topology_features import Weight

        return ns.topology.MulticompartmentConnection(source=src, target=tgt, device="cpu", pipeline=[
            Weight("weight", w, range=[0.0, wmax], nu=NU["MCC"], reduction=red, decay=decay, learning_rule=MCCPostPre, batch_size=B)])
    return ns.topology.Connection(source=src, target=tgt, w=w, update_rule=_rule(ns, rule), nu=NU[rule], reduction=red,
                                  weight_decay=decay, wmin=0.0, wmax=wmax)


def ff(B, n_in, n_hid, T, p_in=0.25, drive=3.0, rule="PostPre", mean=False, decay=0.0, seed=0):
    """Input(n_in) -> LIFNodes(n_hid), one learned connection; `drive` = expected input per target neuron and step."""
    def build():
        ns = _ns()
        g = torch.Generator().manual_seed(7000 + seed)
        scale = 2.0 * drive / max(n_in * p_in, 1e-3)
        net = ns.Network(dt=1.0, batch_size=B)
        X = ns.nodes.Input(n=n_in, traces=True)
        Y = _lif(ns, n_hid)
        net.add_layer(X, "X"); net.add_layer(Y, "Y")
        C = _learned(ns, X, Y, scale * torch.rand(n_in, n_hid, generator=g), rule, mean, decay, 1.5 * scale, B)
        net.add_connection(C, "X", "Y")
        x = torch.bernoulli(p_in * torch.ones(T, B, n_in), generator=g).byte()
        return net, {"X": x}, {}, T
    return build


def dc_one_spike(B, T=8):
    def build():
        ns = _ns()
        torch.manual_seed(11)
        net = ns.models.DiehlAndCook2015(n_inpt=64, n_neurons=40, batch_size=B, inpt_shape=(1, 8, 8), dt=1.0, nu=(1e-3, 1e-2),
                                         norm=20.0, theta_plus=0.05, exc=22.5, inh=60.0)
        cases._set_dc_weights(net, cases._w((64, 40), 12, 1.6))
        g = torch.Generator().manual_seed(13)
        return net, {"X": torch.bernoulli(0.3 * torch.ones(T, B, 1, 8, 8), generator=g).byte()}, {}, T
    return build


def mstdp_dense(B, n_in, n_tgt, T):
    def build():
        ns = _ns()
        g = torch.Generator().manual_seed(21)
        net = ns.Network(dt=1.0, batch_size=B)
        X = ns.nodes.Input(n=n_in, traces=True)
        Y = _lif(ns, n_tgt)
        net.add_layer(X, "X"); net.add_layer(Y, "Y")
        net.add_connection(ns.topology.Connection(source=X, target=Y, w=1.2 * torch.rand(n_in, n_tgt, generator=g) - 0.2,
                                                  update_rule=ns.learning.MSTDP, nu=5e-2, reduction=torch.sum, wmin=-1.0, wmax=1.5,
                                                  tc_plus=15.0, tc_minus=25.0), "X", "Y")
        x = torch.bernoulli(0.25 * torch.ones(T, B, n_in), generator=g).byte()
        return net, {"X": x}, {"reward": 0.7, "a_plus": 0.9, "a_minus": -1.1}, T
    return build


def conv(B, T, in_shape, cout, k, rule, seed):
    def build():
        ns = _ns()
        g = torch.Generator().manual_seed(31 + seed)
        cin, hin, win = in_shape
        ho, wo = hin - k + 1, win - k + 1
        net = ns.Network(dt=1.0, batch_size=B)
        X = ns.nodes.Input(shape=[cin, hin, win], traces=True)
        H = ns.nodes.LIFNodes(shape=[cout, ho, wo], traces=True, thresh=-64.0, refrac=1, tc_decay=60.0)
        net.add_layer(X, "X"); net.add_layer(H, "H")
        K = cin * k * k
        w = (8.0 / K) * torch.rand(cout, cin, k, k, generator=g) - 1.0 / K
        r = {"PostPre": ns.learning.PostPre, "MSTDP": ns.learning.MSTDP}[rule]
        nu = (4e-3, 2e-2) if rule == "PostPre" else 1e-2
        net.add_connection(ns.topology.Conv2dConnection(source=X, target=H, kernel_size=k, w=w, update_rule=r, nu=nu,
                                                        reduction=torch.sum, wmin=-1.0, wmax=1.0), "X", "H")
        x = torch.bernoulli(0.2 * torch.ones(T, B, cin, hin, win), generator=g).byte()
        return net, {"X": x}, ({"reward": 1.0} if rule == "MSTDP" else {}), T
    return build


def recurrent(B, n, T):
    """Input -> Y and a learned Y -> Y connection (src == tgt)."""
    def build():
        ns = _ns()
        g = torch.Generator().manual_seed(41)
        net = ns.Network(dt=1.0, batch_size=B)
        X = ns.nodes.Input(n=40, traces=True)
        Y = _lif(ns, n)
        net.add_layer(X, "X"); net.add_layer(Y, "Y")
        net.add_connection(ns.topology.Connection(source=X, target=Y, w=0.6 * torch.rand(40, n, generator=g)), "X", "Y")
        net.add_connection(ns.topology.Connection(source=Y, target=Y, w=0.4 * torch.rand(n, n, generator=g) - 0.1,
                                                  update_rule=ns.learning.PostPre, nu=(2e-3, 1e-2), reduction=torch.sum,
                                                  wmin=-0.5, wmax=1.0), "Y", "Y")
        return net, {"X": torch.bernoulli(0.25 * torch.ones(T, B, 40), generator=g).byte()}, {}, T
    return build


def two_into_one(B, T):
    """Two learned connections (PostPre, sum; Hebbian, mean) into one target."""
    def build():
        ns = _ns()
        g = torch.Generator().manual_seed(51)
        net = ns.Network(dt=1.0, batch_size=B)
        X = ns.nodes.Input(n=50, traces=True)
        Z = ns.nodes.Input(n=70, traces=True)
        Y = _lif(ns, 45)
        net.add_layer(X, "X"); net.add_layer(Z, "Z"); net.add_layer(Y, "Y")
        net.add_connection(_learned(ns, X, Y, 0.5 * torch.rand(50, 45, generator=g), "PostPre", False, 0.0, 1.0, B), "X", "Y")
        net.add_connection(_learned(ns, Z, Y, 0.3 * torch.rand(70, 45, generator=g), "Hebbian", True, 1e-3, 1.0, B), "Z", "Y")
        x = torch.bernoulli(0.25 * torch.ones(T, B, 50), generator=g).byte()
        z = torch.bernoulli(0.2 * torch.ones(T, B, 70), generator=g).byte()
        return net, {"X": x, "Z": z}, {}, T
    return build


# ---- path predicates: each recomputes one switch of the kernel from the network and the oracle's [T, B, n] rasters ------
def _kind(c) -> str:
    """"dense" / "mstdp" / "conv" for a learned connection, "" for one without a rule."""
    rule = getattr(c, "update_rule", None)
    if rule is None and hasattr(c, "pipeline"):
        rule = c.pipeline[0].learning_rule
    rname = type(rule).__name__
    if rname in ("NoOp", "NoneType"):
        return ""
    if type(c).__name__ == "Conv2dConnection":
        return "conv"
    return "mstdp" if rname.startswith("MSTDP") else "dense"


class Ctx:
    def __init__(self, net, rasters, cap):
        self.net, self.rasters, self.cap = net, rasters, cap
        self.B = next(iter(rasters.values())).shape[1]
        self.n = {k: l.n for k, l in net.layers.items()}

    def learned(self, kinds=("dense",)):
        """(src, tgt, conn) of the learned connections of the given kinds."""
        return [(s, t, c) for (s, t), c in self.net.connections.items() if _kind(c) in kinds]

    def plan(self):
        conns = [(self.n[s], self.n[t], {"dense": "stdp", "mstdp": "mstdp"}.get(_kind(c), "other"))
                 for (s, t), c in self.net.connections.items()]
        return plan(list(self.n.values()), conns, self.B, self.cap)


def _events_per_tile(r):   # r: [T, B, n] -> [T, tiles] number of samples with a spike in the tile
    T, B, n = r.shape
    pad = np.zeros((T, B, nw(n) * TILE), dtype=bool)
    pad[:, :, :n] = r != 0
    return pad.reshape(T, B, -1, TILE).any(-1).sum(1)


def _conv_geo(c):
    cin, hin, win = c.source.shape
    cout, ho, wo = c.target.shape
    kh, kw = c.kernel_size
    return cin, hin, win, cout, ho, wo, kh, kw


PATHS: dict = {
    # phase 3, pre-synaptic term: target traces read from L2 per sample (stage == false), with the __any_sync skip
    "unstaged_target_traces": lambda x: xt_bytes(x.B) == 0 and len(x.learned()) > 0,
    # phase 3: more than SNN_P3_MAXEV samples with a post-synaptic spike in one tile in one step
    "event_overflow": lambda x: any(_events_per_tile(x.rasters[t]).max() > P3_MAXEV for _, t, _ in x.learned()),
    # phase 3: weight rows fetched ahead
    "eager_rows": lambda x: x.B >= EAGER_MIN_B and len(x.learned()) > 0,
    # phase 3: second pass of the sample-group loop
    "second_sample_group_pass": lambda x: -(-x.B // 32) > GROUPS_PER_PASS and len(x.learned()) > 0,
    # gather: second 256-word group of the source, with a spike in it
    "second_gather_group": lambda x: any(nw(x.n[s]) > GATHER_WORDS_PER_PASS and x.rasters[s][:, :, GATHER_WORDS_PER_PASS * 32:].any()
                                         for (s, t), c in x.net.connections.items() if type(c).__name__ != "Conv2dConnection"),
    # per-sample any-spike flags of a wide source
    "wide_source_flags": lambda x: any(nw(x.n[s]) > WIDE_SRC_WORDS for (s, t), c in x.net.connections.items()
                                       if type(c).__name__ != "Conv2dConnection"),
    # a ragged last target tile of a learned connection
    "ragged_target_tile": lambda x: any(x.n[t] % TILE != 0 for _, t, _ in x.learned(("dense", "mstdp"))),
    # phases 1 / 2 split the batch into several sample chunks, the last one shorter
    "ragged_sample_chunks": lambda x: x.plan()[0] > 1 and x.B % x.plan()[1] != 0,
    # phase 3: a tile's rows split into row chunks of unequal length
    "uneven_row_chunks": lambda x: any(nw(x.n[s]) % x.plan()[2][k] != 0 for k, ((s, t), c) in enumerate(x.net.connections.items())
                                       if k in x.plan()[2]),
    # dense MSTDP with its rule state read from L2
    "mstdp_unstaged": lambda x: any(xt_bytes(x.B) == 0 or x.B * 32 + 5 * x.B * x.n[t] + 16 > ACC_BYTES for _, t, _ in x.learned(("mstdp",))),
    # conv gather: source bit rows of the sample chunk not staged (snn_phases.cuh:328)
    "conv_bits_unstaged": lambda x: any(x.plan()[1] * nw(x.n[s]) > CONV_STAGE_WORDS
                                        for (s, t), c in x.net.connections.items() if type(c).__name__ == "Conv2dConnection"),
    # conv gather: filter taps of a tile not staged (snn_phases.cuh:333)
    # (one output channel's cin * kh * kw taps already exceed the limit, so every tile's do)
    "conv_taps_unstaged": lambda x: any(g[0] * g[6] * g[7] > CONV_STAGE_TAPS for g in (_conv_geo(c) for (s, t), c in x.net.connections.items()
                                                                                         if type(c).__name__ == "Conv2dConnection")),
    # conv MSTDP: P- rows not staged (snn_phases.cuh:1079 stage_pm)
    "conv_pm_unstaged": lambda x: any(g[4] * g[5] > GEN_WARPS * 32 * 32 for g in (_conv_geo(c) for _, _, c in x.learned(("conv",)))),
    # conv MSTDP: bit rows not staged (snn_phases.cuh:1082 staged) / source spikes not listed (:1090 listed)
    "conv_rows_unstaged": lambda x: any(nw(x.n[s]) + nw(x.n[t]) > CONV_STAGE_WORDS for s, t, _ in x.learned(("conv",))),
    "conv_unlisted": lambda x: any(nw(x.n[s]) + nw(x.n[t]) > CONV_STAGE_WORDS
                                   or CONV_STAGE_WORDS - nw(x.n[s]) - nw(x.n[t]) - (c.source.shape[0] + 2) < x.n[s]
                                   for s, t, c in x.learned(("conv",))),
    # two layers of the window are one: a learned connection with src == tgt
    "recurrent": lambda x: any(s == t for s, t, _ in x.learned()),
    "two_learned_into_one": lambda x: max(np.unique([t for _, t, _ in x.learned()], return_counts=True)[1], default=0) >= 2,
}


@dataclass
class W:
    name: str
    build: Callable
    paths: Tuple[str, ...] = ()


WINDOW = [W(f"lif_postpre_b{B}", ff(B, 40, 33, 4 if B > 256 else 6, seed=B),
            tuple(p for p, on in (("eager_rows", B >= 64), ("second_sample_group_pass", B > 256), ("unstaged_target_traces", B > 768),
                                  ("ragged_target_tile", True), ("ragged_sample_chunks", B in (33, 65))) if on))
          for B in (1, 31, 32, 33, 63, 64, 65, 255, 256, 257, 768, 769)]
WINDOW += [W(f"{rule.lower()}_mean_decay_b{B}", ff(B, 40, 33, 4 if B > 256 else 6, rule=rule, mean=True,
                                                    decay=2e-3, seed=B + 1),
             ("eager_rows",) + (("second_sample_group_pass",) if B > 256 else ()) + (("unstaged_target_traces",) if B > 768 else ()))
           for rule in ("WDep", "Hebbian", "MCC") for B in (65, 257, 769)]
WINDOW += [
    W("dc_one_spike_b33", dc_one_spike(33), ("ragged_sample_chunks",)),
    W("dc_one_spike_b257", dc_one_spike(257, T=5), ("second_sample_group_pass",)),
    W("overflow_sum", ff(48, 40, 45, 6, drive=6.0, seed=3), ("event_overflow", "ragged_target_tile")),
    W("overflow_mean", ff(80, 40, 33, 6, drive=6.0, mean=True, seed=4), ("event_overflow", "eager_rows")),
] + [W(f"width_src{n}", ff(4, n, 65 if n > 100 else 33, 6, p_in=min(0.25, 40.0 / n + 0.02), drive=4.0, seed=n),
       (("wide_source_flags",) if n > 1024 else ()) + (("second_gather_group",) if n > 8192 else ()) + ("ragged_target_tile",))
     for n in (1, 31, 33, 1023, 1024, 1025, 8300)] + [
    W("width_tgt1", ff(5, 40, 1, 6, seed=61)),
    W("width_tgt31", ff(5, 40, 31, 6, seed=62), ("ragged_target_tile",)),
    W("width_tgt1025", ff(3, 40, 1025, 4, seed=63), ("ragged_target_tile",)),
    W("wide_uneven_rows", ff(41, 1023, 33, 4, p_in=0.05, seed=64), ("uneven_row_chunks", "ragged_sample_chunks", "ragged_target_tile")),
    W("mstdp_dense_unstaged", mstdp_dense(64, 50, 100, 6), ("mstdp_unstaged",)),
    W("conv_postpre_big_maps", conv(9, 3, (1, 128, 128), 8, 3, "PostPre", 0), ("conv_bits_unstaged",)),
    W("conv_mstdp_big_maps", conv(9, 3, (1, 128, 128), 8, 3, "MSTDP", 1),
      ("conv_bits_unstaged", "conv_pm_unstaged", "conv_rows_unstaged", "conv_unlisted")),
    W("conv_postpre_deep_filters", conv(2, 4, (512, 5, 5), 2, 3, "PostPre", 2), ("conv_taps_unstaged",)),
    W("conv_mstdp_deep_filters", conv(2, 4, (512, 5, 5), 2, 3, "MSTDP", 3), ("conv_taps_unstaged",)),
    W("recurrent_b70", recurrent(70, 45, 6), ("recurrent", "eager_rows", "ragged_target_tile")),
    W("two_into_one_b65", two_into_one(65, 6), ("two_learned_into_one", "eager_rows", "ragged_sample_chunks")),
]
BY_NAME = {c.name: c for c in WINDOW}
# the emulated twins run this subset on a one-SM and a seven-SM device too: plan_units cuts them differently
GRID_SUBSET = ["lif_postpre_b65", "lif_postpre_b257", "lif_postpre_b769", "wdep_mean_decay_b257", "overflow_sum", "width_src1025",
               "wide_uneven_rows", "dc_one_spike_b33", "mstdp_dense_unstaged", "two_into_one_b65"]
EMU_CAP = 2 * 3   # tests/emu: SNN_EMU_SMS (default 3) x 2 CTAs (snn_generic.cu:222-224)


def _run_window(case: W, backend: str, env=None):
    """One window of `case` on "oracle", "emu" (tests/emu) or "cuda"; returns (state, counts, rasters)."""
    net, inputs, kw, T = case.build()
    net.force_tier = 1
    dev = "cuda" if backend == "cuda" else "cpu"
    if dev == "cuda":
        net.to("cuda")
        inputs = {k: v.cuda() for k, v in inputs.items()}
    helpers.add_spike_monitors(net, T, device=dev)
    old = {k: os.environ.get(k) for k in (env or {})}
    os.environ.update(env or {})
    try:
        if backend == "emu":
            import emu
            ctx = emu.EmuBackend()
        elif backend == "oracle":
            from oracle.oracle import OracleBackend
            ctx = OracleBackend()
        else:
            ctx = contextlib.nullcontext()
        with ctx as be:
            net.run(inputs=inputs, time=T, one_spike_seed=cases.ONE_SPIKE_SEED, **kw)
        if be is not None:
            assert be.err == 0
        else:
            net.check_errors()
        if backend == "emu":
            assert emu.last_tier == 1, f"window went to tier {emu.last_tier}, not 1"
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
    B = next(iter(net.layers.values())).s.shape[0]
    rasters = {l: net.monitors[f"mon_{l}"].get("s").reshape(T, B, -1).cpu().numpy() for l in net.layers}
    return net, helpers.snapshot(net), helpers.spike_counts(net, T), rasters


_ORACLE = {}


def _oracle(name):
    """The oracle's result of a case (computed once per session: the GPU test and the emulated twins share it)."""
    if name not in _ORACLE:
        _ORACLE[name] = _run_window(BY_NAME[name], "oracle")
    return _ORACLE[name]


def _check_paths(name, cap):
    net, _, counts, rasters = _oracle(name)
    x = Ctx(net, rasters, cap)
    for p in BY_NAME[name].paths:
        assert PATHS[p](x), f"{name} does not reach its path {p!r}"
    learned = [t for _, t, _ in x.learned(("dense", "mstdp", "conv"))]
    assert all(int(counts[f"L/{t}/count"].sum()) > 0 for t in learned), f"{name}: a learned connection's target never spiked"


def test_every_path_is_claimed_by_some_case():
    claimed = {p for c in WINDOW for p in c.paths}
    assert claimed == set(PATHS), f"paths without a case: {set(PATHS) - claimed}"
    assert len(BY_NAME) == len(WINDOW)


@pytest.mark.parametrize("name", list(BY_NAME))
def test_emulated_generic_kernel_on_size_paths(name):
    _check_paths(name, EMU_CAP)
    _, s_emu, c_emu, _ = _run_window(BY_NAME[name], "emu")
    _, s_ref, c_ref, _ = _oracle(name)
    helpers.assert_bit_identical(s_emu, s_ref, f"{name} state (emulated kernel)")
    helpers.assert_bit_identical(c_emu, c_ref, f"{name} spike counts (emulated kernel)")


@pytest.mark.parametrize("name", GRID_SUBSET)
@pytest.mark.parametrize("sms", ["1", "7"])
def test_emulated_size_paths_are_independent_of_the_grid_size(name, sms):
    _, s_emu, c_emu, _ = _run_window(BY_NAME[name], "emu", env={"SNN_EMU_SMS": sms})
    _, s_ref, c_ref, _ = _oracle(name)
    helpers.assert_bit_identical(s_emu, s_ref, f"{name} state (emulated kernel, {sms} SMs)")
    helpers.assert_bit_identical(c_emu, c_ref, f"{name} spike counts (emulated kernel, {sms} SMs)")


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(BY_NAME))
def test_generic_kernel_on_size_paths(name):
    _check_paths(name, EMU_CAP)
    _, s_gpu, c_gpu, _ = _run_window(BY_NAME[name], "cuda")
    _, s_ref, c_ref, _ = _oracle(name)
    helpers.assert_bit_identical(s_gpu, s_ref, f"{name} state")
    helpers.assert_bit_identical(c_gpu, c_ref, f"{name} spike counts")


# ---- single operators --------------------------------------------------------------------------------------------------
def _backends(gpu: bool):
    """(name, context manager factory, device) of the implementation under test and of the oracle."""
    from oracle.oracle import OracleBackend

    if gpu:
        return [("cuda", contextlib.nullcontext, "cuda"), ("oracle", OracleBackend, "cpu")]
    import emu

    return [("emu", emu.EmuBackend, "cpu"), ("oracle", OracleBackend, "cpu")]


def _same_bits(a: torch.Tensor, b: torch.Tensor, what: str):
    a, b = a.detach().cpu().contiguous(), b.detach().cpu().contiguous()
    assert a.shape == b.shape, what
    if not torch.equal(a.view(torch.int32), b.view(torch.int32)):
        d = (a.double() - b.double()).abs()
        raise AssertionError(f"{what}: {(d > 0).sum().item()} entries differ from the oracle, max |d| {d.max().item():.3e}")


def _within(got: torch.Tensor, ref64: torch.Tensor, tol64: torch.Tensor, what: str):
    d = (got.detach().cpu().double() - ref64).abs()
    bad = d > tol64
    assert not bad.any(), (f"{what}: {bad.sum().item()} entries beyond the float64 bound, worst |d| {d[bad].max().item():.3e} "
                           f"vs bound {tol64[bad][d[bad].argmax()].item():.3e}")


COMPUTE = [(B, ns_, bias) for B in (1, 512, 513, 1100) for ns_ in (31, 1025, 8200) for bias in (False, True)]


def _compute_case(B, n_src, bias, gpu):
    from bindsnet_b200.network import nodes, topology

    n_tgt = 45
    assert (-(-B // GEN_WARPS) > COMPUTE_MAX_GRID_Y) == (B > 512)        # the strided sample loop: B > 512
    g = torch.Generator().manual_seed(B * 31 + n_src + bias)
    w = torch.rand(n_src, n_tgt, generator=g) - 0.3
    b = torch.rand(n_tgt, generator=g) - 0.5
    s = torch.bernoulli(min(0.3, 60.0 / n_src) * torch.ones(B, n_src), generator=g).bool()
    outs = []
    for _, mk, dev in _backends(gpu):
        X, Y = nodes.Input(n=n_src), nodes.LIFNodes(n=n_tgt)
        kw = {"b": b} if bias else {}
        C = topology.Connection(X, Y, w=w, **kw).to(dev)
        with mk():
            outs.append(C.compute(s.to(dev)))
    _same_bits(outs[0], outs[1], f"compute B={B} n_src={n_src} bias={bias}")
    sd, wd = s.double(), w.double()
    ref = sd @ wd + (b.double() if bias else 0.0)
    k = s.sum(1, keepdim=True).double() + (1.0 if bias else 0.0)            # fp32 terms summed per output
    tol = k * EPS * (sd @ wd.abs() + (b.double().abs() if bias else 0.0))
    _within(outs[0], ref, tol, f"compute B={B} n_src={n_src} bias={bias} vs float64")


@pytest.mark.parametrize("B,n_src,bias", COMPUTE)
def test_emulated_conn_compute_sizes(B, n_src, bias):
    _compute_case(B, n_src, bias, gpu=False)


@pytest.mark.gpu
@pytest.mark.parametrize("B,n_src,bias", COMPUTE)
def test_conn_compute_sizes(B, n_src, bias):
    _compute_case(B, n_src, bias, gpu=True)


UPDATE_RULES = ["PostPre", "WDep", "Hebbian", "MCC", "recurrent"]
UPDATE = [(rule, B, mean) for rule in UPDATE_RULES[:4] for B in (5, 65, 300, 800) for mean in (False, True)]
UPDATE += [("recurrent", B, False) for B in (5, 300)]


def _update_case(rule, B, mean, gpu):
    """Connection.update (snn_b200_conn_update: phase 3 on the layers' current spikes and traces) after a state built so
    that more than 16 samples spike in one target tile (B > 16), against the oracle and the rule written in float64."""
    from bindsnet_b200.network import nodes, topology

    n_src, n_tgt = 70, 45
    decay = 2e-3 if mean else 0.0
    wmin, wmax = 0.0, 1.0
    g = torch.Generator().manual_seed(100 * B + 10 * UPDATE_RULES.index(rule) + mean)
    rec = rule == "recurrent"
    if rec:
        n_src = n_tgt
    w0 = 1.2 * torch.rand(n_src, n_tgt, generator=g) - 0.1                 # the constructors clamp it into [wmin, wmax]
    ss = torch.bernoulli(0.3 * torch.ones(B, n_src), generator=g).bool()
    xs = torch.rand(B, n_src, generator=g)
    st = torch.bernoulli(0.4 * torch.ones(B, n_tgt), generator=g).bool()
    xt = torch.rand(B, n_tgt, generator=g)
    if rec:
        ss, xs = st, xt
    if B > P3_MAXEV:   # the overflow condition: more than 16 event samples in the first target tile
        assert int(st[:, :TILE].any(1).sum()) > P3_MAXEV
    unstaged = xt_bytes(B) == 0
    assert unstaged == (B > 768)
    res = []
    for _, mk, dev in _backends(gpu):
        X = nodes.Input(n=n_src, traces=True)
        Y = X if rec else nodes.LIFNodes(n=n_tgt, traces=True)
        if rule == "MCC":
            from bindsnet_b200.learning.MCC_learning import PostPre as MCCPostPre
            from bindsnet_b200.network.topology_features import Weight

            C = topology.MulticompartmentConnection(source=X, target=Y, device="cpu", pipeline=[
                Weight("weight", w0.clamp(wmin, wmax), range=[wmin, wmax], nu=NU["MCC"], reduction=torch.mean if mean else torch.sum,
                       decay=decay, learning_rule=MCCPostPre, batch_size=B)])
        else:
            r = {"recurrent": "PostPre"}.get(rule, rule)
            C = topology.Connection(X, Y, w=w0.clone(), update_rule=_rule(_ns(), r), nu=NU[r],
                                    reduction=torch.mean if mean else torch.sum, weight_decay=decay, wmin=wmin, wmax=wmax)
        for l in {id(X): X, id(Y): Y}.values():
            l.compute_decays(1.0); l.set_batch_size(B)
        X.s, X.x = ss.clone(), xs.clone()
        if not rec:
            Y.s, Y.x = st.clone(), xt.clone()
        for m in {id(X): X, id(Y): Y}.values():
            m.to(dev)
        C.to(dev)
        with mk():
            C.update(learning=True)
        res.append(C.w.detach().clone())
    _same_bits(res[0], res[1], f"update {rule} B={B} mean={mean}")

    # float64: the reference's formula for the rule (learning.py PostPre / WeightDependentPostPre / Hebbian, MCC_learning.py
    # PostPre with connection.dt = 1), then the base class' weight decay and clamp
    r = "PostPre" if rule in ("recurrent", "MCC") else rule
    nu0, nu1 = NU["MCC" if rule == "MCC" else r]
    red = (lambda a: a / B) if mean else (lambda a: a)
    sS, xS, sT, xT, w = ss.double(), xs.double(), st.double(), xt.double(), w0.double().clamp(wmin, wmax)
    pre, post = red(sS.T @ xT), red(xS.T @ sT)                               # plain batch sums of the outer products
    if r == "PostPre":
        w1 = w - nu0 * pre + nu1 * post
        mag = (nu0 * pre + nu1 * post).abs()
    elif r == "WDep":
        dpre, dpost = nu0 * pre * (w - wmin), nu1 * post * (wmax - w)
        w1 = w - dpre + dpost
        mag = dpre.abs() + dpost.abs()
    else:
        w1 = w + nu0 * pre + nu1 * post
        mag = (nu0 * pre + nu1 * post).abs()
    if decay:
        w1 = w1 * (1.0 - decay)
    w1 = w1.clamp(wmin, wmax)
    # B fp32 adds per batch sum (all terms >= 0 here, so sum|terms| = the sum), plus a few single roundings: nu scaling,
    # / B, the rule's products, the two updates of w, the decay
    tol = EPS * ((B + 4) * mag + 4.0 * (w.abs() + mag))
    _within(res[0], w1, tol, f"update {rule} B={B} mean={mean} vs float64")


@pytest.mark.parametrize("rule,B,mean", UPDATE)
def test_emulated_conn_update_sizes(rule, B, mean):
    _update_case(rule, B, mean, gpu=False)


@pytest.mark.gpu
@pytest.mark.parametrize("rule,B,mean", UPDATE)
def test_conn_update_sizes(rule, B, mean):
    _update_case(rule, B, mean, gpu=True)


NORMALIZE = [5, 37, 8200]   # fewer rows than SNN_NORM_CHUNKS (16), not a multiple of 16, more than 8192


def _normalize_case(n_src, gpu):
    from bindsnet_b200.network import nodes, topology

    n_tgt, norm = 45, 10.0
    g = torch.Generator().manual_seed(n_src)
    w0 = torch.rand(n_src, n_tgt, generator=g) - 0.25
    w0[:, 7] = 0.0                                                          # an all-zero column: divided by 1
    res = []
    for _, mk, dev in _backends(gpu):
        C = topology.Connection(nodes.Input(n=n_src), nodes.LIFNodes(n=n_tgt), w=w0.clone(), norm=norm).to(dev)
        with mk():
            C.normalize()
        res.append(C.w.detach().clone())
    _same_bits(res[0], res[1], f"normalize n_src={n_src}")
    # topology.py:383-392: w *= norm / |w|.sum(0), zero sums replaced by 1
    w = w0.double()
    cs = w.abs().sum(0)
    cs[cs == 0] = 1.0
    ref = w * (norm / cs)
    tol = ref.abs() * EPS * (n_src + 3)                                     # n_src-term sum of |w| (relative), then 3 roundings
    _within(res[0], ref, tol, f"normalize n_src={n_src} vs float64")


@pytest.mark.parametrize("n_src", NORMALIZE)
def test_emulated_conn_normalize_sizes(n_src):
    _normalize_case(n_src, gpu=False)


@pytest.mark.gpu
@pytest.mark.parametrize("n_src", NORMALIZE)
def test_conn_normalize_sizes(n_src):
    _normalize_case(n_src, gpu=True)


# (source [C, H, W], cout, kernel, stride, padding, dilation).  Dilation: the host API checks the target shape with the
# reference's formula, which leaves dilation out (topology.py:752-772); these geometries satisfy both formulas.
CONV = {
    "dilated_asym": ((3, 12, 11), 4, (2, 2), (3, 2), (2, 1), (2, 2)),
    "asym_stride_pad": ((2, 9, 10), 3, (3, 2), (2, 1), (1, 0), (1, 1)),
    "kernel_1x1": ((6, 7, 5), 3, (1, 1), (1, 1), (0, 0), (1, 1)),
    "deep_filters": ((512, 5, 5), 2, (3, 3), (1, 1), (0, 0), (1, 1)),     # cin * kh * kw = 4608 > 4096
}


def _conv_case(name, gpu):
    from bindsnet_b200.network import nodes, topology

    (cin, hin, win), cout, k, st, pd, dl = CONV[name]
    ho = (hin + 2 * pd[0] - dl[0] * (k[0] - 1) - 1) // st[0] + 1
    wo = (win + 2 * pd[1] - dl[1] * (k[1] - 1) - 1) // st[1] + 1
    B, norm = 7, 0.8
    g = torch.Generator().manual_seed(len(name) * 13 + cin)
    w0 = torch.rand(cout, cin, *k, generator=g) - 0.2
    b = torch.rand(cout, generator=g) - 0.5
    s = torch.bernoulli(0.3 * torch.ones(B, cin, hin, win), generator=g).byte()
    res = []
    for _, mk, dev in _backends(gpu):
        C = topology.Conv2dConnection(nodes.Input(shape=[cin, hin, win]), nodes.LIFNodes(shape=[cout, ho, wo]), kernel_size=k,
                                      stride=st, padding=pd, dilation=dl, w=w0.clone(), b=b.clone(), norm=norm).to(dev)
        with mk():
            out = C.compute(s.to(dev))
            C.normalize()
        res.append((out.detach().clone(), C.w.detach().clone()))
    _same_bits(res[0][0], res[1][0], f"conv compute {name}")
    _same_bits(res[0][1], res[1][1], f"conv normalize {name}")
    sd, wd, bd = s.double(), w0.double(), b.double()
    ref = F.conv2d(sd, wd, bd, stride=st, padding=pd, dilation=dl)
    K = cin * k[0] * k[1]
    tol = (K + 1) * EPS * (F.conv2d(sd, wd.abs(), bd.abs(), stride=st, padding=pd, dilation=dl))
    _within(res[0][0], ref, tol, f"conv compute {name} vs float64")
    # topology.py:824-837: every (out, in) filter scaled by norm / its (signed) sum
    flt = wd.view(cout * cin, -1)
    ssum = flt.sum(1, keepdim=True)
    refw = (flt * (norm / ssum)).view_as(wd)
    rel = (k[0] * k[1]) * EPS * flt.abs().sum(1, keepdim=True) / ssum.abs() + 3 * EPS
    _within(res[0][1], refw, (refw.abs().view(cout * cin, -1) * rel).view_as(wd), f"conv normalize {name} vs float64")


@pytest.mark.parametrize("name", list(CONV))
def test_emulated_conv_operators(name):
    _conv_case(name, gpu=False)


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CONV))
def test_conv_operators(name):
    _conv_case(name, gpu=True)
