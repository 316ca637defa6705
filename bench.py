#!/usr/bin/env python
"""bench.py — headline metric of BASELINE.json: sample·timesteps/s of DiehlAndCook2015
(n_neurons=1600, batch 128 per GPU, 250 timesteps, learning on) on synthetic 28x28 Poisson
spike trains.

    python bench.py --gpus N --steps K --warmup W          # our arm (torchrun for N > 1)
    python bench.py --impl reference --steps K --warmup W  # CPU restatement of the reference

One "step" is one Network.run window: 250 timesteps over the rank's batch of 128 samples
(32 000 sample·timesteps per GPU).  Prints ONE JSON line (rank 0).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_NEURONS, BATCH, T_STEPS, N_INPT = 1600, 128, 250, 784
POOL = 8  # distinct input windows cycled through: 8 x 25 MB = 200 MB > 126 MB of L2
METRIC = "sample·timesteps/s DiehlAndCook2015 n=1600 b=128; 1/2/4/8 GPU vs ref CPU"
UNIT = "sample*timesteps/s"
WORKLOAD = (f"DiehlAndCook2015 n_neurons={N_NEURONS} batch={BATCH}/GPU {T_STEPS} timesteps/window, learning on "
            "(MCC PostPre STDP, one_spike, theta), synthetic Poisson 28x28 (~1.2% density)")


def apply_config(name: str) -> None:
    """--config c3: BASELINE.json configs[2] (n_neurons=6400, batch 256) instead of the metric configuration."""
    global N_NEURONS, BATCH, METRIC, WORKLOAD
    if name == "c3":
        N_NEURONS, BATCH = 6400, 256
        METRIC = "sample·timesteps/s DiehlAndCook2015 n=6400 b=256 (BASELINE.json configs[2])"
    WORKLOAD = (f"DiehlAndCook2015 n_neurons={N_NEURONS} batch={BATCH}/GPU {T_STEPS} timesteps/window, learning on "
                "(MCC PostPre STDP, one_spike, theta), synthetic Poisson 28x28 (~1.2% density)")


def algorithmic_bytes_per_timestep(n=None, B=None, P=N_INPT, monitors=False) -> int:
    """SURVEY.md §8d: read + write of the learned X->Ae weights (STDP + clamp must be visible
    to the next step) + the step's input spikes as delivered (uint8) [+ Ae/Ai rasters]."""
    n, B = n or N_NEURONS, B or BATCH
    return 2 * P * n * 4 + B * P + (2 * B * n if monitors else 0)


def synth_windows(count: int, seed: int, T=T_STEPS, B=None):
    """SURVEY.md §8d synthetic input: per-pixel rate 128*U(0,1)*Bernoulli(0.19) Hz on 1x28x28,
    Poisson-encoded (bindsnet_b200.encoding.poisson, restating encodings.py:99-156)."""
    import torch
    from bindsnet_b200.encoding import poisson

    B = B or BATCH
    g = torch.Generator().manual_seed(seed)
    out = []
    for _ in range(count):
        rate = 128.0 * torch.rand(B, 1, 28, 28, generator=g) * torch.bernoulli(0.19 * torch.ones(B, 1, 28, 28), generator=g)
        torch.manual_seed(int(torch.randint(0, 2**31 - 1, (1,), generator=g)))
        out.append(poisson(rate, time=T, dt=1.0).contiguous())  # [T, B, 1, 28, 28] uint8
    return out


def make_network(device):
    import torch
    from bindsnet_b200.models import DiehlAndCook2015

    torch.manual_seed(1234)
    net = DiehlAndCook2015(n_inpt=N_INPT, n_neurons=N_NEURONS, batch_size=BATCH, inpt_shape=(1, 28, 28), dt=1.0,
                           nu=(1e-4, 1e-2), norm=78.4, theta_plus=0.05, exc=22.5, inh=120.0)
    return net.to(device) if device is not None else net


# --dump-outputs: larger arrays are cut to a fixed, seeded sample of their elements.  The cap keeps the learned 784 x 1600
# weights of the metric configuration whole and c3 (batch 256, n = 6400, two 6400 x 6400 static matrices) under 64 MB
DUMP_MAX_ELEMS = 5 << 18
DUMP_MAX_BYTES = 64 << 20   # --dump-outputs: all files together


def dump_outputs(path: str, net) -> None:
    """--dump-outputs: what a caller of Network.run reads after the last timed window — every layer's spikes, voltages,
    traces, adaptive thresholds and refractory counters and every connection's weights — as float32 DIR/<name>.npy, so
    that two builds can be compared output for output.  An array of more than DUMP_MAX_ELEMS elements is flattened and
    cut to the same seeded sample of positions on every run."""
    import numpy as np
    import torch

    arrays = {}
    for lname, layer in net.layers.items():
        for var in ("s", "v", "x", "theta", "refrac_count"):
            val = getattr(layer, var, None)
            if isinstance(val, torch.Tensor) and val.numel():
                arrays[f"{lname}.{var}"] = val
    for (src, tgt), conn in net.connections.items():
        arrays[f"{src}-{tgt}.w"] = conn.w
    for name, val in arrays.items():
        a = val.detach().float().cpu().numpy()
        if a.size > DUMP_MAX_ELEMS:
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, DUMP_MAX_ELEMS, replace=False))]
        arrays[name] = a
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_MAX_BYTES:   # checked before anything is written: no partial DIR
        raise ValueError(f"--dump-outputs: {total / 2**20:.1f} MB of outputs, more than {DUMP_MAX_BYTES >> 20} MB")
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, f"{name}.npy"), a)


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None
        return self

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def __exit__(self, *exc):
        if self.proc is not None:
            time.sleep(0.15)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        return False

    def summary(self):
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for name, val in zip(names, f[2:6]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


def hbm_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured"
        except Exception:
            pass
    return 6650.0, "fallback"


def host_threads() -> int:
    """Threads the CPU legs use: every core of the box, set explicitly (torchrun exports
    OMP_NUM_THREADS=1 to its children, which must not silently shrink the baseline)."""
    return os.cpu_count() or 1


def cpu_baseline(steps_budget_s: float = 15.0):
    """The oracle's dense restatement of the reference algorithm (oracle/snn_oracle.c, every
    zero of `s.float() @ w` and of the batch-summed outer products multiplied like the reference
    does) on the host cores, on a bounded number of timesteps of the same workload."""
    from oracle.oracle import OracleBackend

    cores = host_threads()
    net = make_network(None)
    x = synth_windows(1, seed=999, T=64)[0]
    with OracleBackend(dense=1, threads=cores) as ob:
        t0 = time.perf_counter(); net.run({"X": x[:2]}, time=2); probe = (time.perf_counter() - t0) / 2
        T_s = int(max(4, min(60, steps_budget_s / max(probe, 1e-3))))
        net.reset_state_variables()
        t0 = time.perf_counter(); net.run({"X": x[:T_s]}, time=T_s); wall = time.perf_counter() - t0
    return {"value": BATCH * T_s / wall, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"{T_s} of {T_STEPS} timesteps of the same workload (n={N_NEURONS}, B={BATCH}), dense mode, "
                      f"{wall:.2f} s wall, OpenMP with {cores} threads (set explicitly)"}


def import_reference():
    """The UNMODIFIED reference from baseline/_ref (baseline/install_ref.sh), imported through a stub
    package because `import bindsnet` itself pulls in matplotlib & co. (SURVEY.md §8c); only the
    sub-packages of the hot path are loaded, in the order the reference's circular imports need."""
    import importlib
    import types

    ref = os.path.join(ROOT, "baseline", "_ref", "bindsnet")
    if not os.path.isdir(ref):
        return None, f"baseline/_ref/bindsnet not found (run baseline/install_ref.sh in the build container)"
    try:
        pkg = types.ModuleType("bindsnet")
        pkg.__path__ = [ref]
        sys.modules["bindsnet"] = pkg
        for sub in ("bindsnet.utils", "bindsnet.network", "bindsnet.learning", "bindsnet.models"):
            importlib.import_module(sub)
        return sys.modules["bindsnet.models"], None
    except Exception as e:  # missing dependency on this box
        return None, f"{type(e).__name__}: {e}"


def reference_baseline(budget_s: float = 20.0):
    """cpu_baseline leg of our arm: the live reference timed on this box's cores on a bounded sample."""
    import torch

    models, why = import_reference()
    if models is None:
        return None
    cores = host_threads()
    old = torch.get_num_threads()
    torch.set_num_threads(cores)
    try:
        torch.manual_seed(1234)
        net = models.DiehlAndCook2015(n_inpt=N_INPT, n_neurons=N_NEURONS, batch_size=BATCH, inpt_shape=(1, 28, 28), dt=1.0,
                                      nu=(1e-4, 1e-2), norm=78.4, theta_plus=0.05, exc=22.5, inh=120.0)
        x = synth_windows(1, seed=999, T=32)[0]
        t0 = time.perf_counter(); net.run({"X": x[:1]}, time=1); probe = time.perf_counter() - t0
        T_ref = int(max(1, min(32, budget_s / max(probe, 1e-3))))
        net.reset_state_variables()
        t0 = time.perf_counter(); net.run({"X": x[:T_ref]}, time=T_ref); wall = time.perf_counter() - t0
    finally:
        torch.set_num_threads(old)
    return {"value": BATCH * T_ref / wall, "unit": UNIT, "cores": cores, "kind": "reference",
            "sample": f"{T_ref} of {T_STEPS} timesteps of the same workload through the unmodified reference "
                      f"(bindsnet.models.DiehlAndCook2015.run, torch CPU, {cores} threads), {wall:.2f} s wall"}


def run_reference(args):
    """--impl reference: the live reference's own `DiehlAndCook2015.run` on the host cores — same network
    (n=1600, B=128, inh=120), same synthetic windows, every step a bounded T_ref-timestep sample of the
    250-step window (the reference costs ~seconds per timestep here: SURVEY.md §0.3)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch

    cores = host_threads()
    torch.set_num_threads(cores)
    models, why = import_reference()
    if models is None:
        emit({"impl": "reference", "unavailable": why})
        return
    torch.manual_seed(1234)
    net = models.DiehlAndCook2015(n_inpt=N_INPT, n_neurons=N_NEURONS, batch_size=BATCH, inpt_shape=(1, 28, 28), dt=1.0,
                                  nu=(1e-4, 1e-2), norm=78.4, theta_plus=0.05, exc=22.5, inh=120.0)
    xs = synth_windows(2, seed=999, T=16)
    # probe one timestep, then size T_ref so that the whole run stays within ~2 minutes
    t0 = time.perf_counter(); net.run({"X": xs[0][:1]}, time=1); probe = time.perf_counter() - t0
    total = max(args.steps + args.warmup, 1)
    T_ref = int(max(1, min(16, 120.0 / (total * max(probe, 1e-3)))))
    for i in range(args.warmup):
        net.reset_state_variables(); net.run({"X": xs[i % 2][:T_ref]}, time=T_ref)
    t0 = time.perf_counter()
    for i in range(args.steps):
        net.reset_state_variables(); net.run({"X": xs[i % 2][:T_ref]}, time=T_ref)
    wall = time.perf_counter() - t0
    value = BATCH * T_ref * args.steps / wall
    sample = (f"{args.steps} x {T_ref} timesteps of the {T_STEPS}-step window through bindsnet.models.DiehlAndCook2015.run "
              f"(unmodified reference, torch {torch.__version__} CPU, {cores} threads), state reset between steps")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * wall / max(args.steps, 1), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "global_batch": BATCH, "timesteps": T_STEPS,
                   "sample": f"each step is a {T_ref}-timestep sample of the {T_STEPS}-step window (state reset between steps)"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "reference", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    if not args.no_cpu_baseline:
        try:
            line["oracle_port"] = cpu_baseline(10.0)   # second, labelled leg: the C restatement on the same cores
        except Exception as e:
            line["oracle_port"] = {"unavailable": f"{type(e).__name__}: {e}"}
    emit(line)


_REAL_STDOUT = None


def quiet_stdout():
    """Libraries (NCCL's version banner, OpenMP, torchrun children) write to fd 1; the contract is ONE
    JSON line on stdout.  Everything but that line is sent to stderr."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line) -> None:
    data = (json.dumps(line) + "\n").encode()
    sys.stdout.flush()
    if _REAL_STDOUT is None:
        os.write(1, data)
    else:
        os.write(_REAL_STDOUT, data)


def run_config4(args) -> None:
    """BASELINE.json configs[3]: Input[1,32,32] -conv k5-> LIFNodes[16,28,28] -> Connection -> LIFNodes(10), MSTDP on both
    connections, Bernoulli(0.1) input, 500 timesteps, batch 128 — the generic window kernel (SURVEY.md §8a rows A11-A13).
    A diagnostic companion of the metric line: device-timed value, the end-to-end leg from pinned host spikes, and the
    oracle's dense restatement on the host cores on a bounded sample."""
    import torch

    import __graft_entry__ as entry
    from bindsnet_b200 import _backend
    from bindsnet_b200.learning import MSTDP
    from bindsnet_b200.network import Network, nodes, topology

    B, T = 128, 500

    def build(device):
        torch.manual_seed(7)
        net = Network(dt=1.0, batch_size=B)
        X = nodes.Input(shape=[1, 32, 32], traces=True)
        H = nodes.LIFNodes(shape=[16, 28, 28], traces=True)
        O = nodes.LIFNodes(n=10, traces=True)
        net.add_layer(X, "X"); net.add_layer(H, "H"); net.add_layer(O, "O")
        net.add_connection(topology.Conv2dConnection(X, H, kernel_size=5, update_rule=MSTDP, nu=1e-2, reduction=torch.sum,
                                                     wmin=-1.0, wmax=1.0), "X", "H")
        net.add_connection(topology.Connection(H, O, update_rule=MSTDP, nu=1e-2, reduction=torch.sum, wmin=-1.0, wmax=1.0), "H", "O")
        return net.to(device) if device is not None else net

    K, W = args.steps, min(max(args.warmup, 1), 2)
    g = torch.Generator().manual_seed(11)
    if args.impl == "reference":
        from oracle.oracle import OracleBackend

        cores, Ts = host_threads(), 10
        x = torch.bernoulli(0.1 * torch.ones(Ts, B, 1, 32, 32), generator=g).byte()
        ref = build(None)
        with OracleBackend(dense=1, threads=cores):
            ref.run({"X": x}, time=Ts, reward=1.0)
            t0 = time.perf_counter()
            for _ in range(K):
                ref.reset_state_variables(); ref.run({"X": x}, time=Ts, reward=1.0)
            wall = (time.perf_counter() - t0) / K
        v = B * Ts / wall
        emit({"impl": "reference", "metric": "sample·timesteps/s conv32x32-16ch-10 MSTDP b=128 (BASELINE.json configs[3])", "value": v, "unit": UNIT,
              "n_gpus": 1, "steps": K, "warmup": 1, "ms_per_step": wall * 1e3, "higher_is_better": True, "dtype": "f32", "data": "synthetic",
              "config": {"workload": "conv 32x32 k5 -> 16x28x28 -> 10, MSTDP on both connections, Bernoulli(0.1) input, B=128", "baseline_config": "c4"},
              "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                               "sample": f"{Ts} of {T} timesteps per step, dense mode, OpenMP with {cores} threads; the live reference's conv MSTDP "
                                         "raises for batch size > 1 (learning.py:2013), so the restatement stands in"},
              "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})
        return
    if not _backend.is_built():
        entry.build()
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    host = [torch.bernoulli(0.1 * torch.ones(T, B, 1, 32, 32), generator=g).byte().pin_memory() for _ in range(2)]
    resident = [h.to(dev) for h in host]
    net = build(dev)

    def window(x):
        net.reset_state_variables()
        net.run({"X": x}, time=T, reward=1.0)

    for i in range(W):
        window(resident[i & 1])
    torch.cuda.synchronize()
    l0 = _backend.launches_total
    with ClockSampler(0) as clocks:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(K):
            window(resident[i & 1])
        e1.record()
        torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / K
    launches = _backend.launches_total - l0
    net.check_errors()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, net)
    # end to end: pinned host spikes in, the output layer's spikes of the last step out, every window
    xdev = torch.empty_like(resident[0])
    out_host = torch.empty(B, 10, dtype=torch.bool).pin_memory()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(K):
        xdev.copy_(host[i & 1], non_blocking=True)
        window(xdev)
        out_host.copy_(net.layers["O"].s, non_blocking=True)
        torch.cuda.synchronize()
        int(out_host.sum())
    e1.record()
    torch.cuda.synchronize()
    ms2 = e0.elapsed_time(e1) / K
    emit({"metric": "sample·timesteps/s conv32x32-16ch-10 MSTDP b=128 (BASELINE.json configs[3])", "value": B * T / (ms * 1e-3), "unit": UNIT,
          "n_gpus": 1, "steps": K, "warmup": W, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
          "dtype": "f32", "data": "synthetic",
          "config": {"workload": "conv 32x32 k5 -> 16x28x28 -> 10, MSTDP on both connections, Bernoulli(0.1) input, B=128, 500 timesteps/window",
                     "global_batch": B, "timesteps": T, "parallelism": "single GPU", "kernel_tier": "generic", "baseline_config": "c4",
                     "l2": "two 65 MB input windows alternate (130 MB > 126 MB L2)"},
          "e2e": {"value": B * T / (ms2 * 1e-3), "unit": UNIT, "h2d_bytes_per_step": T * B * 1024, "d2h_bytes_per_step": B * 10,
                  "note": "pinned host uint8 spikes -> H2D -> Network.run(reward=1.0) -> output-layer spikes D2H, read on the host every window"},
          "gpu_launches": launches, "clocks": clocks.summary(),
          "roofline": c4_roofline(B, T, ms)})


def c4_roofline(B: int, T: int, ms: float) -> dict:
    """SURVEY.md §8d, config 4: input spikes as delivered + read and write of both weight tensors per timestep, state
    resident: B*1024 + 2*(12544*10*4 + 16*1*5*5*4) = 1 137 792 B/step at B = 128."""
    per_step = B * 1024 + 2 * (12544 * 10 * 4 + 16 * 25 * 4)
    peak, src = hbm_peak_gbs()
    ach = per_step * T / (ms * 1e-3) / 1e9
    return {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": None, "kernel_ms": ms,
            "algorithmic_bytes_per_timestep": per_step, "peak_source": src,
            "note": "generic tier; this configuration is not HBM-bound (SURVEY.md 8d: 0.14 us per step at the HBM peak): measured limiter = "
                    "instruction issue (ncu: 88 M warp-instructions per timestep, 1.1 IPC per SM at 25 % occupancy — the conv gather, the "
                    "per-sample eligibility and the [B,12544] neuron / trace / rule state streamed through L2 every step, which the "
                    "algorithmic figure counts as resident) plus three grid barriers per step"}


def main():
    quiet_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None,
                    help="timed windows (default: 320 = a timed region of >= 0.5 s at the metric configuration; 5 for c4, "
                         "which also runs its end-to-end loop and reference arm for that many windows)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--tier", type=int, default=0, help="0 auto, 1 generic kernel, 2 fused DC2015 kernel v1 (grid barrier), 3 fused DC2015 kernel v2 (message exchange)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--config", default="metric", choices=["metric", "c3", "c4"],
                    help="metric: the configuration BASELINE.json's metric is quoted on (DiehlAndCook2015 n=1600, B=128; default); "
                         "c3: configs[2] (n=6400, B=256); c4: configs[3] (conv 32x32 -> 16ch -> 10, MSTDP, 500 timesteps, B=128)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed windows, write the network state the last one left (spikes, voltages, traces, "
                         "thresholds, weights) to DIR/<name>.npy as float32; the inputs depend only on the arguments")
    args = ap.parse_args()
    if args.steps is None:
        args.steps = 5 if args.config == "c4" else 320
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the GPU path computed; it does not apply to --impl reference")
    apply_config(args.config)
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.config == "c4":
        return run_config4(args)
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist

    import __graft_entry__ as entry
    from bindsnet_b200 import _backend

    if not _backend.is_built():
        entry.build()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    from bindsnet_b200.distributed import ShardedWindowRunner
    from bindsnet_b200.network.monitors import Monitor

    net = make_network(dev)
    net.force_tier = args.tier
    runner = ShardedWindowRunner(net) if world > 1 else net
    host = [w.pin_memory() for w in synth_windows(POOL, seed=1234 + rank)]
    resident = [w.to(dev) for w in host]
    K, W = args.steps, args.warmup

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def window(x):
        net.reset_state_variables()  # between windows, like examples/mnist/batch_eth_mnist.py:321
        runner.run({"X": x}, time=T_STEPS)

    # ---- value: inputs resident in HBM ------------------------------------------------------
    for i in range(W):
        window(resident[i % POOL])
    barrier()
    _backend.kernel_events = []
    l0 = _backend.launches_total
    with ClockSampler(local) as clocks:
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(K):
            window(resident[(W + i) % POOL])
        e1.record()
        barrier()
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_total = float(ms)
    launches = _backend.launches_total - l0
    kern_ms = [a.elapsed_time(b) for a, b in _backend.kernel_events]
    _backend.kernel_events = None
    net.check_errors()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, net)   # before the passes below run the same network again
    value = world * BATCH * T_STEPS * K / (ms_total * 1e-3)

    # ---- the FIRST window of a fresh network (W0 as initialised, theta = 0: every neuron still fires easily, so the
    # winner / late-STDP paths are busier than in the steady state the loop above measures) ----------------
    first_ms = None
    if world == 1:
        net0 = make_network(dev)
        net0.force_tier = args.tier
        _backend.kernel_events = []
        net0.run({"X": resident[0]}, time=T_STEPS)
        torch.cuda.synchronize()
        first_ms = sum(a.elapsed_time(b) for a, b in _backend.kernel_events)
        _backend.kernel_events = None
        net0.check_errors()
        del net0

    # ---- the same loop with Ae + Ai spike monitors on (SURVEY.md §8d: report both) -------------------
    K2 = max(1, min(K, 5))
    for lname in ("Ae", "Ai"):
        net.add_monitor(Monitor(net.layers[lname], ["s"], time=T_STEPS, device=dev), f"{lname}_s")
    for i in range(2):
        window(resident[i % POOL])
    barrier()
    m0, m1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    m0.record()
    for i in range(K2):
        window(resident[(2 + i) % POOL])
    m1.record()
    barrier()
    msm = torch.tensor([m0.elapsed_time(m1)], device=dev)
    if world > 1:
        dist.all_reduce(msm, op=dist.ReduceOp.MAX)
    value_monitors = world * BATCH * T_STEPS * K2 / (float(msm) * 1e-3)
    for lname in ("Ae", "Ai"):
        del net.monitors[f"{lname}_s"]
    net.check_errors()

    # ---- e2e: host buffers through the public API, H2D + result D2H inside the timed region --
    from bindsnet_b200.network.monitors import SpikeCounter

    net.add_monitor(SpikeCounter(net.layers["Ae"]), "Ae_spikes")   # per-sample, per-neuron spike counts of the window
    from bindsnet_b200.pipeline import AsyncReadback, WindowPrefetcher

    consumed = [0, 0]  # windows read back on the host, total spikes seen there

    def use(counts_host):
        consumed[0] += 1
        # the host really reads the [B, n] int32 result (numpy: a single-threaded pass; torch's CPU
        # reduction would wake a 128-thread pool per call, which costs milliseconds on this box)
        consumed[1] += int(counts_host.numpy().sum())

    rb = AsyncReadback(depth=2)  # pinned host ring, allocated once

    def e2e_loop(n, first):
        # public API: WindowPrefetcher overlaps the pinned-host -> device copy of window k+1 with
        # the window kernel of window k; AsyncReadback brings window k's [B, n] spike counts to
        # pinned host memory while window k+1 is being launched.  Every copy happens inside the
        # loop (timed region), every result is read on the host before the loop returns.
        pre = WindowPrefetcher(dev, (host[(first + i) % POOL] for i in range(n)))
        for x_dev in pre:
            net.reset_state_variables()
            runner.run({"X": x_dev}, time=T_STEPS)
            pre.release()
            rb.push(net.monitors["Ae_spikes"].get("s"))   # D2H of the step's result
            if len(rb) == rb.depth:
                use(rb.pop())
        while len(rb):
            use(rb.pop())

    e2e_loop(W, 0)
    barrier()
    # host->device bandwidth of this box for one window of spikes (context for the e2e number:
    # 25 MB per window has to cross PCIe inside every timed step)
    h0, h1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    h0.record()
    resident[0].copy_(host[0], non_blocking=True)
    h1.record()
    torch.cuda.synchronize()
    h2d_gbs = host[0].numel() * host[0].element_size() / (h0.elapsed_time(h1) * 1e-3) / 1e9
    t0 = time.perf_counter()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    e2e_loop(K, W)
    e1.record()
    barrier()
    wall_e2e = time.perf_counter() - t0
    ms2 = torch.tensor([max(e0.elapsed_time(e1), 0.0)], device=dev)
    if world > 1:
        dist.all_reduce(ms2, op=dist.ReduceOp.MAX)
    e2e_value = world * BATCH * T_STEPS * K / (float(ms2) * 1e-3)
    net.check_errors()

    # ---- e2e from RATE IMAGES: the on-device encoder (bindsnet_b200.encoding.poisson on CUDA tensors, SURVEY.md §8f
    # rank 1) writes the spike tensor where Network.run reads it; only the [B, 1, 28, 28] float32 rate image
    # (400 KB instead of 25 MB) crosses PCIe per window, the result comes back as above -------------------------
    from bindsnet_b200.encoding import poisson as poisson_dev

    g = torch.Generator().manual_seed(4321 + rank)
    rate_host = [(128.0 * torch.rand(BATCH, 1, 28, 28, generator=g) * torch.bernoulli(0.19 * torch.ones(BATCH, 1, 28, 28), generator=g)).pin_memory()
                 for _ in range(POOL)]
    rate_dev = [torch.empty(BATCH, 1, 28, 28, device=dev) for _ in range(2)]

    def rates_loop(n, first):
        for i in range(n):
            r = rate_dev[i & 1]
            r.copy_(rate_host[(first + i) % POOL], non_blocking=True)          # H2D of this window's input
            x_dev = poisson_dev(r, time=T_STEPS, dt=1.0, seed=1000 + first + i)   # [T, B, 1, 28, 28] uint8, on the device
            net.reset_state_variables()
            runner.run({"X": x_dev}, time=T_STEPS)
            rb.push(net.monitors["Ae_spikes"].get("s"))
            if len(rb) == rb.depth:
                use(rb.pop())
        while len(rb):
            use(rb.pop())

    rates_loop(W, 0)
    barrier()
    r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    r0.record()
    rates_loop(K, W)
    r1.record()
    barrier()
    ms3 = torch.tensor([max(r0.elapsed_time(r1), 0.0)], device=dev)
    if world > 1:
        dist.all_reduce(ms3, op=dist.ReduceOp.MAX)
    e2e_rates_value = world * BATCH * T_STEPS * K / (float(ms3) * 1e-3)
    net.check_errors()

    if rank == 0:
        peak, peak_kind = hbm_peak_gbs()
        per_launch_bytes = algorithmic_bytes_per_timestep() * T_STEPS
        kavg_ms = sum(kern_ms) / max(len(kern_ms), 1)
        achieved = per_launch_bytes / (kavg_ms * 1e-3) / 1e9 if kavg_ms > 0 else 0.0
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "roofline_traffic.json")
        if os.path.exists(tpath) and args.config == "metric":
            try:
                traffic = json.load(open(tpath)).get("dram_bytes_per_launch")
            except Exception:
                traffic = None
        from bindsnet_b200 import _abi
        names = {1: "generic", 2: "fused_dc2015_v1", 3: "fused_dc2015_v2"}
        tier = names[args.tier] if args.tier else f"auto -> {names.get(_backend.last_tier, _backend.last_tier)}"
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms_total / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {
                "workload": WORKLOAD,
                "global_batch": world * BATCH, "timesteps": T_STEPS,
                "parallelism": f"dp{world}: batch shards, one NCCL all-reduce of dW+dtheta per window" if world > 1 else "single GPU",
                "l2": f"inputs cycle through {POOL} distinct windows ({POOL * T_STEPS * BATCH * N_INPT // 1000000} MB > 126 MB L2); the {N_INPT * N_NEURONS * 4 // 1000000} MB weight matrix is resident by design",
                "kernel_tier": tier, "state_reset_between_windows": True, "baseline_config": args.config,
            },
            "value_with_spike_monitors": value_monitors,  # Ae + Ai [T, B, n] rasters written by the kernel every window
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": T_STEPS * BATCH * N_INPT,
                    "d2h_bytes_per_step": BATCH * N_NEURONS * 4,
                    "note": "pinned host uint8 spike trains -> WindowPrefetcher (H2D on a side stream, overlapped) -> Network.run + SpikeCounter on Ae -> AsyncReadback: the [B, n] per-sample spike counts (what label assignment consumes) copied to pinned host memory and read there every window, one window behind the launches",
                    "wall_s": wall_e2e, "h2d_gbs_measured": h2d_gbs, "windows_read_on_host": consumed[0], "ae_spikes_seen_on_host": consumed[1]},
            "e2e_from_rates": {"value": e2e_rates_value, "unit": UNIT, "h2d_bytes_per_step": BATCH * N_INPT * 4,
                               "d2h_bytes_per_step": BATCH * N_NEURONS * 4,
                               "note": "pinned host float32 rate images [B,1,28,28] -> H2D -> bindsnet_b200.encoding.poisson on the device "
                                       "(snn_b200_encode_poisson) -> Network.run + SpikeCounter -> AsyncReadback; encoding inside the timed region"},
            "gpu_launches": launches,
            "clocks": clocks.summary(),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "peak_kind": peak_kind, "kernel_ms": kavg_ms, "first_window_kernel_ms": first_ms,
                         "algorithmic_bytes_per_launch": per_launch_bytes},
        }
        if world == 1 and not args.no_cpu_baseline:
            ref = reference_baseline(20.0)
            port = cpu_baseline()
            line["cpu_baseline"] = ref if ref is not None else port
            line["cpu_baseline_port"] = port   # the C restatement of the same path on the same cores, for orientation
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
