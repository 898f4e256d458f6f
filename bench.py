#!/usr/bin/env python
"""Benchmark of the spline-coupling hot path (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload two_moons_conditional|bounded16] [--dump-outputs DIR]
  python bench.py --impl reference ...        # the reference's CPU implementation of the path

One step = one ``Flow.__call__`` (log-prob) pass over one batch of synthetic events.  At N=1
the workload is the largest single-GPU configuration of BASELINE.json: configs[3] (bounded16:
16-D flow, ShiftBounds + 8 spline couplings, K=32, 16*2^20 events per step per GPU); configs[1]
(two_moons_conditional, 1M events) is reported beside it as ``extras.two_moons_conditional``.
With N>1 (torchrun, one rank per GPU) every rank evaluates its own batch - the eval path shards
over events with no data-path collective, so scaling is "weak" - and the time is the max over
ranks.  ``train_step`` is the data-parallel train step of configs[4] (64M events per optimiser
step, one fixed global batch sliced by rank, NCCL all-reduces), reported at every N.

Printed JSON (one line, rank 0): value = events/s with inputs resident in HBM; e2e = the same
metric through the public API from pinned HOST buffers (H2D of x and c, D2H of log_prob inside
the timed region); roofline for the dominant kernel; cpu_baseline = the numpy oracle ("port",
NOT the reference: JAX is not installable in this image) on a bounded sample of the same
workload.  ``--impl reference`` times that CPU port with all host cores.

``--dump-outputs DIR`` writes what the timed path returned in its last step (log_prob, float32) as DIR/log_prob.npy.
Inputs and parameters are seeded, so the same arguments give the same inputs and two builds can be compared.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # BASELINE.json configs[1]
    "two_moons_conditional": dict(D=2, C=1, K=16, layers=(128, 128), n_couplings=None, roll=1, M=1_000_000),
    # BASELINE.json configs[3] (16-D bounded flow, 8 couplings, K=32); M reduced by --batch
    "bounded16": dict(D=16, C=0, K=32, layers=(128, 128), n_couplings=8, roll=2, M=16 * 2 ** 20),
}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], bf16=d["bf16_tflops"], bf16_sustained=d.get("bf16_tflops_sustained"),
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm=6650.0, bf16=1590.0, bf16_sustained=1400.0, source="fallback (no MEASURED_PEAKS.json beside bench.py)")


def chain_flops_per_event(w):
    d = w["D"] // 2
    F = w["D"] - d + w["C"]
    widths = [F] + list(w["layers"]) + [d * (3 * w["K"] - 1)]
    per = 2 * sum(a * b for a, b in zip(widths[:-1], widths[1:]))
    n = w["D"] if w["n_couplings"] is None else w["n_couplings"]
    return per * n


def default_cpu_sample(w):
    """Bounded CPU sample: about 3e12 conditioner flops (10-30 s of work for the numpy port on 8-16 host cores)."""
    return int(max(20_000, min(40_000_000, 3e12 // chain_flops_per_event(w))))


def synth(w, M, seed):
    """Synthetic events of the workload's shape (two_moons_conditional: two noisy half circles
    with the class label as condition, as examples/two_moons_conditional.ipynb builds them)."""
    rng = np.random.default_rng(seed)
    if w["D"] == 2 and w["C"] == 1:
        lab = rng.integers(0, 2, M)
        t = rng.uniform(0, np.pi, M)
        x = np.where(lab == 0, np.cos(t), 1 - np.cos(t)) + 0.1 * rng.standard_normal(M)
        y = np.where(lab == 0, np.sin(t), 0.5 - np.sin(t)) + 0.1 * rng.standard_normal(M)
        return np.column_stack([x, y]).astype(np.float32), lab.astype(np.float32).reshape(-1, 1)
    x = rng.uniform(0, 1, (M, w["D"])).astype(np.float32)
    c = rng.uniform(0, 1, (M, w["C"])).astype(np.float32) if w["C"] else None
    return x, c


def oracle_ops(w):
    from oracle import zenflow_oracle as zo

    return zo.make_chain(w["D"], w["K"], w["layers"], n_couplings=w["n_couplings"], roll_shift=w["roll"])


def make_variables(w, seed=0):
    """Fixed-seed variables shared by both arms: LeCun-normal kernels, small random biases and
    BatchNorm statistics, ShiftBounds statistics from a 4096-event sample."""
    from oracle import zenflow_oracle as zo

    ops = oracle_ops(w)
    v = zo.init_variables(ops, w["D"], w["C"], seed, randomize_bn=True)
    xs, cs = synth(w, 4096, seed + 1)
    _, _, stats = zo.chain_forward(ops, v, xs, cs, train=True)
    v["batch_stats"]["bijectors_0"] = stats["bijectors_0"]
    return ops, v


# ----------------------------------------------------------------------------------------
# CPU arm: the numpy oracle over all host cores (fork pool, one BLAS thread per worker)
# ----------------------------------------------------------------------------------------
_G = {}


def _cpu_worker(args):
    lo, hi = args
    from oracle import zenflow_oracle as zo

    lp, _ = zo.flow_log_prob(_G["ops"], _G["v"], _G["x"][lo:hi], None if _G["c"] is None else _G["c"][lo:hi])
    return float(lp[np.isfinite(lp)].sum())


def cpu_events_per_s(w, sample, steps=1, warmup=0, cores=None):
    """Events/s of the CPU port on `sample` events per step, sharded over `cores` processes."""
    import multiprocessing as mp

    try:
        from threadpoolctl import threadpool_limits
        threadpool_limits(1)
    except Exception:
        pass
    cores = cores or os.cpu_count() or 1
    ops, v = make_variables(w)
    x, c = synth(w, sample, 123)
    _G.update(ops=ops, v=v, x=x, c=c)
    chunk = int(min(16384, max(256, -(-sample // (4 * cores)))))   # every worker gets several shards per step
    shards = [(i, min(sample, i + chunk)) for i in range(0, sample, chunk)]
    ctx = mp.get_context("fork")
    with ctx.Pool(cores) as pool:
        for _ in range(warmup):
            pool.map(_cpu_worker, shards)
        t0 = time.perf_counter()
        for _ in range(steps):
            pool.map(_cpu_worker, shards)
        dt = time.perf_counter() - t0
    return sample * steps / dt, dt / steps, cores


def run_reference(args):
    """`--impl reference`: the reference's own CPU path.  The real reference needs
    jax+flax+optax (absent from this image and from the GPU box) - try it, else time the
    CPU port of the same path (oracle/) with every host core."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    w = WORKLOADS[args.workload]
    kind = "port"
    try:  # pragma: no cover - cannot succeed in this image
        sys.path.insert(0, "/root/reference/src")
        import jax  # noqa: F401
        import flax  # noqa: F401
        kind = "reference"
    except Exception:
        pass
    # bounded: the whole (--warmup W + --steps K) run stays within ~3x the default sample (a few minutes at most)
    K, W = max(1, args.steps), max(0, args.warmup)
    sample = args.cpu_sample or max(10_000, 3 * default_cpu_sample(w) // (K + W))
    value, sec, cores = cpu_events_per_s(w, sample, steps=K, warmup=W)
    line = {
        "impl": "reference", "metric": "flow_log_prob_events_per_s", "value": value, "unit": "events/s",
        "n_gpus": args.gpus, "steps": K, "warmup": W, "ms_per_step": sec * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": bench_config(args.workload, w, args.batch or w["M"]),
        "cpu_baseline": {"value": value, "unit": "events/s", "cores": cores, "kind": kind,
                         "sample": f"{sample} events/step (bounded sample of the workload in config), numpy fp32 "
                                   f"restatement of the reference path (JAX not installable here), {cores} forked "
                                   f"workers x 1 BLAS thread"},
        "e2e": {"value": value, "unit": "events/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ----------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------
class ClockSampler:
    QUERY = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={index}", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                 "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def stop(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        allsm = []
        for t, line in self.rows:
            p = [v.strip() for v in line.split(",")]
            if len(p) < 7:
                continue
            try:
                clk, mx_ = float(p[0]), float(p[1])
            except ValueError:
                continue
            mx = mx_
            allsm.append(clk)
            if t0 <= t <= t1 + 0.06:
                sm.append(clk)
                for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[3:7]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
        use = sm or allsm[-3:]
        return {"sm_mhz": float(np.median(use)) if use else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def build_flow(w, dev):
    """(flow, variables on `dev`) of a workload, from the fixed-seed variables both arms share."""
    import torch

    from zenflow_b200 import Flow
    from zenflow_b200 import bijectors as bi
    from zenflow_b200.distributions import Beta

    ops, v = make_variables(w)
    mods = []
    for op in ops:
        if op["kind"] == "shift_bounds":
            mods.append(bi.ShiftBounds(margin=op["margin"], bounds=op["bounds"]))
        elif op["kind"] == "roll":
            mods.append(bi.Roll(op["shift"]))
        else:
            mods.append(bi.NeuralSplineCoupling(knots=op["knots"], layers=op["layers"]))
    flow = Flow(bi.Chain(mods), latent=Beta())   # its own latent: the default instance is shared and latches one dim
    tree = {"params": {"bijector": v["params"]}, "batch_stats": {"bijector": v["batch_stats"]}}
    variables = torch.utils._pytree.tree_map(lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev), tree)
    flow.latent._latch_dim(w["D"])
    return flow, variables


def ncu_traffic(workload, M):
    """DRAM bytes per launch of the dominant kernel, from the committed ncu --set full capture of this exact
    (workload, events) pair (profiles/r02_traffic.json: dram__bytes_read.sum + dram__bytes_write.sum)."""
    p = os.path.join(ROOT, "profiles", "r02_traffic.json")
    if not os.path.exists(p):
        return None
    return json.load(open(p)).get(f"{workload}:{M}")


DUMP_MAX_ROWS = 1 << 22   # 16 MiB of float32 per dumped 1-D array


def dump_outputs(out_dir, arrays):
    """Write each array as out_dir/<name>.npy in float32.  An array of more than DUMP_MAX_ROWS rows is replaced by a
    fixed sample of them: the rows np.sort(np.random.default_rng(0).choice(rows, DUMP_MAX_ROWS, replace=False)), so
    runs with the same arguments write the same rows and two builds can be compared output for output."""
    import torch

    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        n = a.shape[0]
        if n > DUMP_MAX_ROWS:
            idx = np.sort(np.random.default_rng(0).choice(n, DUMP_MAX_ROWS, replace=False))
            a = a[torch.from_numpy(idx).to(a.device)]
        np.save(os.path.join(out_dir, name + ".npy"), a.float().cpu().numpy())


def loop_events_per_s(fn, n_events, min_seconds=0.5, warm=3):
    """Device-timed events/s of fn(i) repeated until at least `min_seconds` have been timed (extras)."""
    import torch

    for i in range(warm):
        fn(i)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps, done, ms = 3, 0, 0.0
    while True:
        a.record()
        for i in range(reps):
            fn(warm + done + i)
        b.record()
        torch.cuda.synchronize()
        ms += a.elapsed_time(b)
        done += reps
        if ms >= min_seconds * 1e3 or done >= 4000:
            break
        reps = int(min(2000, max(3, reps * 1.5 * (min_seconds * 1e3 - ms) / max(ms / done, 1e-3) / max(reps, 1) + 1)))
    return n_events * done / (ms * 1e-3), ms / done, done


def run_gpu(args):
    import torch
    import torch.distributed as dist

    from zenflow_b200 import _lib
    from zenflow_b200.utils import rqs_forward_raw

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    # stdout carries exactly ONE JSON line (rank 0): whatever libraries print meanwhile (NCCL's version banner ...)
    # goes to stderr; the descriptor is restored for the final print
    sys.stdout.flush()
    stdout_fd = os.dup(1)
    os.dup2(2, 1)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    w = dict(WORKLOADS[args.workload])
    if args.batch:
        w["M"] = args.batch
    M = w["M"]
    flow, variables = build_flow(w, dev)

    # Inputs beyond L2 (126 MB): either one set is already larger, or enough rotating sets to exceed it twice
    bytes_in = 4 * M * (w["D"] + w["C"])
    bytes_out = 4 * M
    n_sets = min(24, max(2, int(np.ceil(2 * 126e6 / (bytes_in + bytes_out)))))
    xs_h, cs_h = [], []
    for i in range(n_sets):
        x, c = synth(w, M, 1000 + 97 * rank + i)
        xs_h.append(torch.from_numpy(x).pin_memory())
        cs_h.append(None if c is None else torch.from_numpy(c).pin_memory())
    xs_d = [t.to(dev) for t in xs_h]
    cs_d = [None if t is None else t.to(dev) for t in cs_h]
    lp_host = torch.empty(M, dtype=torch.float32).pin_memory()

    def step_device(i):
        return flow.apply(variables, xs_d[i % n_sets], cs_d[i % n_sets])

    # e2e: every step copies its inputs from pinned host memory and its result back to the host.
    # Copies run on side streams so that step i+1's H2D and step i-1's D2H overlap step i's kernel
    # (double-buffered device staging buffers and host result buffers); all of it is inside the timed
    # region: the last step's D2H is drained into the compute stream before the closing event.
    copy_stream = torch.cuda.Stream(device=dev)
    d2h_stream = torch.cuda.Stream(device=dev)
    d2h_done = [torch.cuda.Event() for _ in range(2)]
    lp_hosts = [lp_host, torch.empty(M, dtype=torch.float32).pin_memory()]
    lp_keep = [None, None]   # the device result stays referenced until its copy has been waited for
    stage_x = [torch.empty_like(xs_d[0]) for _ in range(2)]
    stage_c = [None if cs_d[0] is None else torch.empty_like(cs_d[0]) for _ in range(2)]
    h2d_done = [torch.cuda.Event() for _ in range(2)]
    compute_done = [torch.cuda.Event() for _ in range(2)]
    e2e_state = {"primed": -1}

    def _h2d(i):
        b = i & 1
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(compute_done[b])  # the kernel that last read this staging buffer
            stage_x[b].copy_(xs_h[i % n_sets], non_blocking=True)
            if stage_c[b] is not None:
                stage_c[b].copy_(cs_h[i % n_sets], non_blocking=True)
            h2d_done[b].record(copy_stream)

    def step_e2e(i):
        cur = torch.cuda.current_stream()
        if e2e_state["primed"] != i:
            _h2d(i)
        _h2d(i + 1)
        e2e_state["primed"] = i + 1
        b = i & 1
        cur.wait_event(h2d_done[b])
        cur.wait_event(d2h_done[b])     # step i-2's result has left the device: its buffer may be reused
        lp = flow.apply(variables, stage_x[b], stage_c[b])
        compute_done[b].record(cur)
        lp_keep[b] = lp
        with torch.cuda.stream(d2h_stream):
            d2h_stream.wait_event(compute_done[b])
            lp_hosts[b].copy_(lp, non_blocking=True)  # the result back, overlapping the next step's kernel
            d2h_done[b].record(d2h_stream)
        return lp

    def drain_e2e():
        cur = torch.cuda.current_stream()
        for e in d2h_done:
            cur.wait_event(e)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(step, K, W, drain=None):
        for i in range(W):
            step(i)
        barrier()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
        l0 = _lib.launch_count()
        t0 = time.perf_counter()
        for i in range(K):
            ev[i][0].record()
            out = step(W + i)
            if drain is not None and i == K - 1:
                drain()
            ev[i][1].record()
        barrier()
        t1 = time.perf_counter()
        launches = _lib.launch_count() - l0
        total_ms = ev[0][0].elapsed_time(ev[-1][1])  # device time of exactly K back-to-back steps
        per = [a.elapsed_time(b) for a, b in ev]
        if world > 1:
            t = torch.tensor([total_ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            total_ms = float(t.item())
        return total_ms, per, launches, (t0, t1), out

    K, W = args.steps, max(args.warmup, 3)
    sampler = ClockSampler(local) if rank == 0 else None
    total_ms, per, launches, (t0, t1), lp_last = timed(step_device, K, W)
    clocks = sampler.stop(t0, t1) if sampler else None
    value = world * M * K / (total_ms * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"log_prob": lp_last})   # what Flow.__call__ returned in the last timed step
    del lp_last

    e2e_ms, _, _, _, _ = timed(step_e2e, K, W, drain=drain_e2e)
    e2e_value = world * M * K / (e2e_ms * 1e-3)
    # the host buffer of the last timed step must hold that step's result (bit-exact against a device-resident rerun)
    last = W + K - 1
    torch.cuda.synchronize()
    ref = flow.apply(variables, xs_d[last % n_sets], cs_d[last % n_sets])
    e2e_checked = bool(torch.equal(lp_hosts[last & 1], ref.cpu()))
    if not e2e_checked:
        raise RuntimeError("e2e pipeline returned a result that differs from the device-resident path")
    del ref

    extras = {}
    pk = peaks()
    if rank == 0 and world == 1:
        # Flow.sample of the same workload: (i) in-kernel Philox latent draw + inverse chain (the public
        # ``method="sample"``), (ii) the inverse chain on a given latent draw u (the parity mode)
        cond = cs_d[0]
        n_ev = M

        def step_sample(i):
            return flow.apply(variables, cond if cond is not None else n_ev, method="sample", seed=i)

        def step_inv(i):
            return flow.apply(variables, u, cs_d[i % n_sets], method="inverse")

        v_s, ms_s, n_s = loop_events_per_s(step_sample, n_ev, 0.6)
        extras["sample_events_per_s"] = v_s
        extras["sample"] = {"value": v_s, "unit": "events/s", "ms_per_step": ms_s, "steps": n_s,
                            "what": "Flow.sample: Philox latent draw fused into the inverse chain kernel"}
        u = torch.rand(M, w["D"], device=dev) * 0.8 + 0.1
        v_i, ms_i, n_i = loop_events_per_s(step_inv, n_ev, 0.6)
        extras["inverse_events_per_s"] = v_i
        extras["inverse"] = {"value": v_i, "unit": "events/s", "ms_per_step": ms_i, "steps": n_i,
                             "what": "Chain.inverse on a given latent draw (parity mode of Flow.sample)"}
        del u

        # the other single-GPU eval config of BASELINE.json (configs[1] when the headline is configs[3] and vice versa)
        other = "two_moons_conditional" if args.workload != "two_moons_conditional" else "bounded16"
        if not args.no_extras:
            w2 = dict(WORKLOADS[other])
            if other == "bounded16":
                w2["M"] = 4 * 2 ** 20
            flow2, vars2 = build_flow(w2, dev)
            ns2 = min(24, max(2, int(np.ceil(2 * 126e6 / (4 * w2["M"] * (w2["D"] + w2["C"] + 1))))))
            sets2 = [synth(w2, w2["M"], 5000 + i) for i in range(ns2)]
            x2 = [torch.from_numpy(a).to(dev) for a, _ in sets2]
            c2 = [None if b is None else torch.from_numpy(b).to(dev) for _, b in sets2]
            v_lp, ms_lp, n_lp = loop_events_per_s(lambda i: flow2.apply(vars2, x2[i % ns2], c2[i % ns2]), w2["M"], 1.0)
            v_sm, ms_sm, _ = loop_events_per_s(
                lambda i: flow2.apply(vars2, c2[i % ns2] if c2[0] is not None else w2["M"], method="sample", seed=i),
                w2["M"], 0.5)
            fl2 = chain_flops_per_event(w2)
            extras[other] = {
                "config": {"workload": other, "events_per_step": w2["M"], "D": w2["D"], "C": w2["C"], "K": w2["K"],
                           "l2": f"rotating {ns2} input sets"},
                "log_prob_events_per_s": v_lp, "ms_per_step": ms_lp, "steps": n_lp, "sample_events_per_s": v_sm,
                "sample_ms_per_step": ms_sm, "tflops_algorithmic": fl2 * v_lp / 1e12,
                "roofline_frac_tensor": fl2 * v_lp / 1e12 / pk["bf16"], "traffic": ncu_traffic(other, w2["M"])}
            del x2, c2, flow2, vars2

        # the standalone spline stage of this workload's shape against the HBM roof
        d = w["D"] // 2
        P = 3 * w["K"] - 1
        Ms = int(1.5e9 // (4 * d * P))  # 1.5 GB of theta: an order of magnitude beyond L2
        theta = torch.randn(Ms, d, P, device=dev)
        xin = torch.rand(Ms, d, device=dev)
        for _ in range(3):
            rqs_forward_raw(xin, theta, w["K"])
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 20
        a.record()
        for _ in range(reps):
            rqs_forward_raw(xin, theta, w["K"])
        b.record()
        torch.cuda.synchronize()
        st_ms = a.elapsed_time(b) / reps
        alg = 4.0 * (d * P + 2 * d + 1) * Ms
        extras["roofline_spline_stage"] = {
            "kernel": "rqs_stage_kernel (zf_rqs_forward)", "bound": "hbm", "achieved": alg / st_ms / 1e6,
            "peak": pk["hbm"], "unit": "GB/s", "frac": alg / st_ms / 1e6 / pk["hbm"],
            "traffic": ncu_traffic("rqs_stage", Ms), "events": Ms, "bytes_per_event": 4 * (d * P + 2 * d + 1),
            "peak_source": pk["source"]}
        del theta, xin

    # free the eval buffers before the train step takes its share of HBM
    del xs_d, cs_d, stage_x, stage_c, lp_keep
    torch.cuda.empty_cache()
    train_info = bench_train(args, world, rank, dev) if args.train_batch else None
    if rank == 0 and world == 1 and args.deep_set and not args.no_extras:
        extras["deep_set_train_step"] = bench_deep_set(dev)
        extras["small_batch_train_step"] = bench_small_batch_train(dev)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    flops = chain_flops_per_event(w)
    step_ms = total_ms / K
    tflops = flops * M / (step_ms * 1e-3) / 1e12
    simt = os.environ.get("ZF_CHAIN_IMPL", "").startswith("s")
    pp = (w["D"] // 2 == 1) and not simt   # single-dim couplings run the two-tiles-in-flight kernel
    roofline = {
        "kernel": ("chain_kernel<false>: fused conditioner MLPs (fp32 FFMA) + splines + latent" if simt else
                   ("chain_umma_pp_kernel<false>" if pp else "chain_umma_kernel<false>") +
                   " (zf_flow_log_prob): conditioner GEMMs on tcgen05 (3xFP16 split on kind::f16, A in TMEM), "
                   "spline rows read theta from TMEM, latent fused" + ("; two tiles in flight" if pp else "")),
        "bound": "tensor", "achieved": tflops, "peak": pk["bf16"], "unit": "TFLOP/s", "frac": tflops / pk["bf16"],
        "traffic": ncu_traffic(args.workload, M), "flops_per_event": flops,
        "note": "algorithmic fp32 flops (not x3 for the 3xFP16 split: kind::f16 runs at the bf16 rate, so the tensor "
                "pipe executes 3 bf16-equivalents per algorithmic flop); achieved uses the whole step time "
                "(the pack launch included); peak = burst bf16 figure of MEASURED_PEAKS.json, the sustained one "
                "gives frac_sustained; see DESIGN.md for what bounds the kernel (tensor-memory read port + issue slots "
                "of the spline rows, not the tensor pipe)",
        "frac_sustained": (tflops / pk["bf16_sustained"]) if pk.get("bf16_sustained") else None,
        "tensor_pipe_bf16_equivalent_frac": 3 * tflops / pk["bf16"],
        "frac_of_fp32_simt_peak": tflops / 74.4, "peak_source": pk["source"]}

    cpu_sample = args.cpu_sample or default_cpu_sample(w)
    cpu_value, cpu_sec, cores = cpu_events_per_s(w, cpu_sample, steps=1, warmup=0) if world == 1 else (None, None, None)

    line = {
        "metric": "flow_log_prob_events_per_s", "value": value, "unit": "events/s", "n_gpus": world, "steps": K,
        "warmup": W, "ms_per_step": step_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": bench_config(args.workload, w, M),
        "timed_region_s": total_ms * 1e-3,
        "e2e": {"value": e2e_value, "unit": "events/s", "h2d_bytes_per_step": bytes_in, "d2h_bytes_per_step": bytes_out,
                "ms_per_step": e2e_ms / K, "result_checked": e2e_checked},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "roofline": roofline,
        "step_ms_min_median_max": [float(np.min(per)), float(np.median(per)), float(np.max(per))],
    }
    if cpu_value is not None:
        line["cpu_baseline"] = {"value": cpu_value, "unit": "events/s", "cores": cores, "kind": "port",
                                "sample": f"{cpu_sample} events, numpy fp32 restatement of the reference path "
                                          f"(JAX not installable here), {cores} forked workers x 1 BLAS thread, "
                                          f"{cpu_sec:.1f} s"}
    line.update(extras)
    if train_info:
        line["train_step"] = train_info
    sys.stdout.flush()
    os.dup2(stdout_fd, 1)
    print(json.dumps(line), flush=True)
    os.dup2(2, 1)
    if world > 1:
        dist.destroy_process_group()


def bench_small_batch_train(dev, rows=1000, steps=300):
    """The optimiser step as the reference's train() runs it (train.py:80-86,110-117: minibatches of ~1000 rows) on
    two_moons_conditional: bound by the step's launches, so TrainEngine replays it as one CUDA graph (eager beside it)."""
    import torch

    from zenflow_b200 import _lib
    from zenflow_b200._train import TrainEngine

    w = dict(WORKLOADS["two_moons_conditional"])
    out = {"config": {"workload": "two_moons_conditional", "rows_per_step": rows, "D": w["D"], "C": w["C"], "K": w["K"],
                      "optimizer": "nadamw(1e-3)", "data": f"{steps} different minibatches"}}
    x, c = synth(w, rows * 8, 777)
    xd, cd = torch.from_numpy(x).to(dev), torch.from_numpy(c).to(dev)
    for graphs in (False, True):
        flow, variables = build_flow(w, dev)
        eng = TrainEngine(flow, variables, w["D"], w["C"])
        eng.use_graphs = graphs
        batch = lambda i: (xd[(i % 8) * rows:(i % 8 + 1) * rows], cd[(i % 8) * rows:(i % 8 + 1) * rows])
        for i in range(5):
            eng.step(*batch(i))
        torch.cuda.synchronize()
        n0 = _lib.launch_count()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for i in range(steps):
            lp_sum = eng.step(*batch(i))
        b.record()
        torch.cuda.synchronize()
        ms = a.elapsed_time(b) / steps
        key = "graph" if graphs else "eager"
        out[key] = {"ms_per_step": ms, "samples_per_s": rows / ms * 1e3,
                    "gpu_launches_per_step": (_lib.launch_count() - n0) / steps,
                    "loss_last": -float(lp_sum.item()) / rows}
    out["what"] = ("zf_flow_value_and_grad + zf_nadamw_update_dev per step; 'graph' = the captured step replayed as one "
                   "CUDA-graph launch (the default for single-device steps of <= 65,536 rows)")
    return out


def bench_deep_set(dev):
    """BASELINE.json configs[2] (deep_set conditional): examples/deep_set.ipynb's data (1000 sets, sizes
    int(400 Exp / max Exp) + 1, elements N(0,1)^2 padded to 50,000 rows, y ~ N(sqrt(n), 1)^2), DeepSetFlow =
    Phi (BatchNorm -> 3 x Dense(128) -> Dense(8) -> Dropout -> sum-pool) feeding rolling_spline_coupling(2,
    layers=(128,)*6).  Two timings: the flow's fused forward+backward step given c, returning d loss / d c
    (SURVEY.md 8d cfg3), and the whole joint step (Phi forward, flow value-and-grad, Phi backward, AdamW on both)."""
    import torch

    from zenflow_b200 import Flow, _lib
    from zenflow_b200.bijectors import rolling_spline_coupling
    from zenflow_b200.deep_set import DeepSetFlowTrainer, Phi, SumMatrix
    from zenflow_b200.distributions import Beta

    rng = np.random.default_rng(1)
    n = rng.exponential(size=1000)
    n *= 400 / np.max(n)
    sizes = (n + 1).astype(int)
    X = np.concatenate([rng.normal(size=(ni, 2)) for ni in sizes])
    X = np.concatenate([X, np.zeros((50_000 - len(X), 2))]).astype(np.float32)
    y = rng.normal(np.sqrt(sizes), 1, size=(2, len(sizes))).T.astype(np.float32)
    phi = Phi()
    flow = Flow(rolling_spline_coupling(2, layers=(128,) * 6), latent=Beta())
    tr = DeepSetFlowTrainer(phi, phi.init(0, X), flow, flow.init(0, y[:1], np.zeros((1, 8), np.float32)), 2, 2)
    sm = SumMatrix.from_sizes(sizes)
    Xd, yd = torch.from_numpy(X).to(dev), torch.from_numpy(y).to(dev)
    c = tr.phi_eng.forward(Xd, sm, train=False)

    def timed(fn, reps):
        for i in range(5):
            fn(i)
        torch.cuda.synchronize()
        l0 = _lib.launch_count()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for i in range(reps):
            fn(5 + i)
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / reps, (_lib.launch_count() - l0) / reps

    flow_ms, flow_l = timed(lambda i: tr.flow_eng.step(yd, c, want_gc=True, update=False), 100)
    joint_ms, joint_l = timed(lambda i: tr.step(Xd, sm, yd, seed=i), 100)
    losses = [-float(tr.step(Xd, sm, yd, seed=1000 + i).item()) / len(sizes) for i in range(3)]
    return {"config": {"workload": "deep_set", "sets": int(len(sizes)), "rows": 50_000, "D": 2, "C": 8, "K": 16,
                       "layers": [128] * 6, "phi": "BatchNorm -> 3 x Dense(128) -> Dense(8) -> Dropout(0.3) -> sum-pool"},
            "flow_step_given_c": {"ms_per_step": flow_ms, "events_per_s": len(sizes) / flow_ms * 1e3,
                                  "gpu_launches_per_step": flow_l,
                                  "what": "zf_flow_value_and_grad: loss, parameter gradients and d loss / d c, one call"},
            "joint_step": {"ms_per_step": joint_ms, "sets_per_s": len(sizes) / joint_ms * 1e3,
                           "rows_per_s": 50_000 / joint_ms * 1e3, "gpu_launches_per_step": joint_l,
                           "what": "Phi forward (train) + flow value-and-grad + Phi backward + AdamW on both"},
            "loss_after_205_steps": losses[-1],
            "note": "1000 events per step: this config is launch-latency-bound (one batch-statistics phase per bijector)"}


def bench_config(workload, w, M):
    """The `config` object both arms print (the CPU arm's bounded sample is described in cpu_baseline.sample)."""
    bytes_io = 4 * M * (w["D"] + w["C"] + 1)
    n_sets = min(24, max(2, int(np.ceil(2 * 126e6 / bytes_io))))
    return {"workload": workload, "events_per_step_per_gpu": M, "D": w["D"], "C": w["C"], "K": w["K"],
            "layers": list(w["layers"]), "couplings": w["D"] if w["n_couplings"] is None else w["n_couplings"],
            "latent": "Beta(12)", "l2": f"rotating {n_sets} input sets ({n_sets * bytes_io / 1e6:.0f} MB > 126 MB L2)",
            "seed": 0}


def cond16_flow():
    """BASELINE.json configs[4]: 16-D conditional flow, C=4, K=32, ShiftBounds + 8 couplings with Roll(2)."""
    from zenflow_b200 import Flow
    from zenflow_b200 import bijectors as bi

    D, C, K, n_c = 16, 4, 32, 8
    mods = [bi.ShiftBounds()]
    for i in range(n_c - 1):
        mods += [bi.NeuralSplineCoupling(knots=K, layers=(128, 128)), bi.Roll(2)]
    mods.append(bi.NeuralSplineCoupling(knots=K, layers=(128, 128)))
    flow = Flow(bi.Chain(mods))
    variables = flow.init(0, np.zeros((1, D), np.float32), np.zeros((1, C), np.float32))
    return flow, variables, D, C, K, n_c


def global_batch_slice(global_batch, width, seed, lo, hi, dev):
    """Rows [lo, hi) of ONE fixed synthetic global batch (uniform in (0,1)), identical for every world size:
    the batch is generated in fixed 1M-row blocks from a counter-free per-block seed, so a rank only materialises
    the blocks that overlap its slice."""
    import torch

    blk = 1 << 20
    out = torch.empty(hi - lo, width, dtype=torch.float32, device=dev)
    g = torch.Generator(device=dev)
    for b0 in range(lo // blk * blk, hi, blk):
        g.manual_seed(seed * 1_000_003 + b0 // blk)
        rows = min(blk, global_batch - b0)
        t = torch.rand(rows, width, device=dev, generator=g)
        s0, s1 = max(lo, b0), min(hi, b0 + rows)
        out[s0 - lo:s1 - lo] = t[s0 - b0:s1 - b0]
    return out


def bench_train(args, world, rank, dev):
    """The data-parallel train step of train.py:80-86 on BASELINE.json configs[4] (16-D conditional flow, C=4,
    K=32, 8 couplings, Roll(2)): ONE fixed global batch of --train-batch events (default 64*2^20) sliced evenly by
    rank (strong scaling: the loss is the same at every N), BatchNorm / ShiftBounds statistics and the flat
    gradient all-reduced with NCCL.  Samples/s = global batch / step time (max over ranks)."""
    import torch
    import torch.distributed as dist

    from zenflow_b200._train import TrainEngine

    flow, variables, D, C, K, n_c = cond16_flow()
    gb = args.train_batch // world * world
    local = gb // world
    x = global_batch_slice(gb, D, 1234, rank * local, (rank + 1) * local, dev)
    c = global_batch_slice(gb, C, 4321, rank * local, (rank + 1) * local, dev)
    kw = {}
    if args.train_micro_batch:
        kw["micro_batch"] = args.train_micro_batch
    eng = TrainEngine(flow, variables, D, C, group=None, **kw)
    steps, warm = args.train_steps, args.train_warmup
    losses = []
    for _ in range(warm):
        losses.append(eng.step(x, c, global_count=gb).clone())
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    from zenflow_b200 import _lib
    l0 = _lib.launch_count()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        losses.append(eng.step(x, c, global_count=gb).clone())
    b.record()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    launches = _lib.launch_count() - l0
    ms = a.elapsed_time(b)
    ls = torch.cat(losses)          # per-step sums of log-probs over this rank's slice
    tm = torch.tensor([ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        dist.all_reduce(ls, op=dist.ReduceOp.SUM)
    ms = float(tm.item())
    loss_per_step = [-float(v) / gb for v in ls.tolist()]
    flops_fwd = 2 * ((D - D // 2 + C) * 128 + 128 * 128 + 128 * (D // 2) * (3 * K - 1)) * n_c
    return {"samples_per_s": gb * steps / (ms * 1e-3), "ms_per_step": ms / steps, "global_batch": gb,
            "steps": steps, "warmup": warm, "n_gpus": world, "scaling": "strong",
            "loss": loss_per_step[0], "loss_per_step": [float(f"{v:.9g}") for v in loss_per_step],
            "gpu_launches": int(launches), "micro_batch": eng.micro_batch,
            "config": {"workload": "cond16_train", "D": D, "C": C, "K": K, "couplings": n_c, "layers": [128, 128],
                       "optimizer": "nadamw(1e-3)", "data": "one fixed global batch (seed 1234/4321) sliced by rank",
                       "collectives": eng.collectives_note()},
            "tflops_algorithmic": 3 * flops_fwd * gb / (ms / steps * 1e-3) / 1e12,
            "roofline_frac_tensor": 3 * flops_fwd * gb / (ms / steps * 1e-3) / 1e12 / peaks()["bf16"],
            "note": "loss_per_step[0] is the loss of the initial parameters on the fixed global batch: identical at "
                    "every N up to the summation order of the all-reduced double sums"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--workload", default="bounded16", choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=0, help="override events per step per GPU")
    ap.add_argument("--cpu-sample", type=int, default=0)
    ap.add_argument("--train-batch", type=int, default=64 << 20,
                    help="global batch of the data-parallel train step (BASELINE configs[4]: 64M; 0: skip)")
    ap.add_argument("--train-steps", type=int, default=2)
    ap.add_argument("--train-warmup", type=int, default=1)
    ap.add_argument("--train-micro-batch", type=int, default=0, help="override TrainEngine's micro-batch (0: default)")
    ap.add_argument("--no-extras", action="store_true", help="skip the extra legs (other eval config, deep_set)")
    ap.add_argument("--deep-set", type=int, default=1, help="run the deep_set (configs[2]) train-step leg at N=1")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the log_prob of the last timed step (rank 0) to DIR/log_prob.npy, float32; beyond "
                         f"{DUMP_MAX_ROWS} events a fixed sample of them")
    args = ap.parse_args()
    if args.impl == "native" and args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the native path computed; the reference arm has no such output")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
