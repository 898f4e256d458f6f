"""Throughput of the eval-mode log-density and its VJP (zf_flow_log_prob_vjp) on the bench workloads.

For bounded16 (configs[3]: 16-D, ShiftBounds + 8 couplings, K = 32, 16M events) and two_moons_conditional (configs[1]:
2-D conditional, 1M events) it times three calls with CUDA events, each warmed up and repeated:
  log_prob      zf_flow_log_prob (Flow.__call__(train=False))
  vjp_inputs    zf_flow_log_prob_vjp with grads = NULL: d/dx and d/dc only
  vjp_params    zf_flow_log_prob_vjp with the parameter gradients as well
The inputs are far larger than L2 (bounded16: 1 GiB of x), so each pass streams from HBM.  The card's name and power
limit are read in the same run and stored beside the numbers.  Output: JSON on stdout (and in --out FILE); progress on
stderr.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from zenflow_b200 import Flow  # noqa: E402
from zenflow_b200 import bijectors as bi  # noqa: E402
from zenflow_b200._chain import ChainSpec  # noqa: E402

WORKLOADS = {
    "two_moons_conditional": dict(D=2, C=1, K=16, layers=(128, 128), n_couplings=2, roll=1, M=1_000_000),
    "bounded16": dict(D=16, C=0, K=32, layers=(128, 128), n_couplings=8, roll=2, M=16 * 2 ** 20),
}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    lines = q.stdout.strip().splitlines() if q.returncode == 0 else []
    line = lines[torch.cuda.current_device()] if torch.cuda.current_device() < len(lines) else "; ".join(lines)
    return dict(torch_name=torch.cuda.get_device_name(), nvidia_smi=line)


def timeit(fn, n, warm=2):
    for _ in range(warm):
        fn()
        torch.cuda.synchronize()
        print("  warm-up call done", file=sys.stderr, flush=True)
    ts = []
    for _ in range(n):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    ts.sort()
    return dict(ms_min=ts[0], ms_median=ts[len(ts) // 2], ms_max=ts[-1], n=n)


def build(w):
    mods = [bi.ShiftBounds()]
    for _ in range(w["n_couplings"] - 1):
        mods += [bi.NeuralSplineCoupling(knots=w["K"], layers=w["layers"]), bi.Roll(w["roll"])]
    mods.append(bi.NeuralSplineCoupling(knots=w["K"], layers=w["layers"]))
    flow = Flow(bi.Chain(mods))
    D, C, M = w["D"], w["C"], w["M"]
    g = torch.Generator(device="cuda").manual_seed(0)
    x = torch.rand(M, D, device="cuda", generator=g)
    c = torch.rand(M, C, device="cuda", generator=g) if C else None
    v = flow.init(0, x[:2].cpu().numpy(), None if c is None else c[:2].cpu().numpy())
    st = v["batch_stats"]["bijector"]["bijectors_0"]
    for i in range(D):
        st[f"xmin_{i}"] = np.array([-0.05], np.float32)
        st[f"xmax_{i}"] = np.array([1.05], np.float32)
    v = torch.utils._pytree.tree_map(lambda a: torch.from_numpy(np.asarray(a)).cuda(), v)

    def spec_of(self, x, c):
        spec = ChainSpec(D, C)
        self.bijector._emit(spec, self.scope.child("bijector"))
        return spec, self.latent._native()

    spec, (kind, peak) = flow.apply(v, x, c, method=spec_of)
    return spec, kind, peak, x, c


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--out", help="also write the JSON result to this file")
    args = ap.parse_args()
    out = dict(card=card(), workloads={})
    for name, w in WORKLOADS.items():
        spec, kind, peak, x, c = build(w)
        M = w["M"]
        ones = torch.ones(M, device="cuda")
        n = 5 if M > 4_000_000 else 10
        calls = {
            "log_prob": lambda: spec.log_prob(x, c, kind, peak),
            "vjp_inputs": lambda: spec.log_prob_vjp(x, c, kind, peak, ones, want_params=False),
            "vjp_params": lambda: spec.log_prob_vjp(x, c, kind, peak, ones),
        }
        res = dict(workload=w)
        for cname, fn in calls.items():
            t = timeit(fn, n)
            t["events_per_s"] = M / (t["ms_median"] * 1e-3)
            res[cname] = t
            print(f"{name} {cname}: {t}", file=sys.stderr, flush=True)
            torch.cuda.empty_cache()
        out["workloads"][name] = res
        del spec, x, c
        torch.cuda.empty_cache()
    print(json.dumps(out, indent=1))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
