"""Throughput of the inverse chain, sampling and their VJP (zf_chain_inverse_vjp) on the bench workloads.

For bounded16 (configs[3]: 16-D, ShiftBounds + 8 couplings, K = 32, 16M events) and two_moons_conditional (configs[1]:
2-D conditional, 1M events) it times four calls with CUDA events, each warmed up and repeated:
  inverse       zf_chain_inverse (Flow.inverse)
  sample        zf_flow_sample (Flow.sample)
  vjp_inputs    zf_chain_inverse_vjp with grads = NULL: d/dz and d/dc only
  vjp_params    zf_chain_inverse_vjp with the parameter gradients as well
The flows, inputs and timing are those of scripts/eval_grad_perf.py.  The card's name and power limit are read in the
same run and stored beside the numbers.  Output: JSON on stdout (and in --out FILE); progress on stderr.
"""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import torch  # noqa: E402

from eval_grad_perf import WORKLOADS, build, card, timeit  # noqa: E402


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--out", help="also write the JSON result to this file")
    args = ap.parse_args()
    out = dict(card=card(), workloads={})
    for name, w in WORKLOADS.items():
        spec, kind, peak, z, c = build(w)   # z: uniform draws in [0, 1)
        M = w["M"]
        ct = torch.ones_like(z)
        n = 5 if M > 4_000_000 else 10
        calls = {
            "inverse": lambda: spec.inverse(z, c),
            "sample": lambda: spec.sample(M, c, kind, peak, 0),
            "vjp_inputs": lambda: spec.inverse_vjp(z, c, ct, want_params=False),
            "vjp_params": lambda: spec.inverse_vjp(z, c, ct),
        }
        res = dict(workload=w)
        for cname, fn in calls.items():
            t = timeit(fn, n)
            t["events_per_s"] = M / (t["ms_median"] * 1e-3)
            res[cname] = t
            print(f"{name} {cname}: {t}", file=sys.stderr, flush=True)
            torch.cuda.empty_cache()
        out["workloads"][name] = res
        del spec, z, c, ct
        torch.cuda.empty_cache()
    print(json.dumps(out, indent=1))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
