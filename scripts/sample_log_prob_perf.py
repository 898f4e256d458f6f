"""Throughput of sampling with the log-density in one fused pass (zf_flow_sample_log_prob) and of its VJP on the bench
workloads.

For bounded16 (configs[3]: 16-D, ShiftBounds + 8 couplings, K = 32, 16M events) and two_moons_conditional (configs[1]:
2-D conditional, 1M events) it times, with CUDA events, each warmed up and repeated:
  sample              zf_flow_sample (Flow.sample)
  sample_then_lp      zf_flow_sample followed by zf_flow_log_prob on the samples (the two-call composition)
  sample_and_lp       zf_flow_sample_log_prob (Flow.sample_and_log_prob)
  vjp_inputs          zf_flow_sample_log_prob_vjp for g_x = 1 and g_lp = 1 with grads = NULL (d/dc only; drawn latent)
  vjp_params          the same with the parameter gradients
  inverse_vjp_params  zf_chain_inverse_vjp with the parameter gradients (drawn latent), for reference
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
        spec, kind, peak, z, c = build(w)
        M, D = w["M"], w["D"]
        del z
        ones_x = torch.ones(M, D, device="cuda")
        ones_lp = torch.ones(M, device="cuda")
        n = 5 if M > 4_000_000 else 10
        draw = dict(draw_seed=0, n=M)
        calls = {
            "sample": lambda: spec.sample(M, c, kind, peak, 0),
            "sample_then_lp": lambda: spec.log_prob(spec.sample(M, c, kind, peak, 0), c, kind, peak),
            "sample_and_lp": lambda: spec.sample_log_prob(None, c, kind, peak, **draw),
            "vjp_inputs": lambda: spec.sample_log_prob_vjp(None, c, kind, peak, ones_x, ones_lp, want_params=False, **draw),
            "vjp_params": lambda: spec.sample_log_prob_vjp(None, c, kind, peak, ones_x, ones_lp, **draw),
            "inverse_vjp_params": lambda: spec.inverse_vjp(None, c, ones_x, draw=(M, kind, peak, 0)),
        }
        res = dict(workload=w)
        for cname, fn in calls.items():
            t = timeit(fn, n)
            t["events_per_s"] = M / (t["ms_median"] * 1e-3)
            res[cname] = t
            print(f"{name} {cname}: {t}", file=sys.stderr, flush=True)
            torch.cuda.empty_cache()
        out["workloads"][name] = res
        del spec, c, ones_x, ones_lp
        torch.cuda.empty_cache()
    print(json.dumps(out, indent=1))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
