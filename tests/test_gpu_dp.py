"""GPU parity of the data-parallel train step (SURVEY.md 8e): ``TrainEngine`` at world 2 on row shards
reproduces the world-1 loss, flat gradient, updated parameters and running statistics of the same global batch.

Two transports are covered:
  * gloo between two processes that SHARE one GPU (runs on a single-GPU box): the phases are sequenced from the
    host with torch.distributed all-reduces in between (``TrainEngine._step_phased``);
  * NCCL through the C ABI (zf_dp_*, one process per GPU; needs two GPUs): ``zf_flow_value_and_grad`` with the
    statistics all-reduced on the compute stream and the gradient buckets on the side stream.
Also: ``train()`` with shards that disagree on the number of steps raises on every rank instead of hanging.
"""
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

pytestmark = pytest.mark.gpu

D, C, K, LAYERS, NCOUP, ROLL, M = 6, 2, 16, (128, 128), 3, 2, 2048


def _problem():
    from oracle import zenflow_oracle as zo

    rng = np.random.default_rng(11)
    ops = zo.make_chain(D, K, LAYERS, n_couplings=NCOUP, roll_shift=ROLL)
    x = rng.normal(0.3, 1.0, (M, D)).astype(np.float32)
    c = rng.uniform(0, 1, (M, C)).astype(np.float32)
    v = zo.init_variables(ops, D, C, 2, weight_scale=1.2, randomize_bn=True)
    return ops, v, x, c


def _engine(ops, v, **kw):
    from tests.helpers import product_chain
    from zenflow_b200 import Flow
    from zenflow_b200._train import TrainEngine

    flow = Flow(product_chain(ops))
    flow.latent._latch_dim(D)
    fv = {"params": {"bijector": v["params"]}, "batch_stats": {"bijector": v["batch_stats"]}}
    return TrainEngine(flow, fv, D, C, micro_batch=512, **kw)


def _flat_stats(eng):
    out = []
    for g in eng.groups:
        if g["kind"] == "cp":
            out += [g["ra_mean"].double().cpu(), g["ra_var"].double().cpu()]
        else:
            out += [g["xmin"].double().cpu(), g["xmax"].double().cpu()]
    return torch.cat(out).numpy()


def _worker(rank, world, port, backend, devices, out):
    sys.path.insert(0, ROOT)
    import torch.distributed as dist

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(devices[rank])
    dist.init_process_group(backend, rank=rank, world_size=world,
                            **({"device_id": torch.device("cuda", devices[rank])} if backend == "nccl" else {}))
    try:
        ops, v, x, c = _problem()
        lo, hi = rank * M // world, (rank + 1) * M // world
        eng = _engine(ops, v)
        assert eng.world == world and eng.use_nccl == (backend == "nccl")
        res = {}
        for it in range(2):   # two full optimiser steps: gradients, parameters and running statistics all agree
            lp_sum = eng.step(x[lo:hi], c[lo:hi], global_count=M)
            t = lp_sum.clone()
            dist.all_reduce(t)
            res[f"loss{it}"] = -float(t.item()) / M
            res[f"G{it}"] = eng.G.double().cpu().numpy()
            res[f"P{it}"] = eng.P.double().cpu().numpy()
            res[f"S{it}"] = _flat_stats(eng)
        # train(): shards that disagree on the number of minibatch steps must raise on every rank, not hang
        from zenflow_b200 import Flow, train
        from zenflow_b200.bijectors import rolling_spline_coupling

        n_local = 700 if rank == 0 else 300
        X = np.random.default_rng(rank).normal(size=(n_local, 2)).astype(np.float32)
        try:
            train(Flow(rolling_spline_coupling(2)), X, X[:100], epochs=1, batch_size=256, progress=False)
            res["raised"] = False
        except ValueError as e:
            res["raised"] = "disagree" in str(e)
        # equal shards: every rank returns the same histories (global losses) and the same best epoch
        X = np.random.default_rng(5).normal(size=(1024, 2)).astype(np.float32)
        best, be, ltr, lte = train(Flow(rolling_spline_coupling(2)), X[rank * 512:(rank + 1) * 512],
                                   X[rank * 100:(rank + 1) * 100 + 50 * rank], epochs=3, batch_size=128, patience=1,
                                   progress=False)
        res["hist"] = (be, ltr, lte)
        out.put((rank, res))
    finally:
        dist.destroy_process_group()


def _run(backend, devices):
    import torch.multiprocessing as mp

    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    port = 29600 + (os.getpid() % 1500)
    procs = [ctx.Process(target=_worker, args=(r, 2, port, backend, devices, out)) for r in range(2)]
    for p in procs:
        p.start()
    got = {}
    for _ in procs:
        r, res = out.get(timeout=600)
        got[r] = res
    for p in procs:
        p.join(120)
        assert p.exitcode == 0
    # the world-1 reference on the whole batch, in this process
    ops, v, x, c = _problem()
    eng = _engine(ops, v)
    for it in range(2):
        lp_sum = eng.step(x, c)
        loss = -float(lp_sum.item()) / M
        G, P, S = eng.G.double().cpu().numpy(), eng.P.double().cpu().numpy(), _flat_stats(eng)
        for r in (0, 1):
            res = got[r]
            assert abs(res[f"loss{it}"] - loss) <= 1e-6 * abs(loss), (it, r, res[f"loss{it}"], loss)
            eg = np.abs(res[f"G{it}"] - G).max() / np.abs(G).max()
            # step 0: identical parameters on both sides, only the summation order of the all-reduced sums differs.
            # step 1 starts from parameters that already differ by the amplified last bits noted below (up to 2e-5
            # of the largest weight), so its gradient can only be expected to agree to a few 1e-6.
            assert eg <= (1e-6 if it == 0 else 5e-6), f"step {it} rank {r}: flat gradient differs by {eg:.2e} of its largest entry"
            np.testing.assert_allclose(res[f"S{it}"], S, rtol=1e-6, atol=1e-7)
            # NAdamW divides by sqrt(nu): entries with tiny gradients amplify the last-bit differences
            assert np.abs(res[f"P{it}"] - P).max() <= 2e-5 * np.abs(P).max()
        print(f"\n{backend} step {it}: loss {loss:.8f}, world-2 flat gradient within {eg:.2e} of world 1")
    assert got[0]["raised"] and got[1]["raised"]
    assert got[0]["hist"] == got[1]["hist"]
    assert np.isfinite(got[0]["hist"][1]).all()


def test_dp_world2_shared_gpu_gloo_matches_single_device():
    _run("gloo", [0, 0])


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_dp_world2_nccl_c_abi_matches_single_device():
    _run("nccl", [0, 1])


def test_value_and_grad_forward_only_matches_full_call():
    """grads = NULL (the fwd rule of the jax custom_vjp, ffi/zenflow_jax.py): same lp sum and the same statistics
    updates as the full call, gradient buffer untouched."""
    import ctypes as Ct

    from zenflow_b200 import _lib
    from zenflow_b200._device import ptr, stream_ptr

    ops, v, x, c = _problem()
    full = _engine(ops, v)
    full.step(x, c, update=False)
    ref_lp, ref_stats = float(full.lp_sum.item()), _flat_stats(full)

    eng = _engine(ops, v)
    lib = _lib.load()
    xd = torch.as_tensor(x, device="cuda")
    cd = torch.as_tensor(c, device="cuda")
    ws = eng._workspace(M)
    base = (ws.data_ptr() + 255) & ~255
    eng.G.fill_(7.0)
    lp = torch.empty(M, dtype=torch.float32, device="cuda")
    kind, peak = eng.flow.latent._native()
    _lib.check(lib.zf_flow_value_and_grad(stream_ptr(), None, Ct.byref(eng.chain), None, kind, peak, ptr(xd), ptr(cd), M, float(M),
                                          None, ptr(lp), ptr(eng.lp_sum), None, None, None, None, eng._bucket_off, base,
                                          ws.numel() - (base - ws.data_ptr()), eng.micro_batch), "zf_flow_value_and_grad")
    torch.cuda.synchronize()
    assert float(eng.lp_sum.item()) == ref_lp
    np.testing.assert_array_equal(_flat_stats(eng), ref_stats)
    assert bool((eng.G == 7.0).all())
    np.testing.assert_allclose(lp.double().sum().item(), ref_lp, rtol=1e-6)
