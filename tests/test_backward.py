"""Backward pass (SURVEY §8 f-1) on CPU: (1) the oracle's autograd is pinned to gradient fixtures produced by the
unmodified reference under autograd (oracle/make_golden_grads.py); (2) the product's host-side backward orchestration
(FastEGNN._forward_autograd / _FastEGNNFunction: per-layer chain, packed gradient all-reduce, dense stages, parameter
unpacking) reproduces those gradients with the kernels replaced by the torch stand-in; (3) the same under gloo with
world_size=2 against the reference's own 2-rank backward."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

from oracle import fastegnn_oracle as orc
from tests.helpers import DIST_CASE, GOLDEN, SINGLE_CASES, golden_inputs, grad_sample, load_golden


def load_grads(name):
    return np.load(os.path.join(GOLDEN, name + ".grads.npz"))


def rel_err(mine, ref):
    ref = ref.double()
    return float((mine.double() - ref).abs().max() / ref.abs().max().clamp(min=1e-30))


def check_against(named_grads, zg, prefix, tol, dead):
    """Every parameter gradient within `tol` (max-norm relative); parameters the reference leaves without a
    gradient (dead last-layer h / Hv branches, FastEGNN.py:307) must be exactly zero here."""
    worst = ("", 0.0)
    for k, g in named_grads.items():
        ref = torch.from_numpy(zg[prefix + k])
        idx = grad_sample(zg, prefix + k)
        if idx is not None:
            g = g.reshape(-1)[idx]
        if float(ref.abs().max()) == 0.0:
            assert g is None or float(g.abs().max()) == 0.0, k
            dead.append(k)
            continue
        e = rel_err(g, ref)
        if e > worst[1]:
            worst = (k, e)
        assert e <= tol, (k, e)
    return worst


@pytest.mark.parametrize("name", SINGLE_CASES)
def test_oracle_autograd_matches_reference_gradients(name):
    z, kw, sd = load_golden(name)
    zg = load_grads(name)
    inp = golden_inputs(z)
    sd64 = {k: v.double().requires_grad_(True) for k, v in sd.items()}
    inp64 = {k: (v.double() if (v is not None and v.is_floating_point()) else v) for k, v in inp.items()}
    out, X = orc.forward(sd64, **inp64, normalize=kw["normalize"])
    loss = (out * torch.from_numpy(zg["cot.out"])).sum() + (X * torch.from_numpy(zg["cot.X"])).sum()
    assert abs(float(loss) - float(zg["loss"])) <= 1e-10 * max(1.0, abs(float(zg["loss"])))
    keys = [k for k in sd64 if sd64[k].requires_grad]
    grads = torch.autograd.grad(loss, [sd64[k] for k in keys], allow_unused=True)
    dead = []
    worst = check_against({k: (g if g is not None else torch.zeros_like(sd64[k])) for k, g in zip(keys, grads)}, zg,
                          "grad.", 1e-9, dead)
    print(name, "worst", worst, "dead parameters", len(dead))


@pytest.mark.parametrize("name", SINGLE_CASES)
def test_training_path_gradients_match_reference(name):
    from distegnn_b200 import FastEGNN
    from tests.shadow_backend import ShadowBackend
    z, kw, sd = load_golden(name)
    zg = load_grads(name)
    inp = golden_inputs(z)
    m = FastEGNN(hidden_nf=64, world_size=1, **kw)
    m.load_state_dict(sd)
    m._backend = ShadowBackend()
    out, X = m(**inp)
    assert out.requires_grad and X.requires_grad
    loss = (out * torch.from_numpy(zg["cot.out"]).float()).sum() + (X * torch.from_numpy(zg["cot.X"]).float()).sum()
    loss.backward()
    dead = []
    # fp32 against the reference's fp64 gradients; the reference's own fp32 run differs from its fp64 run by up to
    # 3e-5 on these cases (oracle/make_golden_grads.py output)
    worst = check_against({k: (p.grad if p.grad is not None else torch.zeros_like(p)) for k, p in m.named_parameters()},
                          zg, "grad.", 2e-4, dead)
    print(name, "worst", worst, "dead parameters", len(dead))


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _rank(rank, world, port, q):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from distegnn_b200 import FastEGNN
        from tests.shadow_backend import ShadowBackend
        z, kw, sd = load_golden(DIST_CASE)
        zg = load_grads(DIST_CASE)
        inp = golden_inputs(z, f"in{rank}.")
        m = FastEGNN(hidden_nf=64, world_size=world, **kw)
        m.load_state_dict(sd)
        m._backend = ShadowBackend()
        calls = []
        orig = dist.all_reduce

        def counting(t, *a, **k):
            calls.append(tuple(t.shape))
            return orig(t, *a, **k)

        dist.all_reduce = counting
        out, X = m(**inp)
        n_fwd = len(calls)
        loss = (out * torch.from_numpy(zg[f"cot{rank}.out"])).sum() + (X * torch.from_numpy(zg["cot.X"])).sum()
        loss.backward()
        dist.all_reduce = orig
        grads = {k: (p.grad if p.grad is not None else torch.zeros_like(p)).numpy() for k, p in m.named_parameters()}
        q.put((rank, grads, float(loss), n_fwd, len(calls) - n_fwd))
        dist.barrier()
    finally:
        dist.destroy_process_group()


def test_two_partition_gradients_match_reference_world_size_2():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_rank, args=(r, 2, port, q)) for r in range(2)]
    [p.start() for p in procs]
    res = sorted([q.get(timeout=180) for _ in procs], key=lambda t: t[0])
    [p.join(timeout=60) for p in procs]
    z, kw, sd = load_golden(DIST_CASE)
    zg = load_grads(DIST_CASE)
    L = kw["n_layers"]
    for r in range(2):
        assert abs(res[r][2] - float(zg[f"loss{r}"])) <= 1e-4 * max(1.0, abs(float(zg[f"loss{r}"])))
        dead = []
        worst = check_against({k: torch.from_numpy(v) for k, v in res[r][1].items()}, zg, f"grad{r}.", 5e-4, dead)
        print("rank", r, "worst", worst, "dead", len(dead))
        # protocol: L+1 packed collectives forward, L packed collectives backward (the reference: 6 per layer each way)
        assert res[r][3] == L + 1 and res[r][4] == L


def test_inference_path_is_taken_without_grad():
    """no_grad / frozen parameters -> the light inference path (no autograd node, nothing kept)."""
    from distegnn_b200 import FastEGNN
    from tests.shadow_backend import ShadowBackend
    z, kw, sd = load_golden("fluid160_c5")
    inp = golden_inputs(z)
    m = FastEGNN(hidden_nf=64, world_size=1, **kw)
    m.load_state_dict(sd)
    m._backend = ShadowBackend()
    with torch.no_grad():
        out, X = m(**inp)
    assert not out.requires_grad and not X.requires_grad
    for p in m.parameters():
        p.requires_grad_(False)
    out2, X2 = m(**inp)
    assert not out2.requires_grad and out2.grad_fn is None
    assert torch.equal(out, out2) and torch.equal(X, X2)
    for p in m.parameters():
        p.requires_grad_(True)
    out3, X3 = m(**inp)                                   # training path: same numbers, attached to autograd
    assert out3.requires_grad and out3.grad_fn is not None
    assert float((out3 - out).abs().max()) <= 1e-6 and float((X3 - X).abs().max()) <= 1e-6


def test_gradient_accumulation_and_optimizer_step():
    """Two backward calls accumulate (utils/train.py:149-158 accumulates 4 micro-steps); Adam + clip_grad_norm_ run on the
    module's own nn.Parameters and change the next forward."""
    from distegnn_b200 import FastEGNN
    from tests.shadow_backend import ShadowBackend
    z, kw, sd = load_golden("fluid160_c5")
    zg = load_grads("fluid160_c5")
    inp = golden_inputs(z)
    m = FastEGNN(hidden_nf=64, world_size=1, **kw)
    m.load_state_dict(sd)
    m._backend = ShadowBackend()
    cot, cotX = torch.from_numpy(zg["cot.out"]).float(), torch.from_numpy(zg["cot.X"]).float()
    for _ in range(2):
        out, X = m(**inp)
        ((out * cot).sum() + (X * cotX).sum()).backward()
    for k, p in m.named_parameters():
        ref = 2 * torch.from_numpy(zg["grad." + k])
        if float(ref.abs().max()) > 0:
            assert rel_err(p.grad, ref) <= 2e-4, k
    out_before = m(**inp)[0].detach().clone()
    opt = torch.optim.Adam(m.parameters(), lr=1e-3)
    torch.nn.utils.clip_grad_norm_(m.parameters(), 0.3)
    opt.step()
    out_after = m(**inp)[0].detach()
    assert float((out_after - out_before).abs().max()) > 0


def _ddp_rank(rank, world, port, q):
    import torch.distributed as dist
    from torch.nn.parallel import DistributedDataParallel
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from distegnn_b200 import FastEGNN
        from tests.shadow_backend import ShadowBackend
        z, kw, sd = load_golden(DIST_CASE)
        zg = load_grads(DIST_CASE)
        inp = golden_inputs(z, f"in{rank}.")
        m = FastEGNN(hidden_nf=64, world_size=world, **kw)
        m.load_state_dict(sd)
        m._backend = ShadowBackend()
        ddp = DistributedDataParallel(m, find_unused_parameters=True)      # reference main.py:196
        node_attr = inp["node_attr"] if kw["node_attr_nf"] > 0 else None
        out, X = ddp(inp["node_feat"], inp["node_loc"], inp["node_vel"], inp["loc_mean"], inp["edge_index"],
                     inp["data_batch"], inp["edge_attr"], node_attr)        # positional, as utils/train.py:63-71
        ((out * torch.from_numpy(zg[f"cot{rank}.out"])).sum() + (X * torch.from_numpy(zg["cot.X"])).sum()).backward()
        q.put((rank, {k: p.grad.numpy() for k, p in m.named_parameters() if p.grad is not None}))
        dist.barrier()
    finally:
        dist.destroy_process_group()


def test_ddp_wrapper_averages_the_reference_rank_gradients():
    """DistributedDataParallel(find_unused_parameters=True) around the module, as the reference wraps it: after backward
    every rank holds the MEAN over ranks of the per-rank gradients — here the mean of the reference's own rank gradients."""
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_ddp_rank, args=(r, 2, port, q)) for r in range(2)]
    [p.start() for p in procs]
    res = sorted([q.get(timeout=180) for _ in procs], key=lambda t: t[0])
    [p.join(timeout=60) for p in procs]
    zg = load_grads(DIST_CASE)
    for k, g0 in res[0][1].items():
        ref = 0.5 * (torch.from_numpy(zg["grad0." + k]).double() + torch.from_numpy(zg["grad1." + k]).double())
        assert np.array_equal(g0, res[1][1][k]), k                       # identical on both ranks
        if float(ref.abs().max()) > 0:
            assert rel_err(torch.from_numpy(g0), ref) <= 5e-4, k
