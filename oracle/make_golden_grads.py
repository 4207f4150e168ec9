"""Generate GRADIENT fixtures (tests/golden/*.grads.npz) by running the UNMODIFIED reference module under autograd.

Run in the build container only (``/root/reference`` does not exist on the GPU box):

    python oracle/make_golden_grads.py

For every case of oracle/make_golden.py (same seeded inputs, same weights, read back from the committed forward
fixtures so that both stay consistent) the reference ``FastEGNN`` is run on CPU in float64 with gradients enabled and
the scalar  L = <node_loc_out, cot_out> + <virtual_loc_out, cot_X>  (seeded random cotangents, stored in the fixture)
is back-propagated: the fixture holds d L / d parameter for every parameter of the reference's state_dict.
For the 2-partition case the reference's real ``world_size=2`` branch runs under gloo (``torch.Tensor.cuda`` patched to
the identity, float32): each rank back-propagates  L_r = <node_loc_out_r, cot_out_r> + <virtual_loc_out, cot_X>  through
the reference's differentiable all-reduce (``_AllReduce``, FastEGNN.py:10-43) and stores ITS parameter gradients.

Test infrastructure; not imported by the product.
"""
from __future__ import annotations

import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)
from make_golden import OUT, import_reference  # noqa: E402
from tests.helpers import DIST_CASE, MAX_FIXTURE_BYTES, SINGLE_CASES, golden_inputs, load_golden  # noqa: E402

GRAD_SAMPLE = 1536      # entries kept of each large gradient when the whole fixture would exceed MAX_FIXTURE_BYTES


def cotangents(seed, n, B, C, dtype):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(n, 3, generator=g, dtype=torch.float64).to(dtype), \
        torch.randn(B, 3, C, generator=g, dtype=torch.float64).to(dtype)


def sample_large_grads(blob, seed=0):
    """Each nonzero gradient of more than GRAD_SAMPLE entries -> a seeded sample of its flat entries ("grad.<k>") that
    includes the entry of largest magnitude, plus their sorted flat indices ("idx.grad.<k>"; tests.helpers.grad_sample).
    All-zero gradients stay whole: they compress to nothing and the tests check them entry by entry."""
    rng = np.random.default_rng(seed)
    out = {}
    for k, v in blob.items():
        flat = v.reshape(-1)
        if k.startswith("grad.") and flat.size > GRAD_SAMPLE and np.abs(flat).max() > 0:
            idx = np.unique(np.append(rng.choice(flat.size, GRAD_SAMPLE - 1, replace=False), np.abs(flat).argmax()))
            out["idx." + k] = idx.astype(np.int32)
            out[k] = flat[idx]
        else:
            out[k] = v
    return out


def reference_grads(FastEGNN, kw, sd, inp, cot_out, cot_X, dtype, world_size=1):
    model = FastEGNN(hidden_nf=64, world_size=world_size, **kw)
    model.load_state_dict(sd)
    model = model.to(dtype)
    cast = lambda t: t.to(dtype) if (t is not None and t.is_floating_point()) else t
    out, X = model(cast(inp["node_feat"]), cast(inp["node_loc"]), cast(inp["node_vel"]), cast(inp["loc_mean"]),
                   inp["edge_index"], inp["data_batch"], cast(inp["edge_attr"]), cast(inp.get("node_attr")))
    loss = (out * cot_out).sum() + (X * cot_X).sum()
    loss.backward()
    return {k: (p.grad if p.grad is not None else torch.zeros_like(p)).detach().clone()
            for k, p in model.named_parameters()}, float(loss)


def _rank_main(rank, world, port, kw, sd, parts, q):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.Tensor.cuda = lambda self, *a, **k: self          # reference hard-codes .cuda()
    FastEGNN = import_reference()
    n, B, C = parts[rank]["node_loc"].shape[0], parts[rank]["loc_mean"].shape[0], kw["virtual_channels"]
    cot_out, _ = cotangents(100 + rank, n, B, C, torch.float32)
    _, cot_X = cotangents(99, n, B, C, torch.float32)       # the virtual output is identical on every rank
    grads, loss = reference_grads(FastEGNN, kw, sd, parts[rank], cot_out, cot_X, torch.float32, world_size=world)
    q.put((rank, {k: v.numpy() for k, v in grads.items()}, cot_out.numpy(), cot_X.numpy(), loss))
    dist.barrier()
    dist.destroy_process_group()


def main():
    FastEGNN = import_reference()
    for name in SINGLE_CASES:
        z, kw, sd = load_golden(name)
        inp = golden_inputs(z)
        n, B, C = inp["node_loc"].shape[0], inp["loc_mean"].shape[0], kw["virtual_channels"]
        cot_out, cot_X = cotangents(7, n, B, C, torch.float64)
        grads, loss = reference_grads(FastEGNN, kw, sd, inp, cot_out, cot_X, torch.float64)
        g32, _ = reference_grads(FastEGNN, kw, sd, inp, cot_out.float(), cot_X.float(), torch.float32)
        blob = {"grad." + k: v.numpy() for k, v in grads.items()}
        blob.update({"cot.out": cot_out.numpy(), "cot.X": cot_X.numpy(), "loss": np.array(loss)})
        path = os.path.join(OUT, name + ".grads.npz")
        np.savez_compressed(path, **blob)
        if os.path.getsize(path) > MAX_FIXTURE_BYTES:
            np.savez_compressed(path, **sample_large_grads(blob))
        worst = max(float((g32[k].double() - grads[k]).abs().max() / grads[k].abs().max().clamp(min=1e-30)) for k in grads)
        print(name, "loss", loss, "params", len(grads), "max rel |grad32 - grad64| over parameters", worst)

    import torch.multiprocessing as mp
    z, kw, sd = load_golden(DIST_CASE)
    parts = [golden_inputs(z, f"in{r}.") for r in range(2)]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_rank_main, args=(r, 2, 29613, kw, sd, parts, q)) for r in range(2)]
    [p.start() for p in procs]
    res = sorted([q.get() for _ in procs], key=lambda t: t[0])
    [p.join() for p in procs]
    blob = {}
    for r, grads, cot_out, cot_X, loss in res:
        blob.update({f"grad{r}." + k: v for k, v in grads.items()})
        blob[f"cot{r}.out"] = cot_out
        blob["cot.X"] = cot_X
        blob[f"loss{r}"] = np.array(loss)
    np.savez_compressed(os.path.join(OUT, DIST_CASE + ".grads.npz"), **blob)
    print(DIST_CASE, "losses", [r[4] for r in res])


if __name__ == "__main__":
    main()
