"""Generate the golden fixtures under tests/golden/ by running the UNMODIFIED reference module.

Run in the build container only (``/root/reference`` does not exist on the GPU box):

    python oracle/make_golden.py

What it does
  * injects a stub for ``torch_geometric.nn.global_mean_pool`` (PyG is not installed; semantics:
    scatter-sum by graph id / count.clamp(min=1)) and imports ``models/FastEGNN.py`` as it lies;
  * for each case builds seeded inputs, constructs the reference ``FastEGNN`` under
    ``torch.manual_seed``, optionally scales the 1-wide coord heads ("trained-like"), runs its
    ``forward`` on CPU in fp32 (and fp64 for the tolerance basis) and stores inputs, state_dict and
    outputs (final + per-layer h/x/X/Hv captured with forward hooks) as a compressed ``.npz``;
  * for the 2-partition case it runs the reference's real ``world_size=2`` branch under
    ``torch.distributed`` + gloo in two spawned processes, with ``torch.Tensor.cuda`` patched to the
    identity (the reference hard-codes ``.cuda()`` at FastEGNN.py:196,226,260).

Test infrastructure; not imported by the product.
"""
from __future__ import annotations

import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
REF = "/root/reference"
OUT = os.path.join(ROOT, "tests", "golden")
INIT_SEED = 0                       # torch.manual_seed before the reference constructor
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
from tests.helpers import MAX_FIXTURE_BYTES, tensor_digest  # noqa: E402


def import_reference():
    def global_mean_pool(x, batch, size=None):
        n = int(batch.max().item()) + 1 if size is None else size
        tot = x.new_zeros((n, x.size(1)))
        tot.index_add_(0, batch, x)
        cnt = torch.bincount(batch, minlength=n).clamp(min=1).to(x.dtype)
        return tot / cnt.unsqueeze(-1)

    tg = types.ModuleType("torch_geometric")
    tgnn = types.ModuleType("torch_geometric.nn")
    tgnn.global_mean_pool = global_mean_pool
    tg.nn = tgnn
    sys.modules["torch_geometric"] = tg
    sys.modules["torch_geometric.nn"] = tgnn
    if REF not in sys.path:
        sys.path.insert(0, REF)
    from models.FastEGNN import FastEGNN  # noqa: E402  (the unmodified reference)
    return FastEGNN


def _rand_graph(rng, n, e, self_loops=True):
    row = rng.integers(0, n, size=e)
    col = rng.integers(0, n, size=e)
    if not self_loops:
        col = np.where(col == row, (col + 1) % n, col)
    return np.stack([row, col]).astype(np.int64)


def build_cases():
    """name -> (model kwargs, inputs dict of numpy arrays, coord head scale)."""
    sys.path.insert(0, ROOT)
    from distegnn_b200 import synth
    cases = {}

    # 1. N-body-like, fully connected, normalize=True (config/nbody_fastegnn.yaml), init weights
    w = synth.WORKLOADS["nbody100"]
    p = synth.make_partitions(w, n_nodes=24, seed=1)[0]
    cases["nbody24_norm"] = (dict(node_feat_nf=2, node_attr_nf=0, edge_attr_nf=2, virtual_channels=3,
                                  n_layers=4, normalize=True), p, 1.0)

    # 2. fluid-like radius graph, F=3, Na=2, C=5, trained-like coord heads
    w = synth.WORKLOADS["fluid113k"]
    p = synth.make_partitions(w, n_nodes=160, seed=2)[0]
    cases["fluid160_c5"] = (dict(node_feat_nf=3, node_attr_nf=2, edge_attr_nf=2, virtual_channels=5,
                                 n_layers=2, normalize=False), p, 100.0)

    # 3. batch of 3 graphs, C=8, random multigraph with self loops, duplicates and isolated nodes
    rng = np.random.default_rng(3)
    sizes = [17, 40, 9]
    n = sum(sizes)
    batch = np.repeat(np.arange(3), sizes)
    eis, off = [], 0
    for s in sizes:
        eis.append(_rand_graph(rng, s - 3, 4 * s) + off)        # last 3 nodes of each graph isolated
        off += s
    ei = np.concatenate(eis, axis=1)
    ei = ei[:, rng.permutation(ei.shape[1])]
    pos = rng.uniform(0, 3, size=(n, 3)).astype(np.float32)
    loc_mean = np.stack([pos[batch == b].mean(0) for b in range(3)]).astype(np.float32)
    p = dict(node_feat=torch.from_numpy(rng.normal(size=(n, 1)).astype(np.float32)),
             node_loc=torch.from_numpy(pos),
             node_vel=torch.from_numpy(rng.normal(size=(n, 3)).astype(np.float32)),
             loc_mean=torch.from_numpy(loc_mean), edge_index=torch.from_numpy(ei),
             data_batch=torch.from_numpy(batch.astype(np.int64)),
             edge_attr=torch.from_numpy(rng.uniform(0, 2, size=(ei.shape[1], 1)).astype(np.float32)),
             node_attr=None)
    cases["batch3_c8_multigraph"] = (dict(node_feat_nf=1, node_attr_nf=0, edge_attr_nf=1,
                                          virtual_channels=8, n_layers=2, normalize=False), p, 30.0)
    return cases


def _to_np(d):
    return {k: (v.numpy() if isinstance(v, torch.Tensor) else v) for k, v in d.items() if v is not None}


def run_reference(FastEGNN, kw, inp, scale, dtype, world_size=1):
    torch.manual_seed(INIT_SEED)
    model = FastEGNN(hidden_nf=64, world_size=world_size, **kw)
    sd = model.state_dict()
    for k in sd:
        if k.endswith("coord_mlp_r.2.weight") or k.endswith("coord_mlp_r_virtual.2.weight") \
                or k.endswith("coord_mlp_v_virtual.2.weight"):
            sd[k] = sd[k] * scale
    model.load_state_dict(sd)
    model = model.to(dtype)
    trace = {"h": [], "x": [], "Hv": [], "X": []}

    def hook(_m, _i, out):
        trace["h"].append(out[0].detach().clone())
        trace["x"].append(out[1].detach().clone())
        trace["Hv"].append(out[2].detach().clone())
        trace["X"].append(out[3].detach().clone())

    for i in range(kw["n_layers"]):
        getattr(model, f"gcl_{i}").register_forward_hook(hook)
    cast = lambda t: t.to(dtype) if (t is not None and t.is_floating_point()) else t
    with torch.no_grad():
        out, X = model(cast(inp["node_feat"]), cast(inp["node_loc"]), cast(inp["node_vel"]),
                       cast(inp["loc_mean"]), inp["edge_index"], inp["data_batch"],
                       cast(inp["edge_attr"]), cast(inp.get("node_attr")))
    return {k: v for k, v in model.state_dict().items()}, out, X, trace


def _rank_main(rank, world, port, kw, parts, scale, q):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.Tensor.cuda = lambda self, *a, **k: self          # reference hard-codes .cuda()
    FastEGNN = import_reference()
    sd, out, X, trace = run_reference(FastEGNN, kw, parts[rank], scale, torch.float32, world_size=world)
    q.put((rank, out.numpy(), X.numpy(), [t.numpy() for t in trace["h"]]))
    dist.barrier()
    dist.destroy_process_group()


def main():
    os.makedirs(OUT, exist_ok=True)
    FastEGNN = import_reference()
    for name, (kw, inp, scale) in build_cases().items():
        sd, out32, X32, tr = run_reference(FastEGNN, kw, inp, scale, torch.float32)
        _, out64, X64, _ = run_reference(FastEGNN, kw, inp, scale, torch.float64)
        blob = {"in." + k: v for k, v in _to_np(inp).items()}
        blob.update({"sd." + k: v.numpy() for k, v in sd.items()})
        blob.update({"out.node_loc": out32.numpy(), "out.virtual_loc": X32.numpy(),
                     "out64.node_loc": out64.numpy(), "out64.virtual_loc": X64.numpy()})
        for key in ("h", "x", "Hv", "X"):
            for i, t in enumerate(tr[key]):
                blob[f"trace.{key}.{i}"] = t.numpy()
        blob["meta.kw"] = np.array(repr(kw))
        path = os.path.join(OUT, name + ".npz")
        np.savez_compressed(path, **blob)
        if os.path.getsize(path) > MAX_FIXTURE_BYTES:
            # untouched init too large to store: keep its seed and a digest per tensor instead; tests.helpers.load_golden
            # regenerates the weights and checks them against the digests
            assert scale == 1.0, name
            blob = {k: v for k, v in blob.items() if not k.startswith("sd.")}
            blob["meta.seed"] = np.array(INIT_SEED)
            blob.update({"sdsha." + k: np.array(tensor_digest(v)) for k, v in sd.items()})
            np.savez_compressed(path, **blob)
        print(name, "N", inp["node_feat"].shape[0], "E", inp["edge_index"].shape[1],
              "max|out32-out64|", float((out32.double() - out64).abs().max()))

    # 2-partition DistEGNN through the reference's own world_size=2 branch (gloo)
    import torch.multiprocessing as mp
    sys.path.insert(0, ROOT)
    from distegnn_b200 import synth
    w = synth.WORKLOADS["fluid113k"]
    parts = synth.make_partitions(w, world_size=2, split_mode="random", n_nodes=300, seed=5)
    kw = dict(node_feat_nf=3, node_attr_nf=2, edge_attr_nf=2, virtual_channels=5, n_layers=2,
              normalize=False)
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_rank_main, args=(r, 2, 29611, kw, parts, 100.0, q)) for r in range(2)]
    [p.start() for p in procs]
    res = sorted([q.get() for _ in procs], key=lambda t: t[0])
    [p.join() for p in procs]
    torch.manual_seed(0)
    sd, _, _, _ = run_reference(FastEGNN, kw, parts[0], 100.0, torch.float32)   # same seed ⇒ same weights
    blob = {"sd." + k: v.numpy() for k, v in sd.items()}
    for r, p in enumerate(parts):
        blob.update({f"in{r}." + k: v for k, v in _to_np(p).items()})
        blob[f"out{r}.node_loc"] = res[r][1]
        blob[f"out{r}.virtual_loc"] = res[r][2]
        for i, h in enumerate(res[r][3]):
            blob[f"trace{r}.h.{i}"] = h
    blob["meta.kw"] = np.array(repr(kw))
    np.savez_compressed(os.path.join(OUT, "dist2_fluid300_c5.npz"), **blob)
    print("dist2_fluid300_c5", [p["node_feat"].shape[0] for p in parts],
          [p["edge_index"].shape[1] for p in parts],
          "virtual_loc rank diff", float(np.abs(res[0][2] - res[1][2]).max()))


if __name__ == "__main__":
    main()
