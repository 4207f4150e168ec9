"""GPU parity tests (run on the B200 box): the CUDA path through the C ABI against
  * the reference-generated golden fixtures,
  * the oracle on seeded inputs,
  * each kernel's torch restatement (tests/shadow_backend.py) in isolation,
  * size-independent properties at larger sizes (SE(3) equivariance, edge-order invariance,
    partition/block-diagonal equivalence).
Tolerances (fp32 path; SURVEY §8c): |out − ref64| ≤ 1e-5·max(1,|out|), relative displacement error
≤ 1e-4, equivariance residual ≤ 1e-4 (the reference's own gate, equivariant_test.py:62).
"""
import os

import numpy as np
import pytest
import torch

from distegnn_b200 import FastEGNN, _lib, synth
from oracle import fastegnn_oracle as orc
from tests.helpers import SINGLE_CASES, golden_inputs, golden_trace, grad_sample, load_golden, max_abs, rel_disp_err
from tests.shadow_backend import ShadowBackend

pytestmark = pytest.mark.gpu

ABS_TOL = 1e-5
REL_DISP_TOL = 1e-4


def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device (no fallback)"
    return torch.device("cuda:0")


def to_dev(inp):
    return {k: (v.to(dev()) if v is not None else None) for k, v in inp.items()}


def cuda_model(kw, sd, world_size=1):
    m = FastEGNN(hidden_nf=64, world_size=world_size, **kw)
    m.load_state_dict(sd)
    return m.to(dev()).eval()


def oracle64(sd, inp, normalize):
    sd64 = {k: v.double() for k, v in sd.items()}
    i64 = {k: (v.double() if (v is not None and v.is_floating_point()) else v) for k, v in inp.items()}
    return orc.forward(sd64, **i64, normalize=normalize)


def check_close(out, X, ref, refX, pos, what=""):
    out, X = out.cpu(), X.cpu()
    e_abs, scale = max_abs(out, ref), max(1.0, float(ref.abs().max()))
    e_rel = rel_disp_err(out, ref, pos)
    e_X = max_abs(X, refX)
    msg = f"{what}: abs {e_abs:.3e} (scale {scale:.2f}) rel-disp {e_rel:.3e} virtual {e_X:.3e}"
    print(msg)
    assert e_abs <= ABS_TOL * scale, msg
    assert e_rel <= REL_DISP_TOL, msg
    assert e_X <= ABS_TOL * max(1.0, float(refX.abs().max())), msg


def test_library_loaded_and_abi():
    lib = _lib.load()
    assert lib.distegnn_abi_version() == 2


def test_tcgen05_building_block():
    """D = A·Wᵀ on the tensor cores with the 3xTF32 split must be fp32-accurate (and plain TF32 must not
    be — that is why the split exists)."""
    from tests.twin_backend import load_testing
    lib = load_testing()
    g = torch.Generator().manual_seed(0)
    A = torch.randn(128, 64, generator=g).to(dev())
    W = (torch.randn(64, 64, generator=g) / 8).to(dev())
    ref = A.double() @ W.double().t()
    errs = {}
    for variant in (0, 2, 4):
        D = torch.zeros(128, 64, device=dev())
        rc = lib.distegnn_selftest_umma(A.data_ptr(), W.data_ptr(), D.data_ptr(), variant,
                                        torch.cuda.current_stream().cuda_stream)
        assert rc == 0
        torch.cuda.synchronize()
        errs[variant] = max_abs(D, ref)
    print("tcgen05 selftest errs", errs)
    assert errs[0] <= 1e-5 and errs[2] <= 1e-5      # 3xTF32, A in TMEM / in shared memory
    assert errs[4] > 1e-4                           # single-pass TF32 is not fp32-accurate


def test_edge_kernel_tensor_core_vs_fma_twin():
    """The tcgen05 edge kernel against its independent fp32-FMA implementation on a 300k-node graph
    (both normalisation modes, with and without the Σm output)."""
    from tests.twin_backend import twin_backend
    be = twin_backend()
    w = synth.WORKLOADS["synth1m"]
    inp = to_dev(synth.make_partitions(w, n_nodes=300_000, seed=7)[0])
    sd = orc.init_state_dict(3, 2, 2, 64, 8, 1, seed=2, coord_gain=1.0)
    m = cuda_model(dict(node_feat_nf=3, node_attr_nf=2, edge_attr_nf=2, virtual_channels=8, n_layers=1), sd)
    lp = m._packed_params(dev())["layers"][0]
    N, E = inp["node_loc"].shape[0], inp["edge_index"].shape[1]
    rowptr, row, col, perm = be.build_csr(inp["edge_index"], N)
    ea = be.gather_rows(inp["edge_attr"], perm)
    g = torch.Generator().manual_seed(3)
    P, Q = torch.randn(N, 64, generator=g).to(dev()), torch.randn(N, 64, generator=g).to(dev())
    x4 = torch.zeros(N, 4, device=dev())
    x4[:, :3] = inp["node_loc"]
    for flags in (0, _lib.FLAG_NORMALIZE, _lib.FLAG_LAST):
        outs = []
        for fn in (be.edge_layer_simt, be.edge_layer, be.edge_layer_tf32, be.edge_layer_t16):
            agg_m, agg_x = torch.zeros(N, 64, device=dev()), torch.zeros(N, 4, device=dev())
            fn((N, E, 2, 8, 2), flags, row, col, ea, x4, P, Q, lp, None if flags & _lib.FLAG_LAST else agg_m,
               agg_x)
            torch.cuda.synchronize()
            outs.append((agg_m, agg_x))
        for name, o in (("fp16-split column-split (production)", outs[1]), ("3xTF32", outs[2]),
                        ("fp16-split thread-per-row", outs[3])):
            em = max_abs(o[0], outs[0][0]) / max(1e-9, float(outs[0][0].abs().max()))
            ex = max_abs(o[1], outs[0][1]) / max(1e-9, float(outs[0][1].abs().max()))
            print(f"flags {flags} {name}: rel err agg_m {em:.3e} agg_x {ex:.3e}")
            assert em <= 1e-5 and ex <= 1e-5


def test_edge_kernel_fp16_range_rescue():
    """Activations far outside the fp16 range (up to ~1e7) must still come out fp32-accurate: rows that
    overflow are re-encoded with a per-row power-of-two scale inside the kernel."""
    from tests.twin_backend import twin_backend
    be = twin_backend()
    w = synth.WORKLOADS["water3d_10k"]
    inp = to_dev(synth.make_partitions(w, n_nodes=20_000, seed=9)[0])
    sd = orc.init_state_dict(2, 0, 2, 64, 3, 1, seed=2, coord_gain=1.0)
    m = cuda_model(dict(node_feat_nf=2, node_attr_nf=0, edge_attr_nf=2, virtual_channels=3, n_layers=1), sd)
    lp = m._packed_params(dev())["layers"][0]
    N, E = inp["node_loc"].shape[0], inp["edge_index"].shape[1]
    rowptr, row, col, perm = be.build_csr(inp["edge_index"], N)
    ea = be.gather_rows(inp["edge_attr"], perm)
    g = torch.Generator().manual_seed(4)
    P, Q = torch.randn(N, 64, generator=g).to(dev()), torch.randn(N, 64, generator=g).to(dev())
    big = torch.rand(N, generator=g) < 0.05                      # 5 % of the destination rows get huge features
    scale = torch.where(big, 10 ** (3 + 4 * torch.rand(N, generator=g)), torch.ones(N)).to(dev())
    P = P * scale[:, None]
    x4 = torch.zeros(N, 4, device=dev())
    x4[:, :3] = inp["node_loc"]
    outs = []
    for fn in (be.edge_layer_simt, be.edge_layer, be.edge_layer_t16):
        agg_m, agg_x = torch.zeros(N, 64, device=dev()), torch.zeros(N, 4, device=dev())
        fn((N, E, 2, 3, 0), 0, row, col, ea, x4, P, Q, lp, agg_m, agg_x)
        torch.cuda.synchronize()
        outs.append((agg_m, agg_x[:, :3]))
    # fp64 reference of the same stage (torch restatement in double)
    ref_m, ref_x = torch.zeros(N, 64, device=dev(), dtype=torch.float64), torch.zeros(N, 4, device=dev(),
                                                                                      dtype=torch.float64)
    ShadowBackend().edge_layer((N, E, 2, 3, 0), 0, row, col, ea.double(), x4.double(), P.double(), Q.double(),
                               lp.double(), ref_m, ref_x)
    ref_x = ref_x[:, :3]
    assert float(ref_m.abs().max()) > 1e5                        # the case really leaves the fp16 range
    assert torch.isfinite(outs[1][0]).all() and torch.isfinite(outs[1][1]).all()

    def rowwise(o, r):                                           # rows differ by 7 orders of magnitude
        return float(((o.double() - r).abs().amax(dim=1) / r.abs().amax(dim=1).clamp(min=1e-9)).max())

    e_simt = (rowwise(outs[0][0], ref_m), rowwise(outs[0][1], ref_x))
    e_f16 = (rowwise(outs[1][0], ref_m), rowwise(outs[1][1], ref_x))
    e_t16 = (rowwise(outs[2][0], ref_m), rowwise(outs[2][1], ref_x))
    print(f"fp16 range rescue: row-wise rel err vs fp64  fp32-FMA twin {e_simt}  fp16-split tensor core: "
          f"column-split {e_f16}  thread-per-row {e_t16}")
    assert torch.isfinite(outs[2][0]).all() and torch.isfinite(outs[2][1]).all()
    for e_k in (e_f16, e_t16):
        assert e_k[0] <= 2e-5
        # Δx·φ has heavy cancellation at these magnitudes (fp32 FMA itself is at ~4e-5): the 22-bit operand split
        # may lose up to 2 more bits than fp32's 24, never the range
        assert e_k[1] <= max(8 * e_simt[1], 2e-5) and e_k[1] <= 1e-3


def test_edge_kernel_silu_batch_guard():
    """The tensor-core kernels take one reciprocal per FOUR SiLUs (1/d_i from the product d0·d1·d2·d3, common.cuh
    silu4p).  Pre-activations around −20 … −45 make that product leave the fp32 range while every single d stays
    finite; the stage-level guard must then redo the rows with per-element reciprocals.  Rows with such
    pre-activations sit next to ordinary ones in the same warp / quad."""
    from tests.twin_backend import twin_backend
    be = twin_backend()
    w = synth.WORKLOADS["water3d_10k"]
    inp = to_dev(synth.make_partitions(w, n_nodes=20_000, seed=11)[0])
    sd = orc.init_state_dict(2, 0, 2, 64, 3, 1, seed=3, coord_gain=1.0)
    m = cuda_model(dict(node_feat_nf=2, node_attr_nf=0, edge_attr_nf=2, virtual_channels=3, n_layers=1), sd)
    lp = m._packed_params(dev())["layers"][0]
    N, E = inp["node_loc"].shape[0], inp["edge_index"].shape[1]
    rowptr, row, col, perm = be.build_csr(inp["edge_index"], N)
    ea = be.gather_rows(inp["edge_attr"], perm)
    g = torch.Generator().manual_seed(5)
    P, Q = torch.randn(N, 64, generator=g), torch.randn(N, 64, generator=g)
    shifted = torch.rand(N, generator=g) < 0.1                    # 10 % of the destination rows
    shift = torch.where(shifted, -(18 + 30 * torch.rand(N, generator=g)), torch.zeros(N))
    cols = torch.rand(N, 64, generator=g) < 0.3                   # only some columns: mixed quads
    P = (P + shift[:, None] * cols).to(dev())
    Q = Q.to(dev())
    x4 = torch.zeros(N, 4, device=dev())
    x4[:, :3] = inp["node_loc"]
    outs = []
    for fn in (be.edge_layer_simt, be.edge_layer, be.edge_layer_t16):
        agg_m, agg_x = torch.zeros(N, 64, device=dev()), torch.zeros(N, 4, device=dev())
        fn((N, E, 2, 3, 0), 0, row, col, ea, x4, P, Q, lp, agg_m, agg_x)
        torch.cuda.synchronize()
        outs.append((agg_m, agg_x[:, :3]))
    ref_m, ref_x = torch.zeros(N, 64, device=dev(), dtype=torch.float64), torch.zeros(N, 4, device=dev(),
                                                                                      dtype=torch.float64)
    ShadowBackend().edge_layer((N, E, 2, 3, 0), 0, row, col, ea.double(), x4.double(), P.double(), Q.double(),
                               lp.double(), ref_m, ref_x)
    e_m0 = float((outs[0][0].double() - ref_m).abs().max() / ref_m.abs().max())
    for name, o in (("column-split", outs[1]), ("thread-per-row", outs[2])):
        assert torch.isfinite(o[0]).all() and torch.isfinite(o[1]).all()
        e_m = float((o[0].double() - ref_m).abs().max() / ref_m.abs().max())
        e_x = float((o[1].double() - ref_x[:, :3]).abs().max() / ref_x[:, :3].abs().max())
        print(f"silu batch guard [{name}]: rel err vs fp64  agg_m {e_m:.2e} (fp32-FMA twin {e_m0:.2e})  agg_x {e_x:.2e}")
        assert e_m <= 5e-6 and e_x <= 5e-5


@pytest.mark.parametrize("C,B", [(8, 1), (5, 1), (3, 7), (1, 2), (16, 3)])
def test_virtual_kernel_tensor_core_vs_fma_twin(C, B):
    """tcgen05 virtual-stage kernel against its fp32-FMA twin (single graph and a batch whose tiles
    straddle graph boundaries; C = 8 / 5 / 3 exercise full and ragged row tiles)."""
    from tests.twin_backend import twin_backend
    be = twin_backend()
    N = 100_003
    g = torch.Generator().manual_seed(C)
    sd = orc.init_state_dict(3, 0, 2, 64, C, 1, seed=5, coord_gain=1.0)
    m = cuda_model(dict(node_feat_nf=3, node_attr_nf=0, edge_attr_nf=2, virtual_channels=C, n_layers=1), sd)
    lp = m._packed_params(dev())["layers"][0]
    d = dev()
    batch = torch.sort(torch.randint(0, B, (N,), generator=g))[0].to(torch.int32).to(d)
    x4 = torch.zeros(N, 4, device=d)
    x4[:, :3] = torch.randn(N, 3, generator=g).to(d)
    Hn = torch.randn(N, 64, generator=g).to(d)
    Xv = torch.randn(B, 3, C, generator=g).to(d)
    G = torch.randn(B, C, 64, generator=g).to(d)
    K = 4 + 3 * C + 64 * C
    for flags in (0, _lib.FLAG_LAST):
        outs = []
        for fn in (be.virtual_layer_simt, be.virtual_layer, be.virtual_layer_tf32, be.virtual_layer_cs):
            agg_v, trans_v = torch.zeros(N, 64, device=d), torch.zeros(N, 4, device=d)
            vsum = torch.zeros(B, K, device=d)
            fn((N, B, 2, C, 0), flags, batch, x4, Hn, Xv, G, lp, None if flags else agg_v, trans_v, vsum)
            torch.cuda.synchronize()
            outs.append((agg_v, trans_v[:, :3], vsum))
        for impl, o in (("fp16-split thread-per-row (production)", outs[1]), ("3xTF32", outs[2]),
                        ("fp16-split column-split", outs[3])):
            for name, x, y in zip(("agg_v", "trans_v", "vsum"), o, outs[0]):
                err = max_abs(x, y) / max(1e-9, float(y.abs().max()))
                print(f"C={C} B={B} flags={flags} {impl} {name}: rel err {err:.3e}")
                assert err <= 2e-5, (impl, name, err)


@pytest.mark.parametrize("F,B", [(3, 1), (1, 11), (16, 2)])
def test_embed_kernel_tensor_core_vs_fma_twin(F, B):
    from tests.twin_backend import twin_backend
    be = twin_backend()
    N, C = 50_003, 3
    d = dev()
    g = torch.Generator().manual_seed(F)
    sd = orc.init_state_dict(F, 0, 2, 64, C, 1, seed=1)
    m = cuda_model(dict(node_feat_nf=F, node_attr_nf=0, edge_attr_nf=2, virtual_channels=C, n_layers=1), sd)
    pk = m._packed_params(d)
    feat, loc = (torch.randn(N, F, generator=g) * 3).to(d), torch.randn(N, 3, generator=g).to(d)
    batch = torch.sort(torch.randint(0, B, (N,), generator=g))[0].to(d)
    K = 4 + 3 * C + 64 * C
    outs = []
    for fn in (be.embed_simt, be.embed):
        z = lambda *s, dt=torch.float32: torch.zeros(*s, device=d, dtype=dt)
        h, x4, b32, P, Q, Hn, vsum = z(N, 64), z(N, 4), z(N, dt=torch.int32), z(N, 64), z(N, 64), z(N, 64), z(B, K)
        fn((N, B, F, 2, C, 0), feat, loc, batch, pk["emb_wt"], pk["emb_b"], pk["layers"][0], h, x4, b32, P, Q, Hn, vsum)
        torch.cuda.synchronize()
        outs.append(dict(h=h, x4=x4, b32=b32.float(), P=P, Q=Q, Hn=Hn, vsum=vsum[:, :4]))
    for k in outs[0]:
        err = max_abs(outs[1][k], outs[0][k]) / max(1e-9, float(outs[0][k].abs().max()))
        print(f"embed F={F} B={B} {k}: rel err {err:.3e}")
        assert err <= 2e-5, (k, err)


@pytest.mark.parametrize("Na,B,big", [(2, 1, False), (0, 9, False), (2, 1, True)])
def test_node_kernel_tensor_core_vs_fma_twin(Na, B, big):
    """tcgen05 node-update kernel against its fp32-FMA twin: single graph / batch with straddling tiles, with and
    without node attributes, last-layer mode, and (big) features far outside the fp16 range."""
    from tests.twin_backend import twin_backend
    be = twin_backend()
    N, C = 70_001, 5
    d = dev()
    g = torch.Generator().manual_seed(Na + B)
    sd = orc.init_state_dict(3, Na, 2, 64, C, 2, seed=8, coord_gain=1.0)
    m = cuda_model(dict(node_feat_nf=3, node_attr_nf=Na, edge_attr_nf=2, virtual_channels=C, n_layers=2), sd)
    lps = m._packed_params(d)["layers"]
    R = lambda *s: torch.randn(*s, generator=g).to(d)
    batch = torch.sort(torch.randint(0, B, (N,), generator=g))[0].to(torch.int32).to(d)
    deg = torch.randint(0, 30, (N,), generator=g)
    rowptr = torch.zeros(N + 1, dtype=torch.int32)
    rowptr[1:] = torch.cumsum(deg, 0).to(torch.int32)
    rowptr = rowptr.to(d)
    h, agg_m, agg_v, vel, attr = R(N, 64), R(N, 64) * 5, R(N, 64), R(N, 3), (R(N, Na) if Na else None)
    if big:
        sc = torch.where(torch.rand(N, generator=g) < 0.03, 10 ** (3 + 3 * torch.rand(N, generator=g)),
                         torch.ones(N)).to(d)
        h, agg_m = h * sc[:, None], agg_m * sc[:, None]
    x4, agg_x, trans_v = torch.zeros(N, 4, device=d), torch.zeros(N, 4, device=d), torch.zeros(N, 4, device=d)
    x4[:, :3], agg_x[:, :3], trans_v[:, :3] = R(N, 3), R(N, 3), R(N, 3)
    K = 4 + 3 * C + 64 * C
    for flags in (0, _lib.FLAG_LAST):
        outs = []
        for fn in (be.node_layer_simt, be.node_layer):
            new = lambda *s: torch.zeros(*s, device=d)
            h2, x42, P2, Q2, Hn2, loc, vsum = new(N, 64), new(N, 4), new(N, 64), new(N, 64), new(N, 64), new(N, 3), new(B, K)
            last = bool(flags)
            fn((N, B, 2, C, Na), flags, rowptr, batch, h, x4, vel, attr, None if last else agg_m, agg_x,
               None if last else agg_v, trans_v, lps[0], None if last else lps[1], None if last else h2, x42,
               None if last else P2, None if last else Q2, None if last else Hn2, loc if last else None, vsum)
            torch.cuda.synchronize()
            outs.append(dict(h2=h2, x=x42[:, :3], P=P2, Q=Q2, Hn=Hn2, loc=loc, vsum=vsum[:, :4]))
        if big:      # fp64 restatement of the stage: rows differ by 6 orders of magnitude, heads cancel heavily
            D = lambda t_: None if t_ is None else t_.double()
            z = lambda *s_: torch.zeros(*s_, device=d, dtype=torch.float64)
            h2, x42, P2, Q2, Hn2, loc, vsum = z(N, 64), z(N, 4), z(N, 64), z(N, 64), z(N, 64), z(N, 3), z(B, K)
            last = bool(flags)
            ShadowBackend().node_layer((N, B, 2, C, Na), flags, rowptr, batch, D(h), D(x4), D(vel), D(attr),
                                       None if last else D(agg_m), D(agg_x), None if last else D(agg_v), D(trans_v),
                                       lps[0].double(), None if last else lps[1].double(), h2, x42, P2, Q2, Hn2,
                                       loc if last else None, vsum)
            ref64 = dict(h2=h2, x=x42[:, :3], P=P2, Q=Q2, Hn=Hn2, loc=loc, vsum=vsum[:, :4])
        for k in outs[0]:
            if big:
                r = ref64[k]
                rw = lambda o: float(((o.double() - r).abs().amax(1) / r.abs().amax(1).clamp(min=1e-6)).max())
                e_fma, e_tc = rw(outs[0][k]), rw(outs[1][k])
                print(f"Na={Na} B={B} big flags={flags} {k}: row-wise rel err vs fp64: fp32-FMA {e_fma:.3e}  tensor-core {e_tc:.3e}")
                assert e_tc <= max(8 * e_fma, 2e-5) and e_tc <= 2e-3, (k, e_fma, e_tc)
            else:
                ref, got = outs[0][k], outs[1][k]
                err = max_abs(got, ref) / max(1e-9, float(ref.abs().max()))
                print(f"Na={Na} B={B} flags={flags} {k}: rel err {err:.3e}")
                assert err <= 2e-5, (k, err)


@pytest.mark.parametrize("name", SINGLE_CASES)
def test_golden_fixtures(name):
    z, kw, sd = load_golden(name)
    inp = golden_inputs(z)
    m = cuda_model(kw, sd)
    with torch.no_grad():
        out, X = m(**to_dev(inp))
    check_close(out, X, torch.from_numpy(z["out64.node_loc"]), torch.from_numpy(z["out64.virtual_loc"]),
                inp["node_loc"], name)


def _stage_inputs(kw, sd, inp):
    """Run the torch stand-in on the GPU to get every intermediate buffer of layer 0."""
    m = cuda_model(kw, sd)
    m._backend = ShadowBackend()
    return m


@pytest.mark.parametrize("name", SINGLE_CASES)
def test_per_layer_trace_against_reference(name):
    """h, x, Hv and X after EVERY layer of the CUDA path against the traces the unmodified reference produced
    (forward hooks in oracle/make_golden.py) — not just the final coordinates: parity is deceptively easy at init,
    coordinates barely see a wrong edge MLP (SURVEY §7).  The training-path forward keeps each layer's inputs, i.e. the
    previous layer's outputs; one extra (dummy) layer makes the last real layer's h'/Hv' live (they are dead code
    otherwise, FastEGNN.py:307)."""
    z, kw, sd = load_golden(name)
    inp = golden_inputs(z)
    L = kw["n_layers"]
    ref = {k: golden_trace(z, k) for k in ("h", "x", "Hv", "X")}
    assert all(len(v) == L for v in ref.values())
    sdx = dict(sd)
    for k, v in sd.items():
        if k.startswith(f"gcl_{L - 1}."):
            sdx[k.replace(f"gcl_{L - 1}.", f"gcl_{L}.")] = v.clone()
    m = cuda_model(dict(kw, n_layers=L + 1), sdx).train()
    kept = []
    m._keep_state = kept
    m(**to_dev(inp))
    torch.cuda.synchronize()
    layers = kept[0]["layers"]
    assert len(layers) == L + 1
    worst = {}
    for l in range(L):
        nxt = layers[l + 1]                      # inputs of layer l+1 == outputs of layer l
        got = dict(h=nxt["h"], x=nxt["x4"][:, :3], Hv=nxt["Hv"].transpose(1, 2), X=nxt["Xv"])
        for k, g in got.items():
            r = ref[k][l]
            e = max_abs(g.cpu(), r) / max(1.0, float(r.abs().max()))
            worst[k] = max(worst.get(k, 0.0), e)
            assert e <= 2e-5, f"{name} layer {l} {k}: rel err {e:.3e}"
    print(f"{name}: per-layer trace vs reference, worst relative error " +
          ", ".join(f"{k} {v:.2e}" for k, v in worst.items()))


def _kernel_vs_shadow(name):
    z, kw, sd = load_golden(name)
    inp = to_dev(golden_inputs(z))
    return z, kw, sd, inp


@pytest.mark.parametrize("name", SINGLE_CASES)
def test_each_kernel_against_torch_restatement(name):
    """Drive both backends through layer 0 with identical inputs and compare every output buffer."""
    from distegnn_b200.backend import cuda_backend
    z, kw, sd, inp = _kernel_vs_shadow(name)
    m = cuda_model(kw, sd)
    pk = m._packed_params(dev())
    A, C, Na, F = kw["edge_attr_nf"], kw["virtual_channels"], kw["node_attr_nf"], kw["node_feat_nf"]
    N, E, B = inp["node_loc"].shape[0], inp["edge_index"].shape[1], inp["loc_mean"].shape[0]
    K = 4 + 3 * C + 64 * C
    res = {}
    for tag, be in (("cuda", cuda_backend()), ("ref", ShadowBackend())):
        new = lambda *s, dt=torch.float32: torch.zeros(*s, dtype=dt, device=dev())
        h, P, Q, Hn, agg_m, agg_v = (new(N, 64) for _ in range(6))
        x4, agg_x, trans_v = new(N, 4), new(N, 4), new(N, 4)
        b32, vsum, G = new(N, dt=torch.int32), new(B, K), new(B, C, 64)
        Xv = inp["loc_mean"].unsqueeze(-1).repeat(1, 1, C).contiguous()
        Hv = pk["hv0"].unsqueeze(0).repeat(B, 1, 1).contiguous()
        rowptr, row, col, perm = be.build_csr(inp["edge_index"].contiguous(), N)
        ea = be.gather_rows(inp["edge_attr"], perm)
        be.embed((N, B, F, A, C, Na), inp["node_feat"], inp["node_loc"], inp["data_batch"], pk["emb_wt"],
                 pk["emb_b"], pk["layers"][0], h, x4, b32, P, Q, Hn, vsum)
        vs0 = vsum.clone()
        be.virtual_update((B, A, C, Na), _lib.FLAG_INIT, vsum, Xv, Hv, None, pk["layers"][0], G)
        G0 = G.clone()
        vsum.zero_()
        flags = _lib.FLAG_NORMALIZE if kw["normalize"] else 0
        be.edge_layer((N, E, A, C, Na), flags, row, col, ea, x4, P, Q, pk["layers"][0], agg_m, agg_x)
        be.virtual_layer((N, B, A, C, Na), flags, b32, x4, Hn, Xv, G, pk["layers"][0], agg_v, trans_v, vsum)
        vs1 = vsum.clone()
        h2, x42, P2, Q2, Hn2 = new(N, 64), new(N, 4), new(N, 64), new(N, 64), new(N, 64)
        be.node_layer((N, B, A, C, Na), flags, rowptr, b32, h, x4, inp["node_vel"], inp["node_attr"], agg_m,
                      agg_x, agg_v, trans_v, pk["layers"][0], pk["layers"][1], h2, x42, P2, Q2, Hn2, None,
                      vsum)
        vs2 = vsum.clone()
        be.virtual_update((B, A, C, Na), 0, vsum, Xv, Hv, pk["layers"][0], pk["layers"][1], G)
        torch.cuda.synchronize()
        res[tag] = dict(rowptr=rowptr, row=row, col=col, ea=ea, h=h, x4=x4[:, :3], b32=b32, P=P, Q=Q, Hn=Hn,
                        vs0=vs0[:, :4], G0=G0, agg_m=agg_m, agg_x=agg_x[:, :3], agg_v=agg_v,
                        trans_v=trans_v[:, :3], vs1=vs1[:, 4:], h2=h2, x42=x42[:, :3], P2=P2, Q2=Q2, Hn2=Hn2,
                        vs2=vs2[:, :4], Xv=Xv, Hv=Hv, G1=G)
    bad = []
    for k in res["ref"]:
        a, b = res["cuda"][k], res["ref"][k]
        if a.dtype in (torch.int32, torch.int64):
            if k in ("rowptr", "row", "b32"):
                ok = torch.equal(a, b)
            else:   # col: same multiset per row (stable sort makes it identical)
                ok = torch.equal(a, b)
            err = 0.0 if ok else 1.0
        else:
            scale = max(1e-6, float(b.abs().max()))
            err = max_abs(a, b) / scale
            ok = err <= 2e-5
        print(f"{name:24s} {k:8s} rel err {err:.3e}")
        if not ok:
            bad.append((k, err))
    assert not bad, bad


def _rotation(seed):
    rng = np.random.default_rng(seed)
    q, _ = np.linalg.qr(rng.normal(size=(3, 3)))
    if np.linalg.det(q) < 0:
        q[:, 0] = -q[:, 0]
    return torch.from_numpy(q.astype(np.float32))


def test_equivariance_reference_script_on_gpu():
    """equivariant_test.py restated (10 nodes, 20 random edges incl. self loops/duplicates, F=1, A=1,
    C=3, 4 layers, atol 1e-4) — several seeds, through the CUDA path."""
    for seed in range(5):
        torch.manual_seed(seed)
        m = FastEGNN(node_feat_nf=1, node_attr_nf=0, edge_attr_nf=1, hidden_nf=64, virtual_channels=3,
                     world_size=1, n_layers=4).to(dev())
        g = torch.Generator().manual_seed(100 + seed)
        n, e = 10, 20
        x, v = torch.rand(n, 3, generator=g) * 10, torch.rand(n, 3, generator=g) * 10
        f = torch.rand(n, 1, generator=g) * 10
        ei = torch.randint(0, 10, (2, e), generator=g)
        ea = torch.rand(e, 1, generator=g) * 10
        b = torch.zeros(n, dtype=torch.long)
        R, t = _rotation(seed), torch.randn(3, generator=g) * 5
        d = dev()
        with torch.no_grad():
            out, _ = m(f.to(d), x.to(d), v.to(d), x.mean(0, keepdim=True).to(d), ei.to(d), b.to(d), ea.to(d))
            xr = x @ R + t
            out_r, _ = m(f.to(d), xr.to(d), (v @ R).to(d), xr.mean(0, keepdim=True).to(d), ei.to(d), b.to(d),
                         ea.to(d))
        assert torch.allclose(out.cpu() @ R + t, out_r.cpu(), atol=1e-4)


@pytest.mark.parametrize("wname,n,coord_gain", [("water3d_10k", 10_000, 0.05), ("fluid113k", 30_000, 0.05),
                                                ("nbody100", 100, 0.001)])
def test_workloads_against_oracle(wname, n, coord_gain):
    """BASELINE.json configs at sizes the fp64 oracle finishes in seconds, trained-like coord heads."""
    w = synth.WORKLOADS[wname]
    inp = synth.make_partitions(w, n_nodes=n, seed=3)[0]
    sd = orc.init_state_dict(w.node_feat_nf, w.node_attr_nf, w.edge_attr_nf, 64, w.virtual_channels, 4,
                             seed=4, coord_gain=coord_gain)
    kw = dict(node_feat_nf=w.node_feat_nf, node_attr_nf=w.node_attr_nf, edge_attr_nf=w.edge_attr_nf,
              virtual_channels=w.virtual_channels, n_layers=4, normalize=w.normalize)
    m = cuda_model(kw, sd)
    with torch.no_grad():
        out, X = m(**to_dev(inp))
    ref, refX = oracle64(sd, inp, w.normalize)
    check_close(out, X, ref, refX, inp["node_loc"], wname)


def test_batched_graphs_against_oracle():
    """N-body style batch: 40 graphs x 100 nodes fully connected (tiles straddle graph boundaries)."""
    w = synth.WORKLOADS["nbody100"]
    parts = [synth.make_partitions(w, seed=s)[0] for s in range(40)]
    n = 100
    cat = lambda k: torch.cat([p[k] for p in parts])
    inp = dict(node_feat=cat("node_feat"), node_loc=cat("node_loc"), node_vel=cat("node_vel"),
               loc_mean=cat("loc_mean"),
               edge_index=torch.cat([p["edge_index"] + i * n for i, p in enumerate(parts)], 1),
               data_batch=torch.arange(40).repeat_interleave(n), edge_attr=cat("edge_attr"), node_attr=None)
    sd = orc.init_state_dict(2, 0, 2, 64, 3, 4, seed=9, coord_gain=0.01)
    kw = dict(node_feat_nf=2, node_attr_nf=0, edge_attr_nf=2, virtual_channels=3, n_layers=4, normalize=True)
    m = cuda_model(kw, sd)
    with torch.no_grad():
        out, X = m(**to_dev(inp))
    ref, refX = oracle64(sd, inp, True)
    check_close(out, X, ref, refX, inp["node_loc"], "nbody batch 40")


def test_edge_cases():
    d = dev()
    sd = orc.init_state_dict(2, 0, 2, 64, 3, 2, seed=1, coord_gain=0.1)
    kw = dict(node_feat_nf=2, node_attr_nf=0, edge_attr_nf=2, virtual_channels=3, n_layers=2)
    m = cuda_model(kw, sd)
    g = torch.Generator().manual_seed(0)
    for n, ei in [(7, torch.zeros(2, 0, dtype=torch.long)),                       # no edges at all
                  (1, torch.zeros(2, 3, dtype=torch.long)),                       # single node, self loops
                  (300, torch.stack([torch.zeros(299, dtype=torch.long), torch.arange(1, 300)])),  # star: deg 299
                  (129, torch.randint(0, 129, (2, 128 * 3 + 1), generator=g))]:  # ragged last tile
        inp = dict(node_feat=torch.randn(n, 2, generator=g), node_loc=torch.randn(n, 3, generator=g),
                   node_vel=torch.randn(n, 3, generator=g), loc_mean=torch.zeros(1, 3), edge_index=ei,
                   data_batch=torch.zeros(n, dtype=torch.long),
                   edge_attr=torch.rand(ei.shape[1], 2, generator=g), node_attr=None)
        with torch.no_grad():
            out, X = m(**to_dev(inp))
        ref, refX = oracle64(sd, inp, False)
        check_close(out, X, ref, refX, inp["node_loc"], f"edge case n={n} e={ei.shape[1]}")
    with pytest.raises(ValueError):
        m(torch.zeros(4, 3, device=d), torch.zeros(4, 3, device=d), torch.zeros(4, 3, device=d),
          torch.zeros(1, 3, device=d), torch.zeros(2, 0, dtype=torch.long, device=d),
          torch.zeros(4, dtype=torch.long, device=d), torch.zeros(0, 2, device=d))


def test_cuda_graph_replay_matches_eager():
    """model.cuda_graph = True: captured forward == eager forward, replays track in-place input updates, and a new
    input tensor triggers a re-capture instead of a stale replay."""
    w = synth.WORKLOADS["water3d_10k"]
    inp = to_dev(synth.make_partitions(w, n_nodes=10_000, seed=4)[0])
    sd = orc.init_state_dict(2, 0, 2, 64, 3, 4, seed=6, coord_gain=0.05)
    kw = dict(node_feat_nf=2, node_attr_nf=0, edge_attr_nf=2, virtual_channels=3, n_layers=4)
    m = cuda_model(kw, sd)
    with torch.no_grad():
        e_out, e_X = m(**inp)
        m.cuda_graph = True
        g_out, g_X = m(**inp)                     # capture + first replay
        g_out2, _ = m(**inp)                      # replay
        assert len(m._graph_cache) == 1
        assert max_abs(g_out, e_out) <= 1e-6 and max_abs(g_X, e_X) <= 1e-6 and max_abs(g_out2, e_out) <= 1e-6
        inp["node_loc"].add_(0.01)                # in-place update of a keyed tensor: same graph, new contents
        inp["loc_mean"].add_(0.01)
        g_out3, _ = m(**inp)
        m.cuda_graph = False
        e_out3, _ = m(**inp)
        assert len(m._graph_cache) == 1 and max_abs(g_out3, e_out3) <= 1e-6 and max_abs(g_out3, g_out) > 1e-3
        m.cuda_graph = True
        inp2 = {**inp, "node_vel": inp["node_vel"].clone() * 2}
        g_out4, _ = m(**inp2)                     # different tensor -> new capture
        m.cuda_graph = False
        e_out4, _ = m(**inp2)
        assert len(m._graph_cache) == 2 and max_abs(g_out4, e_out4) <= 1e-6


def test_large_graph_properties():
    """config-5-like density at 200k nodes (≈4M edges): SE(3) equivariance, invariance to a random
    permutation of the edge list, and agreement with the fp32 oracle (one forward on host cores)."""
    w = synth.WORKLOADS["synth1m"]
    inp = synth.make_partitions(w, n_nodes=200_000, seed=0)[0]
    sd = orc.init_state_dict(3, 2, 2, 64, 8, 4, seed=2, coord_gain=0.05)
    kw = dict(node_feat_nf=3, node_attr_nf=2, edge_attr_nf=2, virtual_channels=8, n_layers=4)
    m = cuda_model(kw, sd)
    di = to_dev(inp)
    with torch.no_grad():
        out, X = m(**di)
        perm = torch.randperm(inp["edge_index"].shape[1], generator=torch.Generator().manual_seed(1)).to(dev())
        out_p, X_p = m(**{**di, "edge_index": di["edge_index"][:, perm].contiguous(),
                          "edge_attr": di["edge_attr"][perm].contiguous()})
        R, t = _rotation(5).to(dev()), torch.tensor([0.3, -1.0, 2.0], device=dev())
        xr = di["node_loc"] @ R + t
        out_r, _ = m(**{**di, "node_loc": xr, "node_vel": di["node_vel"] @ R,
                        "loc_mean": di["loc_mean"] @ R + t})
    scale = float(out.abs().max())
    assert max_abs(out, out_p) <= 2e-6 * max(1.0, scale)
    assert max_abs(X, X_p) <= 2e-6 * max(1.0, scale)
    assert max_abs(out @ R + t, out_r) <= 1e-4
    ref, refX = orc.forward(sd, **inp)
    check_close(out, X, ref, refX, inp["node_loc"], "synth 200k")


def test_full_size_config5_properties():
    """BASELINE.json config 5 at FULL size on one GPU (1,000,000 nodes, ~20.6 M directed edges, C = 8): the CPU
    oracle cannot check this size in reasonable time, so the checks are size-independent properties —
    SE(3) equivariance (the reference's own test, atol 1e-4), invariance to the order of the edge list, run-to-run
    reproducibility, and finiteness."""
    w = synth.WORKLOADS["synth1m"]
    inp = synth.make_partitions(w, seed=0)[0]
    assert inp["node_loc"].shape[0] == 1_000_000 and inp["edge_index"].shape[1] > 20_000_000
    sd = orc.init_state_dict(3, 2, 2, 64, 8, 4, seed=2, coord_gain=0.05)
    m = cuda_model(dict(node_feat_nf=3, node_attr_nf=2, edge_attr_nf=2, virtual_channels=8, n_layers=4), sd)
    di = to_dev(inp)
    with torch.no_grad():
        out, X = m(**di)
        out2, X2 = m(**di)
        perm = torch.randperm(inp["edge_index"].shape[1], generator=torch.Generator().manual_seed(1)).to(dev())
        out_p, X_p = m(**{**di, "edge_index": di["edge_index"][:, perm].contiguous(),
                          "edge_attr": di["edge_attr"][perm].contiguous()})
        R, t = _rotation(7).to(dev()), torch.tensor([-0.7, 0.4, 1.5], device=dev())
        out_r, X_r = m(**{**di, "node_loc": di["node_loc"] @ R + t, "node_vel": di["node_vel"] @ R,
                          "loc_mean": di["loc_mean"] @ R + t})
    assert torch.isfinite(out).all() and torch.isfinite(X).all()
    disp = float((out - di["node_loc"]).abs().max())
    assert disp > 1e-4                                               # the model really moves the particles
    scale = max(1.0, float(out.abs().max()))
    print(f"1M nodes: displacement scale {disp:.3e}; rerun diff {max_abs(out, out2):.2e}; "
          f"edge-permutation diff {max_abs(out, out_p):.2e}; equivariance residual "
          f"{max_abs(out @ R + t, out_r):.2e}; virtual {max_abs(X.permute(0, 2, 1) @ R + t, X_r.permute(0, 2, 1)):.2e}")
    assert max_abs(out, out2) <= 2e-6 * scale and max_abs(X, X2) <= 2e-6 * scale
    assert max_abs(out, out_p) <= 2e-6 * scale and max_abs(X, X_p) <= 2e-6 * scale
    assert max_abs(out @ R + t, out_r) <= 1e-4
    assert max_abs(X.permute(0, 2, 1) @ R + t, X_r.permute(0, 2, 1)) <= 1e-4


# ---- backward kernels (SURVEY §8 f-1): each stage against torch.autograd on its float64 restatement --------------------
def _rel(a, b):
    return float((a.double() - b).abs().max() / b.abs().max().clamp(min=1e-30))


@pytest.mark.gpu
@pytest.mark.parametrize("flags,A", [(0, 2), (_lib.FLAG_NORMALIZE, 2), (_lib.FLAG_LAST, 2), (0, 0)])
def test_edge_stage_backward(flags, A):
    from tests import shadow_autograd as sa
    from tests.twin_backend import twin_backend
    be = twin_backend()
    w = synth.WORKLOADS["water3d_10k"]
    inp = to_dev(synth.make_partitions(w, n_nodes=6_000, seed=21)[0])
    C, Na = 3, 0
    sd = orc.init_state_dict(2, Na, A, 64, C, 1, seed=5, coord_gain=1.0)
    m = cuda_model(dict(node_feat_nf=2, node_attr_nf=Na, edge_attr_nf=A, virtual_channels=C, n_layers=1), sd)
    lp = m._packed_params(dev())["layers"][0]
    N, E = inp["node_loc"].shape[0], inp["edge_index"].shape[1]
    rowptr, row, col, perm = be.build_csr(inp["edge_index"], N)
    ea = be.gather_rows(inp["edge_attr"], perm)[:, :A].contiguous() if A else None
    g = torch.Generator().manual_seed(6)
    P, Q = torch.randn(N, 64, generator=g).to(dev()), torch.randn(N, 64, generator=g).to(dev())
    x4 = torch.zeros(N, 4, device=dev())
    x4[:, :3] = inp["node_loc"]
    g_m = torch.randn(N, 64, generator=g).to(dev())
    g_x = torch.zeros(N, 4, device=dev())
    g_x[:, :3] = torch.randn(N, 3, generator=g).to(dev())
    last = bool(flags & _lib.FLAG_LAST)
    # reference: autograd in float64
    Pd, Qd, xd, lpd = (t.double().requires_grad_(True) for t in (P, Q, x4[:, :3], lp))
    am, ax = sa.edge_stage((N, E, A, C, Na), flags, row, col, ea.double() if A else None, xd, Pd, Qd, lpd)
    loss = (ax * g_x[:, :3].double()).sum() + (0 if last else (am * g_m.double()).sum())
    rP, rQ, rx, rlp = torch.autograd.grad(loss, (Pd, Qd, xd, lpd))
    # kernels: the tensor-core production kernel and its fp32-FMA twin
    offs, _ = _lib.param_layout(A, C, Na)
    for name, fn in (("tcgen05", be.edge_layer_bwd), ("fp32-FMA twin", be.edge_layer_bwd_simt)):
        gP, gQ, gx4, glp = (torch.zeros_like(t) for t in (P, Q, x4, lp))
        fn((N, E, A, C, Na), flags, row, col, ea, x4, P, Q, lp, None if last else g_m, g_x, gP, gQ, gx4, glp)
        torch.cuda.synchronize()
        errs = dict(P=_rel(gP, rP), Q=_rel(gQ, rQ), x=_rel(gx4[:, :3], rx), params=_rel(glp, rlp))
        for k in ("E_W1R", "E_W1E", "E_W2", "E_B2", "E_WC", "E_BC", "E_W3"):
            n = {"E_W1E": A * 64, "E_W2": 4096, "E_WC": 4096}.get(k, 64)
            if n:
                errs[k] = _rel(glp[offs[k]:offs[k] + n], rlp[offs[k]:offs[k] + n])
        print(f"edge stage backward [{name}] flags={flags} A={A}: rel err vs float64 autograd "
              + ", ".join(f"{k} {v:.1e}" for k, v in errs.items()))
        assert max(errs.values()) <= 2e-5, name


@pytest.mark.gpu
@pytest.mark.parametrize("C,B,last", [(8, 1, False), (3, 5, False), (5, 1, True), (16, 2, False), (1, 3, False)])
def test_virtual_stage_backward(C, B, last):
    from tests import shadow_autograd as sa
    from tests.twin_backend import twin_backend
    be = twin_backend()
    A, Na, N = 2, 0, 5_003
    sd = orc.init_state_dict(2, Na, A, 64, C, 1, seed=8, coord_gain=1.0)
    m = cuda_model(dict(node_feat_nf=2, node_attr_nf=Na, edge_attr_nf=A, virtual_channels=C, n_layers=1), sd)
    lp = m._packed_params(dev())["layers"][0]
    offs, _ = _lib.param_layout(A, C, Na)
    g = torch.Generator().manual_seed(9)
    rnd = lambda *s: torch.randn(*s, generator=g).to(dev())
    batch = torch.sort(torch.randint(0, B, (N,), generator=g)).values.to(torch.int32).to(dev())
    x4 = torch.zeros(N, 4, device=dev())
    x4[:, :3] = rnd(N, 3)
    Hn, Xv, G = rnd(N, 64), rnd(B, 3, C), rnd(B, C, 64)
    K = 4 + 3 * C + 64 * C
    g_aggv, g_tv, g_vsum = rnd(N, 64), torch.zeros(N, 4, device=dev()), rnd(B, K)
    g_tv[:, :3] = rnd(N, 3)
    if last:
        g_vsum[:, 4 + 3 * C:] = 0
    flags = _lib.FLAG_LAST if last else 0
    # reference
    xd, Hd, Xd, Gd, lpd = (t.double().requires_grad_(True) for t in (x4[:, :3], Hn, Xv, G, lp))
    av, tv, tail = sa.virtual_stage((N, B, A, C, Na), flags, batch, xd, Hd, Xd, Gd, lpd)
    loss = (tv * g_tv[:, :3].double()).sum() + (tail * g_vsum[:, 4:].double()).sum()
    if not last:
        loss = loss + (av * g_aggv.double()).sum()
    rx, rH, rX, rG, rlp = torch.autograd.grad(loss, (xd, Hd, Xd, Gd, lpd))
    # kernels: the tensor-core production kernel and its fp32-FMA twin
    wT = torch.stack([lp[offs[k]:offs[k] + 4096].view(64, 64).t().contiguous() for k in ("V_W2", "V_WXV", "V_WX")])
    wimg = be.virtual_bwd_prepare(A, C, Na, lp)
    for name, fn, w in (("tcgen05", be.virtual_layer_bwd, wimg), ("fp32-FMA twin", be.virtual_layer_bwd_simt, wT)):
        gHn, gxv = torch.empty(N, 64, device=dev()), torch.empty(N, 4, device=dev())
        gG, gXv, glp = torch.zeros_like(G), torch.zeros_like(Xv), torch.zeros_like(lp)
        fn((N, B, A, C, Na), flags, batch, x4, Hn, Xv, G, lp, w, None if last else g_aggv, g_tv, g_vsum, gHn, gxv, gG, gXv,
           glp)
        torch.cuda.synchronize()
        errs = dict(Hn=_rel(gHn, rH), x=_rel(gxv[:, :3], rx), G=_rel(gG, rG), Xv=_rel(gXv, rX))
        for k in ("V_W1R", "V_W2", "V_B2", "V_WXV", "V_BXV", "V_W3XV", "V_WX", "V_BX", "V_W3X"):
            n = 4096 if k in ("V_W2", "V_WXV", "V_WX") else 64
            errs[k] = _rel(glp[offs[k]:offs[k] + n], rlp[offs[k]:offs[k] + n])
        print(f"virtual stage backward [{name}] C={C} B={B} last={last}: rel err vs float64 autograd "
              + ", ".join(f"{k} {v:.1e}" for k, v in errs.items()))
        assert max(errs.values()) <= 2e-5, name


# ---- the whole training path on the GPU: forward kernels + backward kernels + dense stages, against the reference's own
# gradients (fixtures from oracle/make_golden_grads.py) and against float64 autograd through the oracle -------------------
def _param_grad_errors(model, ref_grads, samples=None):
    """`samples`: parameter -> flat indices of the entries `ref_grads` holds (tests.helpers.grad_sample), None = all."""
    errs, dead = {}, 0
    for k, p in model.named_parameters():
        ref = ref_grads[k]
        g = p.grad if p.grad is not None else torch.zeros_like(p)
        if samples and samples[k] is not None:
            g = g.reshape(-1)[samples[k].to(g.device)]
        if float(ref.abs().max()) == 0.0:
            assert float(g.abs().max()) == 0.0, k
            dead += 1
            continue
        errs[k] = float((g.detach().cpu().double() - ref.double()).abs().max() / ref.double().abs().max())
    return errs, dead


@pytest.mark.gpu
@pytest.mark.parametrize("name", SINGLE_CASES)
def test_training_path_gradients_against_reference_fixtures(name):
    import numpy as np
    from tests.helpers import GOLDEN
    import os
    z, kw, sd = load_golden(name)
    zg = np.load(os.path.join(GOLDEN, name + ".grads.npz"))
    inp = to_dev(golden_inputs(z))
    m = cuda_model(kw, sd).train()
    out, X = m(**inp)
    assert out.requires_grad and X.requires_grad
    loss = (out * torch.from_numpy(zg["cot.out"]).float().to(dev())).sum() + \
           (X * torch.from_numpy(zg["cot.X"]).float().to(dev())).sum()
    loss.backward()
    assert abs(float(loss) - float(zg["loss"])) <= 1e-4 * max(1.0, abs(float(zg["loss"])))
    keys = [k for k, _ in m.named_parameters()]
    errs, dead = _param_grad_errors(m, {k: torch.from_numpy(zg["grad." + k]) for k in keys},
                                    {k: grad_sample(zg, "grad." + k) for k in keys})
    worst = max(errs, key=errs.get)
    print(f"{name}: training-path gradients vs reference fp64: worst {worst} {errs[worst]:.2e}; {dead} dead parameters")
    assert errs[worst] <= 2e-4          # the reference's own fp32 run is within 3e-5 of its fp64 run on these cases


@pytest.mark.gpu
@pytest.mark.parametrize("wname,n,normalize", [("fluid113k", 4000, False), ("water3d_10k", 3000, True)])
def test_training_path_gradients_against_oracle_autograd(wname, n, normalize):
    w = synth.WORKLOADS[wname]
    host = synth.make_partitions(w, n_nodes=n, seed=31)[0]
    F, Na, A, C = w.node_feat_nf, w.node_attr_nf, 2, w.virtual_channels
    sd = orc.init_state_dict(F, Na, A, 64, C, 3, seed=12, coord_gain=0.05)
    kw = dict(node_feat_nf=F, node_attr_nf=Na, edge_attr_nf=A, virtual_channels=C, n_layers=3, normalize=normalize)
    g = torch.Generator().manual_seed(13)
    cot_out, cot_X = torch.randn(n, 3, generator=g), torch.randn(1, 3, C, generator=g)
    # oracle, float64, CPU autograd
    sd64 = {k: v.double().requires_grad_(True) for k, v in sd.items()}
    inp64 = {k: (v.double() if (v is not None and v.is_floating_point()) else v) for k, v in host.items()}
    o64, X64 = orc.forward(sd64, **inp64, normalize=normalize)
    l64 = (o64 * cot_out.double()).sum() + (X64 * cot_X.double()).sum()
    keys = list(sd64)
    ref = dict(zip(keys, torch.autograd.grad(l64, [sd64[k] for k in keys], allow_unused=True)))
    ref = {k: (v if v is not None else torch.zeros_like(sd64[k])) for k, v in ref.items()}
    # product
    m = cuda_model(kw, sd).train()
    out, X = m(**to_dev(host))
    loss = (out * cot_out.to(dev())).sum() + (X * cot_X.to(dev())).sum()
    loss.backward()
    errs, dead = _param_grad_errors(m, ref)
    worst = max(errs, key=errs.get)
    print(f"{wname} n={n} normalize={normalize}: gradients vs oracle fp64 autograd: worst {worst} {errs[worst]:.2e}, "
          f"median {sorted(errs.values())[len(errs) // 2]:.2e}; loss {float(loss):.6f} vs {float(l64):.6f}")
    assert errs[worst] <= 5e-4


@pytest.mark.gpu
def test_training_steps_reduce_the_loss():
    """utils/train.py:149-158 in miniature: Adam + gradient clipping on the MSE of the predicted positions."""
    w = synth.WORKLOADS["water3d_10k"]
    host = synth.make_partitions(w, n_nodes=5000, seed=41)[0]
    sd = orc.init_state_dict(2, 0, 2, 64, 3, 4, seed=3, coord_gain=1.0)
    m = cuda_model(dict(node_feat_nf=2, node_attr_nf=0, edge_attr_nf=2, virtual_channels=3, n_layers=4), sd).train()
    inp = to_dev(host)
    target = inp["node_loc"] + 0.01 * inp["node_vel"] + 0.002
    opt = torch.optim.Adam(m.parameters(), lr=5e-4)
    losses = []
    for _ in range(12):
        opt.zero_grad()
        out, X = m(**inp)
        loss = torch.nn.functional.mse_loss(out, target)
        loss.backward()
        torch.nn.utils.clip_grad_norm_(m.parameters(), 0.3)
        opt.step()
        losses.append(float(loss))
    print("training losses", [f"{l:.3e}" for l in losses])
    assert losses[-1] < 0.7 * losses[0]


# ---- on-device graph construction (SURVEY §8 f-2) against scipy's cKDTree (the synthetic-data generator's own builder) ----
def _edge_set(ei):
    ei = ei.cpu().numpy()
    return set(zip(ei[0].tolist(), ei[1].tolist()))


@pytest.mark.gpu
@pytest.mark.parametrize("n,r,B,loop", [(20_000, 0.075, 1, False), (3_000, 0.2, 7, False), (500, 0.5, 3, True),
                                        (1, 0.1, 1, False)])
def test_radius_graph_matches_kdtree(n, r, B, loop):
    from scipy.spatial import cKDTree
    from distegnn_b200 import radius_graph
    rng = np.random.default_rng(5)
    side = synth.box_side(n, r, 15.0) if B == 1 else 2.0
    pos = rng.uniform(0, side, size=(n, 3)).astype(np.float32)
    batch = np.sort(rng.integers(0, B, size=n)).astype(np.int64)
    ref = set()
    for g in range(B):
        ids = np.nonzero(batch == g)[0]
        if len(ids) == 0:
            continue
        pairs = cKDTree(pos[ids].astype(np.float64)).query_pairs(r, output_type="ndarray")
        for i, j in pairs:
            ref.add((int(ids[i]), int(ids[j])))
            ref.add((int(ids[j]), int(ids[i])))
        if loop:
            ref.update((int(i), int(i)) for i in ids)
    ei, ea = radius_graph(torch.from_numpy(pos).to(dev()), r, None if B == 1 else torch.from_numpy(batch).to(dev()),
                          loop=loop, max_num_neighbors=n)
    mine = _edge_set(ei)
    # pairs whose length is within one fp32 ulp of r may fall on either side (cKDTree works in float64)
    d = np.linalg.norm(pos[ei[0].cpu().numpy()].astype(np.float64) - pos[ei[1].cpu().numpy()].astype(np.float64), axis=1)
    border = {e for e in (mine ^ ref) if abs(np.linalg.norm(pos[e[0]].astype(np.float64) - pos[e[1]].astype(np.float64)) - r) < 1e-6}
    assert (mine ^ ref) == border, (len(mine), len(ref), len(mine ^ ref))
    assert ei.shape[1] == len(mine)                                   # no duplicates
    assert bool((ei[0][1:] >= ei[0][:-1]).all())                      # grouped by destination row, ascending
    assert ea.shape == (ei.shape[1], 2) and float((ea[:, 0].cpu().double() - torch.from_numpy(d)).abs().max() if len(d) else 0.0) <= 1e-6
    print(f"radius_graph n={n} r={r} B={B} loop={loop}: {ei.shape[1]} edges, {len(border)} border pairs")


@pytest.mark.gpu
def test_radius_graph_feeds_the_model_like_the_host_built_graph():
    """Same model output whether the graph comes from the host builder (cKDTree) or from the device builder."""
    from distegnn_b200 import radius_graph
    w = synth.WORKLOADS["water3d_10k"]
    host = synth.make_partitions(w, n_nodes=8000, seed=3)[0]
    sd = orc.init_state_dict(2, 0, 2, 64, 3, 2, seed=4, coord_gain=0.05)
    m = cuda_model(dict(node_feat_nf=2, node_attr_nf=0, edge_attr_nf=2, virtual_channels=3, n_layers=2), sd)
    inp = to_dev(host)
    with torch.no_grad():
        out_h, X_h = m(**inp)
        ei, ea = radius_graph(inp["node_loc"], w.radius)
        assert ei.shape[1] == inp["edge_index"].shape[1]
        out_d, X_d = m(**{**inp, "edge_index": ei, "edge_attr": ea})
    assert max_abs(out_h, out_d) <= 2e-6 and max_abs(X_h, X_d) <= 2e-6


@pytest.mark.gpu
def test_training_path_gradients_batched_nbody():
    """BASELINE config 1 shape (N-body, fully connected, normalize=True) as a batch of graphs: tiles straddle graph
    boundaries in every kernel, forward and backward; gradients against float64 autograd through the oracle."""
    w = synth.WORKLOADS["nbody100"]
    nb, n = 12, 100
    parts = [synth.make_partitions(w, seed=50 + s)[0] for s in range(nb)]
    cat = lambda k: torch.cat([p[k] for p in parts])
    inp = dict(node_feat=cat("node_feat"), node_loc=cat("node_loc"), node_vel=cat("node_vel"), loc_mean=cat("loc_mean"),
               edge_index=torch.cat([p["edge_index"] + i * n for i, p in enumerate(parts)], 1),
               data_batch=torch.arange(nb).repeat_interleave(n), edge_attr=cat("edge_attr"), node_attr=None)
    sd = orc.init_state_dict(2, 0, 2, 64, 3, 4, seed=19, coord_gain=0.05)
    kw = dict(node_feat_nf=2, node_attr_nf=0, edge_attr_nf=2, virtual_channels=3, n_layers=4, normalize=True)
    g = torch.Generator().manual_seed(23)
    cot_out, cot_X = torch.randn(nb * n, 3, generator=g), torch.randn(nb, 3, 3, generator=g)
    sd64 = {k: v.double().requires_grad_(True) for k, v in sd.items()}
    inp64 = {k: (v.double() if (v is not None and v.is_floating_point()) else v) for k, v in inp.items()}
    o64, X64 = orc.forward(sd64, **inp64, normalize=True)
    keys = list(sd64)
    ref = dict(zip(keys, torch.autograd.grad((o64 * cot_out.double()).sum() + (X64 * cot_X.double()).sum(),
                                             [sd64[k] for k in keys], allow_unused=True)))
    ref = {k: (v if v is not None else torch.zeros_like(sd64[k])) for k, v in ref.items()}
    m = cuda_model(kw, sd).train()
    out, X = m(**to_dev(inp))
    ((out * cot_out.to(dev())).sum() + (X * cot_X.to(dev())).sum()).backward()
    errs, dead = _param_grad_errors(m, ref)
    worst = max(errs, key=errs.get)
    print(f"nbody batch {nb}x{n}: gradients vs oracle fp64 autograd: worst {worst} {errs[worst]:.2e}, "
          f"median {sorted(errs.values())[len(errs) // 2]:.2e}")
    assert errs[worst] <= 5e-4


@pytest.mark.gpu
def test_random_partitioner_on_device_matches_host_restatement():
    """split_large_graph_random (device) against the host restatement of distribute_graphs.py:17-51 in synth.py:
    same chunks from the same seed, same edge sets and edge lengths per partition, global loc_mean everywhere."""
    from distegnn_b200 import split_large_graph_random
    w = synth.WORKLOADS["fluid113k"]
    n, P, seed = 30_000, 4, 7
    pts = synth.make_points(w, seed, n)
    host = synth.make_partitions(w, world_size=P, split_mode="random", seed=seed, n_nodes=n)
    d = dev()
    t = lambda a: torch.from_numpy(a).to(d)
    parts = split_large_graph_random(t(pts["pos"]), t(pts["feat"]), t(pts["pos"]), t(pts["vel"]), t(pts["attr"]), w.radius, P,
                                     generator=torch.Generator().manual_seed(seed))
    assert len(parts) == P
    for mine, ref in zip(parts, host):
        assert torch.equal(mine["pos"].cpu(), ref["node_loc"]) and torch.equal(mine["x"].cpu(), ref["node_feat"])
        assert float((mine["loc_mean"].cpu() - ref["loc_mean"]).abs().max()) <= 1e-5
        a, b = _edge_set(mine["edge_index"]), _edge_set(ref["edge_index"])
        border = {e for e in (a ^ b)
                  if abs(float(np.linalg.norm(ref["node_loc"][e[0]].double().numpy() - ref["node_loc"][e[1]].double().numpy())) - w.radius) < 1e-6}
        assert (a ^ b) == border, (len(a), len(b))
        assert mine["edge_attr"].shape == (mine["edge_index"].shape[1], 2)


@pytest.mark.gpu
def test_shard_input_path_matches_edge_index_path(tmp_path):
    """SURVEY §8 f-4: the pre-sorted CSR shard (int32 ids, edge_attr in CSR order, pinned host memory) fed straight to the
    kernels — no radix sort, no permutation — gives the outputs of the int64 edge_index path."""
    from distegnn_b200.shards import read_shard, shard_from_forward_inputs, write_shard
    w = synth.WORKLOADS["fluid113k"]
    host = synth.make_partitions(w, n_nodes=20_000, seed=8)[0]
    sd = orc.init_state_dict(w.node_feat_nf, w.node_attr_nf, 2, 64, w.virtual_channels, 2, seed=6, coord_gain=0.05)
    m = cuda_model(dict(node_feat_nf=w.node_feat_nf, node_attr_nf=w.node_attr_nf, edge_attr_nf=2,
                        virtual_channels=w.virtual_channels, n_layers=2), sd)
    p = str(tmp_path / "part0.shard")
    write_shard(p, shard_from_forward_inputs(host))
    sh = read_shard(p).pinned()
    with torch.no_grad():
        out_a, X_a = m(**to_dev(host))
        builds = m._graphs.builds
        out_b, X_b = m(**sh.to(dev()))
        assert m._graphs.builds == builds                    # nothing was sorted for the shard
    torch.cuda.synchronize()
    assert max_abs(out_a, out_b) <= 2e-6 and max_abs(X_a, X_b) <= 2e-6
    print(f"shard: {sh.nbytes() / 2**20:.1f} MiB on the wire vs "
          f"{sum(v.numel() * v.element_size() for v in host.values() if v is not None) / 2**20:.1f} MiB for the tensors of the reference API")


# ---- virtual-node sync: the library's own exchange (csrc/comm.cuh) -------------------------------------------------------
def _solo_comm(max_slots, slot_floats):
    """A communicator of world size 1 on this process' GPU: the same kernel path (push, flag, wait, ordered reduce),
    with the only 'peer' being the rank itself — what a single-GPU box can exercise of the collective."""
    import ctypes as C
    lib = _lib.load()
    nb = lib.distegnn_comm_handle_bytes()
    mine = (C.c_ubyte * nb)()
    h = C.c_void_p()
    _lib.check(lib.distegnn_comm_init(0, 1, max_slots, slot_floats, C.byref(h), mine), "comm_init")
    _lib.check(lib.distegnn_comm_connect(h, mine), "comm_connect")

    class Solo:
        handle = h

        @staticmethod
        def status():
            v = C.c_int(0)
            _lib.check(lib.distegnn_comm_status(h, C.byref(v)), "comm_status")
            return v.value

        @staticmethod
        def destroy():
            lib.distegnn_comm_destroy(h)
    return Solo


@pytest.mark.gpu
def test_packed_allreduce_single_rank_is_identity_and_replayable():
    from distegnn_b200.backend import cuda_backend
    be = cuda_backend()
    comm = _solo_comm(max_slots=5, slot_floats=540)
    try:
        g = torch.Generator().manual_seed(0)
        for n in (1, 540, 541, 5 * 540):                         # partial slot, one slot, two slots, full capacity
            buf = torch.randn(n, generator=g).to(dev())
            want = buf.clone()
            for _ in range(3):                                   # epochs advance, parity double-buffer flips
                be.allreduce_packed(comm, buf)
            torch.cuda.synchronize()
            assert torch.equal(buf, want)
        with pytest.raises(ValueError, match="capacity"):
            be.allreduce_packed(comm, torch.zeros(5 * 540 + 1, device=dev()))
        # under CUDA-graph capture: the per-slot epoch lives in device memory, so replays stay consistent
        buf = torch.randn(700, generator=g).to(dev())
        want = buf.clone()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            be.allreduce_packed(comm, buf)
        torch.cuda.current_stream().wait_stream(side)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            be.allreduce_packed(comm, buf)
        for _ in range(4):
            graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(buf, want) and comm.status() == 0
    finally:
        torch.cuda.synchronize()
        comm.destroy()


@pytest.mark.gpu
@pytest.mark.parametrize("C,B", [(8, 1), (5, 3), (16, 2)])
def test_fused_sync_update_equals_plain_update(C, B):
    """virtual_update with a communicator (all-reduce inside the kernel) == without, on one rank; FLAG_ZERO_VSUM clears the
    statistics, without it the (summed) statistics stay in vsum; the INIT flavour initialises Xv / Hv itself."""
    from distegnn_b200.backend import cuda_backend
    be = cuda_backend()
    A, Na = 2, 0
    K = 4 + 3 * C + 64 * C
    sd = orc.init_state_dict(2, Na, A, 64, C, 2, seed=4, coord_gain=1.0)
    m = cuda_model(dict(node_feat_nf=2, node_attr_nf=Na, edge_attr_nf=A, virtual_channels=C, n_layers=2), sd)
    pk = m._packed_params(dev())
    g = torch.Generator().manual_seed(1)
    vs = torch.randn(B, K, generator=g).to(dev())
    vs[:, 3] = torch.tensor([1000.0 + 7 * b for b in range(B)])
    loc_mean = torch.randn(B, 3, generator=g).to(dev())
    comm = _solo_comm(max_slots=B, slot_floats=K)
    try:
        res = {}
        for tag, cm, zero in (("plain", None, 0), ("fused", comm, 0), ("fused_zero", comm, _lib.FLAG_ZERO_VSUM)):
            v = vs.clone()
            Xv, Hv, G = (torch.full((B, 3, C), 7.0, device=dev()), torch.full((B, C, 64), 7.0, device=dev()),
                         torch.empty(B, C, 64, device=dev()))
            be.virtual_update((B, A, C, Na), _lib.FLAG_INIT | zero, v, Xv, Hv, None, pk["layers"][0], G,
                              loc_mean, pk["hv0"], cm)
            v0 = v.clone()
            v.copy_(vs)
            be.virtual_update((B, A, C, Na), zero, v, Xv, Hv, pk["layers"][0], pk["layers"][1], G, comm=cm)
            torch.cuda.synchronize()
            res[tag] = (Xv, Hv, G, v0, v.clone())
        for tag in ("fused", "fused_zero"):
            for a, b in zip(res[tag][:3], res["plain"][:3]):
                assert torch.equal(a, b), tag
        assert torch.equal(res["fused"][4], vs) and torch.equal(res["plain"][4], vs)
        assert float(res["fused_zero"][3].abs().max()) == 0.0 and float(res["fused_zero"][4].abs().max()) == 0.0
        # the INIT flavour wrote Xv = loc_mean per channel and Hv = virtual_node_feat before updating
        Xv0 = torch.empty(B, 3, C, device=dev())
        Hv0 = torch.empty(B, C, 64, device=dev())
        G0 = torch.empty(B, C, 64, device=dev())
        be.virtual_update((B, A, C, Na), _lib.FLAG_INIT, vs.clone(), Xv0, Hv0, None, pk["layers"][0], G0, loc_mean, pk["hv0"])
        torch.cuda.synchronize()
        assert torch.equal(Xv0, loc_mean.unsqueeze(-1).expand(B, 3, C)) and torch.equal(Hv0, pk["hv0"].expand(B, C, 64))
        assert comm.status() == 0
    finally:
        torch.cuda.synchronize()
        comm.destroy()


@pytest.mark.gpu
def test_forward_leaves_accumulators_clean_and_launches_only_kernels():
    """No memset / copy launches in steady state: the consumers clear vsum / agg_m / agg_x (FLAG_ZERO_*), so after every
    forward the workspace accumulators are zero again and back-to-back forwards agree; a forward is 2 + 4L launches."""
    from distegnn_b200.backend import cuda_backend
    w = synth.WORKLOADS["fluid113k"]
    inp = to_dev(synth.make_partitions(w, n_nodes=20_011, seed=5)[0])
    sd = orc.init_state_dict(3, 2, 2, 64, 5, 4, seed=2, coord_gain=0.05)
    m = cuda_model(dict(node_feat_nf=3, node_attr_nf=2, edge_attr_nf=2, virtual_channels=5, n_layers=4), sd)
    be = cuda_backend()
    with torch.no_grad():
        o1, X1 = m(**inp)
        n0 = be.launches
        o2, X2 = m(**inp)
        assert be.launches - n0 == 2 + 4 * 4
        torch.cuda.synchronize()
        ws = next(iter(m._workspaces.values()))
        for k in ("vsum", "agg_m", "agg_x"):
            assert float(ws[k].abs().max()) == 0.0, k
        assert not ws["dirty"]
        assert max_abs(o1, o2) <= 2e-6 and max_abs(X1, X2) <= 2e-6
        assert o1.data_ptr() != o2.data_ptr()                  # results are fresh tensors, not workspace views
    ref, refX = oracle64(sd, {k: (v.cpu() if v is not None else None) for k, v in inp.items()}, False)
    check_close(o2, X2, ref, refX, inp["node_loc"].cpu(), "self-cleaning workspace")


@pytest.mark.gpu
def test_validation_on_device():
    """Bad data_batch / edge ids are caught by the device-side counters (embed / CSR build) and raise."""
    inp = to_dev(synth.make_partitions(synth.WORKLOADS["water3d_10k"], n_nodes=3_000, seed=9)[0])
    sd = orc.init_state_dict(2, 0, 2, 64, 3, 2, seed=0)
    m = cuda_model(dict(node_feat_nf=2, node_attr_nf=0, edge_attr_nf=2, virtual_channels=3, n_layers=2), sd)
    with torch.no_grad():
        good, _ = m(**inp)
        b = inp["data_batch"].clone()
        b[100] = 1
        with pytest.raises(ValueError, match="data_batch"):
            m(**dict(inp, data_batch=b))
        ei = inp["edge_index"].clone()
        ei[0, 5] = inp["node_loc"].shape[0]
        with pytest.raises(ValueError, match="edge_index"):
            m(**dict(inp, edge_index=ei))
        again, _ = m(**inp)                                      # dirty workspace after the failures is re-zeroed
        assert max_abs(good, again) <= 2e-6


@pytest.mark.gpu
@pytest.mark.parametrize("split_mode,extra", [("random", ["--cuda-graph", "--grads", "--nodes", "12000"]),
                                               ("kmeans", ["--nodes", "30000"])])
def test_multi_gpu_parity_under_torchrun(split_mode, extra):
    """2 ranks (2 GPUs) under torchrun: every rank's CUDA path + the peer-memory exchange vs the partitioned float64
    oracle (oracle/dist_check.py).  Skipped on a single-GPU box — bench.py runs the same check under the driver's
    multi-GPU launches and puts it into its JSON line (`dist_parity`)."""
    import subprocess
    import sys
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 CUDA devices")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", "29541", os.path.join(root, "scripts", "dist_parity.py"), "--workload",
           "fluid113k", "--split-mode", split_mode, *extra]
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=root)
    print(p.stdout[-3000:], p.stderr[-1500:])
    assert p.returncode == 0 and "DIST_PARITY PASS" in p.stdout


@pytest.mark.gpu
def test_tma_gather4_building_block():
    """cp.async.bulk.tensor.2d ...tile::gather4 through a tensor map whose box (72 floats) is wider than the row (64):
    four rows per instruction land at a pitch of 72 floats with a zero-filled tail — the padded staging layout of the edge
    kernel — and out-of-range row coordinates come back as zeros instead of faulting."""
    from tests.twin_backend import check, load_testing
    lib = load_testing()
    g = torch.Generator().manual_seed(0)
    n_rows, groups = 1000, 5
    src = torch.randn(n_rows, 64, generator=g).to(dev())
    idx = torch.randint(0, n_rows, (4 * groups,), generator=g, dtype=torch.int32)
    idx[5], idx[6] = n_rows + 3, -2                                  # out of bounds -> zeros
    idx_d = idx.to(dev())
    out = torch.empty(groups, 4, 72, device=dev())
    check(lib.distegnn_selftest_gather4(src.data_ptr(), n_rows, idx_d.data_ptr(), groups, 72, 1, out.data_ptr(),
                                        torch.cuda.current_stream().cuda_stream), "selftest_gather4")
    torch.cuda.synchronize()
    want = torch.zeros(groups * 4, 72, device=dev())
    ok = (idx_d >= 0) & (idx_d < n_rows)
    want[ok, :64] = src[idx_d[ok].long()]
    assert torch.equal(out.reshape(groups * 4, 72), want)


# ---- f-2: graph construction and partitioning on the device, CSR out ---------------------------------------------------
def _csr_edge_set(g, ea=None):
    E = g.num_edges if g.n_edges_dev is None else int(g.n_edges_dev.item())
    row, col = g.rows()[:E].cpu().numpy().astype(np.int64), g.col[:E].cpu().numpy().astype(np.int64)
    return set(zip(row.tolist(), col.tolist())), E


@pytest.mark.gpu
@pytest.mark.parametrize("n,r,B,loop", [(5000, 0.075, 1, False), (3000, 0.1, 3, False), (400, 0.3, 2, True), (1, 0.5, 1, False)])
def test_radius_graph_csr_matches_kdtree(n, r, B, loop):
    """One C-ABI call, everything decided on the device: same edge set as scipy's cKDTree (pairs within one fp32 ulp of r
    excepted), rows ascending (a valid CSR), edge_attr = the edge length in every column; capacity mode = same graph
    without any host synchronisation."""
    from scipy.spatial import cKDTree
    from distegnn_b200.partition import radius_graph_csr
    rng = np.random.default_rng(7)
    pos = rng.uniform(0, 1.0, size=(n, 3)).astype(np.float32)
    batch = np.sort(rng.integers(0, B, size=n)).astype(np.int64)
    batch[0], batch[-1] = 0, B - 1
    want, near = set(), set()
    for b in range(B):
        idx = np.nonzero(batch == b)[0]
        if len(idx) == 0:
            continue
        t = cKDTree(pos[idx].astype(np.float64))
        for i, j in t.query_pairs(r * (1 + 1e-6), output_type="ndarray"):
            d = float(np.linalg.norm(pos[idx[i]].astype(np.float64) - pos[idx[j]].astype(np.float64)))
            pair = {(int(idx[i]), int(idx[j])), (int(idx[j]), int(idx[i]))}
            (near if abs(d - r) <= 2e-7 * max(r, 1.0) else want).update(pair) if d < r * (1 + 1e-6) else None
        if loop:
            want.update((int(i), int(i)) for i in idx)
    pd, bd = torch.from_numpy(pos).to(dev()), (torch.from_numpy(batch).to(dev()) if B > 1 else None)
    g, ea = radius_graph_csr(pd, r, bd, loop=loop)
    got, E = _csr_edge_set(g)
    assert len(got) == E, "duplicate edges"
    assert want - near <= got <= want | near
    g.validate(dev())                                          # monotone rowptr ending at E, columns in range
    if E:
        rows, cols = g.rows().long(), g.col.long()
        d = (pd[rows] - pd[cols]).norm(dim=1)
        assert float((ea[:, 0] - d).abs().max()) <= 1e-6 and torch.equal(ea[:, 0], ea[:, 1])
    gc, eac = radius_graph_csr(pd, r, bd, loop=loop, capacity=E + 100, n_graphs=B)
    assert gc.n_edges_dev is not None and not gc.overflowed() and int(gc.n_edges_dev.item()) == E
    assert torch.equal(gc.rowptr, g.rowptr) and torch.equal(gc.col[:E], g.col) and torch.equal(eac[:E], ea)
    if E > 10:
        small, _ = radius_graph_csr(pd, r, bd, loop=loop, capacity=E // 2, n_graphs=B)
        assert small.overflowed()


@pytest.mark.gpu
def test_device_built_graph_feeds_the_model_without_host_sync():
    """Rollout shape: positions change every step, the graph is rebuilt on the device with a capacity (no host read of the
    edge count), the model reads the count on the device: same outputs as the host-built int64 edge_index path."""
    from distegnn_b200.partition import radius_graph_csr
    w = synth.WORKLOADS["fluid113k"]
    inp = to_dev(synth.make_partitions(w, n_nodes=20_000, seed=3)[0])
    sd = orc.init_state_dict(3, 2, 2, 64, 5, 4, seed=1, coord_gain=0.05)
    m = cuda_model(dict(node_feat_nf=3, node_attr_nf=2, edge_attr_nf=2, virtual_channels=5, n_layers=4), sd)
    node = {k: v for k, v in inp.items() if k not in ("edge_index", "edge_attr")}
    with torch.no_grad():
        ref, refX = m(**inp)
        cap = int(inp["edge_index"].shape[1] * 1.3)
        m(**node, **dict(zip(("edge_index", "edge_attr"), radius_graph_csr(inp["node_loc"], w.radius, capacity=cap))))   # warm-up
        torch.cuda.synchronize()
        pos = inp["node_loc"].clone()
        outs = []
        # the loop below must not synchronise: torch would raise on .item()/.cpu() under this guard
        with torch.cuda.StreamContext(torch.cuda.current_stream()):
            torch.cuda.set_sync_debug_mode("error")
            try:
                for step in range(3):
                    g, ea = radius_graph_csr(pos, w.radius, capacity=cap)
                    out, X = m(**dict(node, node_loc=pos), edge_index=g, edge_attr=ea)
                    outs.append(out)
                    pos = out                                  # next step starts from the predicted positions
            finally:
                torch.cuda.set_sync_debug_mode("default")
        torch.cuda.synchronize()
    assert max_abs(outs[0], ref) <= 2e-6 and not g.overflowed()
    # step 2 against the reference path on the same positions
    with torch.no_grad():
        from distegnn_b200 import radius_graph
        ei, ea2 = radius_graph(outs[0], w.radius)
        want, _ = m(**dict(node, node_loc=outs[0]), edge_index=ei, edge_attr=ea2)
    assert max_abs(outs[1], want) <= 5e-6


@pytest.mark.gpu
@pytest.mark.parametrize("n,P", [(30_000, 8), (113_140, 8), (20_000, 2)])
def test_kmeans_on_device_matches_sklearn(n, P):
    """Lloyd iterations on the device from sklearn's own k-means++ seeding: label agreement with
    KMeans(n_clusters=P, random_state=0, n_init='auto').fit_predict (distribute_graphs.py:188-198)."""
    from sklearn.cluster import KMeans
    from distegnn_b200.partition import kmeans_labels
    w = synth.WORKLOADS["fluid113k"]
    pos = synth.make_points(w, seed=4, n_nodes=n)["pos"]
    want = KMeans(n_clusters=P, random_state=0, n_init="auto").fit_predict(pos.astype(np.float32))
    got = kmeans_labels(torch.from_numpy(pos).to(dev()), P).cpu().numpy()
    agree = float((got == want).mean())
    print(f"k-means n={n} P={P}: label agreement with sklearn {agree:.6f}, cluster sizes {np.bincount(got, minlength=P).tolist()}")
    assert agree >= 0.999


@pytest.mark.gpu
def test_split_large_graph_on_device_kmeans_and_random():
    """The device partitioner (k-means / random chunks + per-chunk CSR radius graphs) gives the same partitions as the host
    restatement of distribute_graphs.py, and the model accepts them as they are."""
    from distegnn_b200.partition import split_large_graph
    w = synth.WORKLOADS["fluid113k"]
    n, P = 24_000, 4
    pts = synth.make_points(w, seed=6, n_nodes=n)
    d = dev()
    pos, vel = torch.from_numpy(pts["pos"]).to(d), torch.from_numpy(pts["vel"]).to(d)
    feat, attr = torch.from_numpy(pts["feat"]).to(d), torch.from_numpy(pts["attr"]).to(d)
    for mode in ("kmeans", "random"):
        host = synth.make_partitions(w, world_size=P, split_mode=mode, seed=6, n_nodes=n)
        mine = split_large_graph(pos, feat, pos + 0.01 * vel, vel, attr, w.radius, P, split_mode=mode,
                                 generator=torch.Generator().manual_seed(6))
        for r in range(P):
            assert torch.equal(mine[r]["pos"].cpu(), host[r]["node_loc"]), (mode, r)
            he = set(zip(host[r]["edge_index"][0].tolist(), host[r]["edge_index"][1].tolist()))
            ge, E = _csr_edge_set(mine[r]["edge_index"])
            assert len(ge ^ he) <= max(2, int(2e-5 * len(he))), (mode, r, len(ge ^ he))     # pairs within an ulp of r


# ---- f-1: backward of the per-node stage and of the embedding prologue (csrc/node_layer_bwd.cu) ---------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("Na,last,N", [(2, False, 5_003), (0, False, 300), (2, True, 1_111), (0, False, 128)])
def test_node_stage_backward(Na, last, N):
    """distegnn_node_layer_bwd against float64 autograd through the stage's torch restatement (tests/shadow_backend.py):
    every data gradient and every parameter-gradient field, isolated nodes and a ragged last tile included."""
    from distegnn_b200.backend import cuda_backend
    be, sh = cuda_backend(), ShadowBackend()
    A, C, B = 2, 3, 2
    g = torch.Generator().manual_seed(N + Na)
    sd = orc.init_state_dict(3, Na, A, 64, C, 2, seed=2, coord_gain=1.0)
    m = cuda_model(dict(node_feat_nf=3, node_attr_nf=Na, edge_attr_nf=A, virtual_channels=C, n_layers=2), sd)
    pk = m._packed_params(dev())
    lp, lpn = pk["layers"][0], pk["layers"][1]
    K = 4 + 3 * C + 64 * C
    rnd = lambda *s: torch.randn(*s, generator=g)
    deg = torch.randint(0, 6, (N,), generator=g)
    rowptr = torch.zeros(N + 1, dtype=torch.int32)
    rowptr[1:] = torch.cumsum(deg, 0).to(torch.int32)
    batch32 = torch.sort(torch.randint(0, B, (N,), generator=g)).values.to(torch.int32)
    t = dict(h=rnd(N, 64), vel=rnd(N, 3), attr=rnd(N, Na) if Na else None, agg_m=rnd(N, 64) * 3, agg_v=rnd(N, 64),
             g_x=rnd(N, 3), g_vsum=rnd(B, K), g_h=rnd(N, 64), g_P=rnd(N, 64), g_Q=rnd(N, 64), g_Hn=rnd(N, 64))
    flags = _lib.FLAG_LAST if last else 0
    total = lp.numel()

    def run(backend, dt, device):
        c = lambda v: None if v is None else v.to(device=device, dtype=dt)
        o = dict(g_h=torch.empty(N, 64, dtype=dt, device=device), g_x=torch.empty(N, 3, dtype=dt, device=device),
                 g_agg_x=torch.empty(N, 4, dtype=dt, device=device), g_trans_v=torch.empty(N, 4, dtype=dt, device=device),
                 g_agg_m=torch.zeros(N, 64, dtype=dt, device=device), g_agg_v=torch.zeros(N, 64, dtype=dt, device=device),
                 g_lp=torch.zeros(total, dtype=dt, device=device), g_lpn=torch.zeros(total, dtype=dt, device=device))
        backend.node_layer_bwd((N, B, A, C, Na), flags, rowptr.to(device), batch32.to(device), c(t["h"]), c(t["vel"]),
                               c(t["attr"]), None if last else c(t["agg_m"]), None if last else c(t["agg_v"]),
                               lp.to(device=device, dtype=dt), None if last else lpn.to(device=device, dtype=dt),
                               c(t["g_x"]), c(t["g_vsum"]), None if last else c(t["g_h"]), None if last else c(t["g_P"]),
                               None if last else c(t["g_Q"]), None if last else c(t["g_Hn"]), o["g_h"], o["g_x"],
                               o["g_agg_x"], o["g_trans_v"], None if last else o["g_agg_m"], None if last else o["g_agg_v"],
                               o["g_lp"], None if last else o["g_lpn"])
        return o
    got = run(be, torch.float32, dev())
    torch.cuda.synchronize()
    want = run(sh, torch.float64, torch.device("cpu"))
    worst = {}
    for k in want:
        a_, b_ = got[k].cpu().double(), want[k]
        if k in ("g_agg_x", "g_trans_v"):
            a_, b_ = a_[:, :3], b_[:, :3]
        den = float(b_.abs().max())
        if den == 0.0:
            assert float(a_.abs().max()) == 0.0, k
            continue
        worst[k] = float((a_ - b_).abs().max()) / den
        assert worst[k] <= 2e-5, (k, worst[k])
    print(f"node stage backward Na={Na} last={last} N={N}: " + ", ".join(f"{k} {v:.1e}" for k, v in worst.items()))


@pytest.mark.gpu
@pytest.mark.parametrize("F,N", [(3, 4_001), (1, 77), (16, 1_000)])
def test_embed_backward(F, N):
    from distegnn_b200.backend import cuda_backend
    be, sh = cuda_backend(), ShadowBackend()
    A, C, Na, B = 2, 5, 0, 1
    g = torch.Generator().manual_seed(F)
    sd = orc.init_state_dict(F, Na, A, 64, C, 1, seed=3)
    m = cuda_model(dict(node_feat_nf=F, node_attr_nf=Na, edge_attr_nf=A, virtual_channels=C, n_layers=1), sd)
    lp0 = m._packed_params(dev())["layers"][0]
    feat, h0 = torch.randn(N, F, generator=g), torch.randn(N, 64, generator=g)
    gs = [torch.randn(N, 64, generator=g) for _ in range(4)]

    def run(backend, dt, device):
        c = lambda v: v.to(device=device, dtype=dt)
        o = (torch.zeros(F, 64, dtype=dt, device=device), torch.zeros(64, dtype=dt, device=device),
             torch.zeros(lp0.numel(), dtype=dt, device=device))
        backend.embed_bwd((N, B, F, A, C, Na), c(feat), c(h0), c(lp0), *[c(x) for x in gs], *o)
        return o
    got = run(be, torch.float32, dev())
    torch.cuda.synchronize()
    want = run(sh, torch.float64, torch.device("cpu"))
    for a_, b_, name in zip(got, want, ("g_emb_wt", "g_emb_b", "g_lp0")):
        e = float((a_.cpu().double() - b_).abs().max() / b_.abs().max())
        print(f"embed backward F={F} N={N} {name}: rel err {e:.1e}")
        assert e <= 2e-5


@pytest.mark.gpu
@pytest.mark.parametrize("C,B,mode", [(8, 1, "mid"), (5, 3, "mid"), (3, 2, "last"), (16, 2, "init"), (1, 4, "mid")])
def test_virtual_update_backward(C, B, mode):
    """distegnn_virtual_update_bwd against float64 autograd through the stage's torch restatement."""
    from distegnn_b200.backend import cuda_backend
    be, sh = cuda_backend(), ShadowBackend()
    A, Na = 2, 0
    K = 4 + 3 * C + 64 * C
    g = torch.Generator().manual_seed(C * 10 + B)
    sd = orc.init_state_dict(2, Na, A, 64, C, 2, seed=6, coord_gain=1.0)
    m = cuda_model(dict(node_feat_nf=2, node_attr_nf=Na, edge_attr_nf=A, virtual_channels=C, n_layers=2), sd)
    pk = m._packed_params(dev())
    lp, lpn = pk["layers"][0], pk["layers"][1]
    flags = {"mid": 0, "last": _lib.FLAG_LAST, "init": _lib.FLAG_INIT}[mode]
    vs = torch.randn(B, K, generator=g)
    vs[:, 3] = torch.tensor([500.0 + 13 * b for b in range(B)])
    t = dict(vs=vs, Xv=torch.randn(B, 3, C, generator=g), Hv=torch.randn(B, C, 64, generator=g),
             gX=torch.randn(B, 3, C, generator=g), gH=torch.randn(B, C, 64, generator=g), gG=torch.randn(B, C, 64, generator=g))
    last, init = mode == "last", mode == "init"

    def run(backend, dt, device):
        c = lambda v: v.to(device=device, dtype=dt)
        o = dict(g_vsum=torch.zeros(B, K, dtype=dt, device=device), g_Xv=torch.zeros(B, 3, C, dtype=dt, device=device),
                 g_Hv=torch.zeros(B, C, 64, dtype=dt, device=device), g_lp=torch.zeros(lp.numel(), dtype=dt, device=device),
                 g_lpn=torch.zeros(lp.numel(), dtype=dt, device=device))
        backend.virtual_update_bwd((B, A, C, Na), flags, c(t["vs"]), c(t["Xv"]), c(t["Hv"]), None if init else c(lp),
                                   None if last else c(lpn), c(t["gX"]), None if last else c(t["gH"]),
                                   None if last else c(t["gG"]), o["g_vsum"], o["g_Xv"], None if last else o["g_Hv"],
                                   None if init else o["g_lp"], None if last else o["g_lpn"])
        return o
    got = run(be, torch.float32, dev())
    torch.cuda.synchronize()
    want = run(sh, torch.float64, torch.device("cpu"))
    worst = {}
    for k in want:
        a_, b_ = got[k].cpu().double(), want[k]
        den = float(b_.abs().max())
        if den == 0.0:
            assert float(a_.abs().max()) == 0.0, k
            continue
        worst[k] = float((a_ - b_).abs().max()) / den
        assert worst[k] <= 2e-5, (k, worst[k])
    print(f"virtual update backward C={C} B={B} {mode}: " + ", ".join(f"{k} {v:.1e}" for k, v in worst.items()))
