"""Shared helpers for the test-suite (fixtures loader, error metrics)."""
from __future__ import annotations

import ast
import hashlib
import os

import numpy as np
import torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
SINGLE_CASES = ["nbody24_norm", "fluid160_c5", "batch3_c8_multigraph"]
DIST_CASE = "dist2_fluid300_c5"
INPUT_KEYS = ["node_feat", "node_loc", "node_vel", "loc_mean", "edge_index", "data_batch", "edge_attr",
              "node_attr"]
MAX_FIXTURE_BYTES = 1_000_000       # size limit of one file under tests/golden/


def tensor_digest(t) -> str:
    a = np.ascontiguousarray(t.numpy() if isinstance(t, torch.Tensor) else t)
    return hashlib.sha256(f"{a.dtype.str}{a.shape}".encode() + a.tobytes()).hexdigest()


def load_golden(name):
    z = np.load(os.path.join(GOLDEN, name + ".npz"))
    kw = ast.literal_eval(str(z["meta.kw"]))
    sd = {k[3:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("sd.")}
    if not sd:
        sd = seeded_weights(z, kw)
    return z, kw, sd


def seeded_weights(z, kw):
    """Weights of a fixture that stores them as the seed of the reference's own init plus a sha256 per tensor (the
    full 4-layer weights would not fit MAX_FIXTURE_BYTES): the package's constructor under that seed reproduces the
    reference's init bit for bit, and every tensor is checked against its digest."""
    from distegnn_b200 import FastEGNN
    with torch.random.fork_rng(devices=[]):
        torch.manual_seed(int(z["meta.seed"]))
        sd = FastEGNN(hidden_nf=64, world_size=1, **kw).state_dict()
    want = {k[len("sdsha."):]: str(z[k]) for k in z.files if k.startswith("sdsha.")}
    assert list(sd) == list(want), "state_dict keys differ from the fixture's"
    bad = [k for k in sd if tensor_digest(sd[k]) != want[k]]
    assert not bad, f"seeded init no longer reproduces the fixture's weights: {bad}"
    return sd


def grad_sample(zg, key):
    """Flat indices of the entries a gradient fixture stores under `key`, or None if it stores all of them.  A fixture
    that would exceed MAX_FIXTURE_BYTES keeps a seeded sample of each large gradient; the sample includes the entry of
    largest magnitude, so a max-norm relative error over the sample has the whole tensor's denominator."""
    return torch.from_numpy(zg["idx." + key]).long() if "idx." + key in zg.files else None


def golden_inputs(z, prefix="in."):
    d = {k: (torch.from_numpy(z[prefix + k]) if prefix + k in z.files else None) for k in INPUT_KEYS}
    return d


def golden_trace(z, key, prefix="trace."):
    out, i = [], 0
    while f"{prefix}{key}.{i}" in z.files:
        out.append(torch.from_numpy(z[f"{prefix}{key}.{i}"]))
        i += 1
    return out


def max_abs(a, b):
    return float((a.double() - b.double()).abs().max()) if a.numel() else 0.0


def rel_disp_err(out, ref, pos):
    """‖(out−pos)−(ref−pos)‖∞ / ‖ref−pos‖∞ — parity on the *displacement*, which is what the model
    actually computes (SURVEY §7 'parity is deceptively easy at init')."""
    den = float((ref.double() - pos.double()).abs().max())
    return max_abs(out, ref) / max(den, 1e-30)
