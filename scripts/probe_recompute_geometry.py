"""Apply time of the default operator against the PMGX_LAP_RECOMPUTE_G operator, P1..P8, ~100 M dofs.

On a perturbed box (perturb 0.15: the default runs the streamed-G kernel) and on the uniform box (the default
runs the affine kernel, except at P8).  CUDA events, 3 warm-up and 20 timed applies per round, the two operators
alternated over 2 rounds.  One JSON line per (degree, mesh) on stdout, card name and power limit first.

    python scripts/probe_recompute_geometry.py [ndofs] [degrees] [rounds]
"""
import json
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, ".")
from pmg_dolfinx_b200 import api  # noqa: E402

RECOMPUTE = 8
WARMUP, REPS = 3, 20


def bytes_recompute(P, ncells, ndofs):
    """The recompute kernel's byte model: encoded dofmap 4 B per cell dof, 32 B of geometry dofmap and <= 192 B
    of vertex reads per cell, kappa and perm (12 B per cell), 17 B per dof (x read, y read-modify-write, bc)."""
    return ncells * ((P + 1) ** 3 * 4 + 32 + 192 + 12) + ndofs * 17


def flops_per_point(P, recompute):
    """FP64 operations per quadrature point: the sum-factorised apply (3 forward and 3 transposed contractions of
    length n = P + 1, 2 flops each; the 3x3 flux product with kappa), plus, when G is recomputed, the Jacobian
    from the factored form (6 FMAs), adj(J) (9 x 3), det J (5), the reciprocal (counted as 8) and G = s K K^T
    (6 x 5 + 1)."""
    n = P + 1
    apply = 12 * n + 21
    geometry = 12 + 27 + 5 + 8 + 31
    return apply + (geometry if recompute else 0)


def card():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        pl = "unknown"
    return name, pl


def time_applies(ctx, op, x, y):
    for _ in range(WARMUP):
        op(x, y)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(ctx.stream)
    for _ in range(REPS):
        op(x, y)
    e1.record(ctx.stream)
    ctx.sync()
    return e0.elapsed_time(e1) / REPS


def run(ctx, P, ndofs, perturb, rounds):
    n = api.boxmesh_fit(ndofs, P)
    m = api.BoxMesh(n, perturb=perturb)
    sp = m.space(P)
    d_dm, d_x, d_g = ctx.to_device(sp.dofmap), ctx.to_device(m.xgeom), ctx.to_device(m.geom_dofmap)
    d_k = torch.full((m.n_cells,), 2.0, dtype=torch.float64, device=ctx.device)
    d_bc = ctx.to_device(sp.bc)
    ops = {name: api.MatFreeLaplacian(ctx, P, d_k, d_dm, d_x, d_g, m.lcells, m.bcells, d_bc, sp.n_owned, 0, None,
                                      flags)
           for name, flags in (("default", 0), ("recompute", RECOMPUTE))}
    x, y = api.Vector(ctx, sp.n_owned), api.Vector(ctx, sp.n_owned)
    x.copy_from_host(np.random.default_rng(1).uniform(-1, 1, sp.n_owned))
    ys = {}
    for name, op in ops.items():
        op(x, y)
        ys[name] = y.data_copy()
    diff = float(np.abs(ys["recompute"] - ys["default"]).max() / np.abs(ys["default"]).max())
    ms = {name: [] for name in ops}
    for _ in range(rounds):
        for name, op in ops.items():
            ms[name].append(time_applies(ctx, op, x, y))
    npts = m.n_cells * (P + 1) ** 3
    t_r = min(ms["recompute"])
    out = dict(P=P, perturb=perturb, n=list(n), ndofs=sp.n_owned, cells=m.n_cells,
               kernel={k: op.kernel_name() for k, op in ops.items()},
               ms={k: [round(v, 4) for v in vs] for k, vs in ms.items()},
               gdofs={k: round(sp.n_owned / min(vs) / 1e6, 2) for k, vs in ms.items()},
               recompute_model_GBs=round(bytes_recompute(P, m.n_cells, sp.n_owned) / t_r / 1e6, 1),
               recompute_TFLOPs=round(npts * flops_per_point(P, True) / t_r / 1e9, 2),
               default_TFLOPs=round(npts * flops_per_point(P, False) / min(ms["default"]) / 1e9, 2),
               device_bytes={k: op.device_bytes() for k, op in ops.items()},
               max_rel_diff=diff)
    print(json.dumps(out), flush=True)
    for op in ops.values():
        op.destroy()
    del d_dm, d_x, d_g, d_k, d_bc, x, y
    torch.cuda.empty_cache()


if __name__ == "__main__":
    nd = int(float(sys.argv[1])) if len(sys.argv) > 1 else 100_000_000
    degs = [int(a) for a in sys.argv[2].split(",")] if len(sys.argv) > 2 else list(range(1, 9))
    rounds = int(sys.argv[3]) if len(sys.argv) > 3 else 2
    ctx = api.Context(0)
    name, pl = card()
    print(json.dumps(dict(card=name, power_limit=pl, warmup=WARMUP, reps=REPS, rounds=rounds)), flush=True)
    for P in degs:
        for perturb in (0.15, 0.0):
            run(ctx, P, nd, perturb, rounds)
