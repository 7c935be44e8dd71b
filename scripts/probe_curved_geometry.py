"""Create time, apply time and device memory of a perturbed-trilinear (8-node) against a curved (27-node,
PMGX_LAP_GEOM_Q2) operator on the same box topology, ~100 M dofs per degree.

The 8-node mesh is the box with its interior vertices perturbed by 0.15 h; the 27-node mesh is the annular sector
of tests/curved_reference.py.  Both run the streamed-G kernel, so their applies should take the same time.  Create
is timed with a host clock around pmgx_laplacian_create (which ends in a device synchronise), inputs already on the
device; applies with CUDA events, 3 warm-up and 20 timed applies per round, the two operators alternated over
`rounds` rounds.  One JSON line per degree on stdout, card name and power limit first.

    python scripts/probe_curved_geometry.py [ndofs] [degrees] [rounds]
"""
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from pmg_dolfinx_b200 import api  # noqa: E402
import curved_reference as cr  # noqa: E402
from probe_recompute_geometry import card, time_applies  # noqa: E402  (same directory)


def run(ctx, P, ndofs, rounds):
    n = api.boxmesh_fit(ndofs, P)
    q1 = api.BoxMesh(n, perturb=0.15)
    sp = q1.space(P)
    q2 = cr.q2_box(*n, phi=cr.sector)
    d_dm, d_bc = ctx.to_device(sp.dofmap), ctx.to_device(sp.bc)
    d_k = torch.full((q1.n_cells,), 2.0, dtype=torch.float64, device=ctx.device)
    geo = {"q1_perturbed": (ctx.to_device(q1.xgeom), ctx.to_device(q1.geom_dofmap), 0),
           "q2_curved": (ctx.to_device(q2.verts), ctx.to_device(q2.geom_dofmap), api.LAP_GEOM_Q2)}
    del q2
    ops, create_ms = {}, {}
    for name, (d_x, d_g, flags) in geo.items():
        ctx.sync()
        t0 = time.perf_counter()
        ops[name] = api.MatFreeLaplacian(ctx, P, d_k, d_dm, d_x, d_g, q1.lcells, q1.bcells, d_bc, sp.n_owned, 0, None,
                                         flags)
        create_ms[name] = round((time.perf_counter() - t0) * 1e3, 2)
    x, y = api.Vector(ctx, sp.n_owned), api.Vector(ctx, sp.n_owned)
    x.copy_from_host(np.random.default_rng(1).uniform(-1, 1, sp.n_owned))
    ms = {name: [] for name in ops}
    for _ in range(rounds):
        for name, op in ops.items():
            ms[name].append(time_applies(ctx, op, x, y))
    out = dict(P=P, n=list(n), ndofs=sp.n_owned, cells=q1.n_cells,
               kernel={k: op.kernel_name() for k, op in ops.items()},
               create_ms=create_ms,
               apply_ms={k: [round(v, 4) for v in vs] for k, vs in ms.items()},
               device_bytes={k: op.device_bytes() for k, op in ops.items()})
    print(json.dumps(out), flush=True)
    for op in ops.values():
        op.destroy()
    del d_dm, d_bc, d_k, geo, x, y
    torch.cuda.empty_cache()


if __name__ == "__main__":
    nd = int(float(sys.argv[1])) if len(sys.argv) > 1 else 100_000_000
    degs = [int(a) for a in sys.argv[2].split(",")] if len(sys.argv) > 2 else list(range(1, 9))
    rounds = int(sys.argv[3]) if len(sys.argv) > 3 else 2
    ctx = api.Context(0)
    name, pl = card()
    print(json.dumps(dict(card=name, power_limit=pl, warmup=3, reps=20, rounds=rounds)), flush=True)
    for P in degs:
        run(ctx, P, nd, rounds)
