#!/usr/bin/env python
"""bench.py -- p-MG hot path benchmark (contract: one JSON line on rank 0).

Workload (BASELINE.json configs[4], "examples/pmg"): Poisson on a unit-cube hex mesh, p-multigrid
V-cycle P4 -> P2 -> P1, 4th-kind Chebyshev smoother with 2 iterations per level, lambda_max from
a 20-iteration Jacobi-CG with b = 1 (examples/pmg/main.cpp:306-330), assembled-CSR Jacobi-PCG
coarse solve behind the coarse-solver hook, ~100 M P4 dofs per GPU (weak scaling: the mesh-fit
routine of examples/pmg/main.cpp:412-435 is run on ndofs * n_gpus).  One "step" = one V-cycle
(MultigridPreconditioner::apply, src/pmg.hpp:56-155).  metric = fine-level Gdof/s per V-cycle;
the per-apply throughput of the fine-level operator and its HBM roofline fraction are reported
in "apply" / "roofline".

  python bench.py [--gpus N] [--steps K] [--warmup W] [--ndofs D] [--impl reference] [--dump-outputs DIR]
  torchrun --nproc-per-node N bench.py --gpus N ...     (one rank per GPU, NCCL halo exchange)

--dump-outputs DIR: after the timed V-cycles, write the solution u they left behind (what a caller of
MultigridPreconditioner::apply receives) as DIR/u.npy, a fixed seeded sample of its owned entries in
float64, with their positions in DIR/u_index.npy (float64, exact), so that two builds run with the
same arguments can be compared output for output.  With N ranks each rank writes a sample of at most
2^20 / N entries as u_rank<r>.npy / u_rank<r>_index.npy, so a dump holds at most 2^20 values and
2^20 positions (16 MiB) for any number of ranks.

--impl reference: the reference's CPU path cannot be installed here (DOLFINx/PETSc absent), so
the arm times the oracle's C/OpenMP restatement of the same V-cycle on the host cores, on a
bounded sample of the workload (see "cpu_baseline.sample").
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

DEGREES = (1, 2, 4)
NSMOOTH = 2
# the reference's coarse KSP: CG, maxits = 60, PETSc default rtol 1e-5 (src/amg.hpp:36-40)
COARSE_ITS, COARSE_RTOL = 60, 1e-5
PGRID = {1: (1, 1, 1), 2: (2, 1, 1), 4: (2, 2, 1), 8: (2, 2, 2)}
METRIC = "fine-level Gdof/s per p-MG V-cycle (P4->P2->P1, Chebyshev(2), CSR coarse solve)"
DUMP_SAMPLE, DUMP_SEED = 1 << 20, 20240611   # 2^20 float64 values + positions over all ranks: 16 MiB


def dump_output(torch, v, out_dir, name, sample):
    """Write a fixed seeded sample of at most `sample` entries of the device vector v (all of it when it
    is small) and the sampled positions as out_dir/<name>.npy and out_dir/<name>_index.npy, both float64."""
    n = v.numel()
    idx = np.arange(n) if n <= sample else np.unique(np.random.default_rng(DUMP_SEED).integers(0, n, sample))
    vals = v[torch.from_numpy(idx).to(v.device)].cpu().numpy()
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, f"{name}.npy"), vals.astype(np.float64))
    np.save(os.path.join(out_dir, f"{name}_index.npy"), idx.astype(np.float64))


def b_apply(P, ncells, ndofs):
    """Algorithmic bytes of one operator apply (SURVEY 8d)."""
    return ncells * ((P + 1) ** 3 * 52 + 8) + ndofs * 17


def own_bytes(P, ncells, ndofs):
    """Bytes the affine-geometry kernel needs: one 48-byte geometry vector per cell instead of one per
    quadrature point (dofmap, kappa, x, y, BC marker as in B_apply)."""
    return ncells * ((P + 1) ** 3 * 4 + 48 + 8) + ndofs * 17


def measured_traffic(P, ncells, key=None):
    """DRAM bytes of one apply launch from the committed ncu --set full capture (profiles/), scaled
    by the number of cells if this run's launch differs from the captured one; None if absent."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "apply_traffic.json")))[key or str(P)]
        return (t["dram_bytes_read"] + t["dram_bytes_write"]) * ncells / t["cells"], t["source"]
    except Exception:
        return None, None


def measured_peak():
    try:
        pk = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(pk["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------ clocks --
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, dev):
        self.dev, self.rows, self.proc = dev, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i",
                 str(self.dev)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 7 for i in range(4) if r[3 + i].lower() == "active"})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


# --------------------------------------------------------------------- CPU (oracle) arm --
def cpu_vcycle_setup(n_cells_1d):
    """Oracle V-cycle P4->P2->P1 on an n^3 sample, C/OpenMP kernels (oracle/c/pmg_oracle.c)."""
    from oracle import mesh as om, operator as oo, solvers as osol, cport
    m = om.create_box(n_cells_1d, n_cells_1d, n_cells_1d)
    kap = np.full(m.ncells, 2.0)
    levels, dms = [], {}
    for P in DEGREES:
        dm, bc, nd = om.dofmap(m, P), om.bc_marker(m, P), om.num_dofs(m, P)
        dms[P] = (dm, nd)
        G, _ = cport.geometry(m.verts, m.geom_dofmap, P)
        A = cport.Apply(P, dm, G, kap, bc, nd)
        dinv = 1.0 / oo.diagonal(P, dm, G, kap, bc, nd)
        _, _, al, be, _, _ = osol.cg(A, dinv, np.zeros(nd), np.ones(nd), 20, 1e-6)
        lmax = 1.1 * osol.lanczos_eigenvalues(al, be)[-1]
        levels.append(osol.Level(A, dinv, bc.astype(float), lmax, NSMOOTH))
        if P == DEGREES[0]:
            A0 = oo.assemble_csr(P, dm, G, kap, bc, nd)
            d0 = 1.0 / A0.diagonal()
    pro, res = [], []
    for a, b in zip(DEGREES[:-1], DEGREES[1:]):
        mult = oo.multiplicity(dms[b][0], dms[b][1])
        pro.append((lambda a, b: lambda xc: oo.prolong(a, b, dms[a][0], dms[b][0], xc, dms[b][1]))(a, b))
        res.append((lambda a, b, mult: lambda xf: oo.restrict(a, b, dms[a][0], dms[b][0], xf, dms[a][1], mult))(a, b, mult))
    coarse = lambda u0, b0: osol.cg(lambda v: cport.spmv(A0, v), d0, u0, b0, COARSE_ITS, COARSE_RTOL)[0]
    Pt = DEGREES[-1]
    b = oo.rhs_collocated(m, Pt, oo.f_sines(2, 3, 4, 2.0), om.bc_marker(m, Pt))
    nd = dms[Pt][1]
    step = lambda u: osol.vcycle(levels, pro, res, b, u, coarse_solve=coarse)
    return step, nd, cport.num_threads(), levels[-1].A


def cpu_baseline(steps=2, warmup=1, n=64):
    # torch.distributed.run exports OMP_NUM_THREADS=1: the CPU arm must use every host core it can
    # (VERDICT r1 weak #11), so the OpenMP thread count is set explicitly
    from oracle import cport
    cport.set_num_threads(os.cpu_count() or 1)
    # the hot kernels are the oracle's C/OpenMP routines; numpy's BLAS pool must not spin next to
    # libgomp's threads (measured: 306 -> 61 ms per V-cycle on 8 cores with the BLAS pool at 1 thread)
    try:
        from threadpoolctl import threadpool_limits
        threadpool_limits(limits=1, user_api="blas")
    except Exception:
        pass
    step, nd, threads, A = cpu_vcycle_setup(n)
    u = np.zeros(nd)
    for _ in range(warmup):
        u = step(u)
    t0 = time.perf_counter()
    for _ in range(steps):
        u = step(u)
    dt = (time.perf_counter() - t0) / steps
    x = np.ones(nd)
    y = np.empty(nd)
    A(x, y)
    t0 = time.perf_counter()
    for _ in range(5):
        A(x, y)
    dta = (time.perf_counter() - t0) / 5
    return {"value": nd / dt / 1e9, "unit": "Gdof/s", "cores": threads, "kind": "port",
            "sample": f"oracle C/OpenMP V-cycle P4->P2->P1 on a {n}^3-cell unit cube ({nd} P4 dofs; the GPU arm runs "
                      f"~1e8 P4 dofs per GPU -- the CPU sample is bounded by run time, not the same size), "
                      f"{steps} timed V-cycles after {warmup} warm-up; same smoother settings, "
                      f"Jacobi-PCG coarse solve (<= {COARSE_ITS} its, rtol {COARSE_RTOL}); "
                      f"{threads} OpenMP threads of {os.cpu_count()} host cores",
            "ms_per_step": dt * 1e3, "apply_gdofs": nd / dta / 1e9}


def cpu_baseline_args(args):
    """Timed and warm-up V-cycles and sample size of the CPU leg: the run's --steps / --warmup (at least one
    warm-up cycle), on a bounded sample: 64^3 cells (16.97 M P4 dofs, ~6 s per V-cycle on 8 cores) while
    the whole run stays within a few minutes, else 48^3."""
    return dict(steps=args.steps, warmup=max(args.warmup, 1),
                n=args.cpu_cells or (64 if args.steps + args.warmup <= 24 else 48))


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cb = cpu_baseline(**cpu_baseline_args(args))
    line = {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": "Gdof/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": cb["ms_per_step"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "examples/pmg: P4->P2->P1 V-cycle, ~100M P4 dofs per GPU (BASELINE configs[4])",
                       "sample": cb["sample"],
                       "degrees": list(DEGREES), "smoother_its": NSMOOTH, "coarse": f"CSR Jacobi-PCG <= {COARSE_ITS} its",
                       "note": "reference's DOLFINx/PETSc CPU path not installable here; oracle C/OpenMP port timed"},
            "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": cb["value"], "unit": "Gdof/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def bind_to_gpu_numa_node(local):
    """Pin this rank's host threads (and therefore the first-touch placement of its pinned staging buffers)
    to the NUMA node its GPU hangs off: with 8 ranks on one host every step moves 6.4 GB each way, and
    buffers that land on the far socket halve the PCIe rate (VERDICT r1 weak #10).  Best effort: returns a
    description or None when the topology cannot be read."""
    try:
        import torch
        bus = torch.cuda.get_device_properties(local).pci_bus_id if hasattr(torch.cuda.get_device_properties(local), "pci_bus_id") else None
        dom = getattr(torch.cuda.get_device_properties(local), "pci_domain_id", 0)
        dev = getattr(torch.cuda.get_device_properties(local), "pci_device_id", 0)
        if bus is None:
            return None
        path = f"/sys/bus/pci/devices/{dom:04x}:{bus:02x}:{dev:02x}.0/numa_node"
        node = int(open(path).read().strip())
        if node < 0:
            return None
        cpus = []
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.extend(range(int(a), int(b or a) + 1))
        allowed = sorted(set(cpus) & os.sched_getaffinity(0))
        if not allowed:
            return None
        os.sched_setaffinity(0, allowed)
        return {"numa_node": node, "cpus": len(allowed)}
    except Exception:
        return None


# ------------------------------------------------------------------------------ GPU arm --
def build_problem(ctx, api, torch, mesh, halos_on):
    """Operators, smoothers, interpolators, coarse solver and V-cycle for one rank."""
    lv = []
    for P in DEGREES:
        sp = mesh.space(P, want_coords=(P == DEGREES[-1]))
        halo = api.Halo.from_space(ctx, sp) if halos_on else None
        d = {"P": P, "sp": sp, "halo": halo, "dofmap": ctx.to_device(sp.dofmap), "bc": ctx.to_device(sp.bc)}
        lv.append(d)
    xgeom, gdm = ctx.to_device(mesh.xgeom), ctx.to_device(mesh.geom_dofmap)
    kappa = torch.full((mesh.n_cells,), 2.0, dtype=torch.float64, device=ctx.device)
    ops, smoothers, eigs = [], [], []
    for d in lv:
        sp = d["sp"]
        op = api.MatFreeLaplacian(ctx, d["P"], kappa, d["dofmap"], xgeom, gdm, mesh.lcells, mesh.bcells, d["bc"],
                                  sp.n_owned, sp.n_ghost, d["halo"])
        cg = api.CGSolver(ctx, sp.n_owned, sp.n_ghost)
        cg.set_max_iterations(20)
        cg.set_tolerance(1e-6)
        cg.store_coefficients(True)
        x, y = api.Vector(ctx, sp.n_owned, sp.n_ghost), api.Vector(ctx, sp.n_owned, sp.n_ghost)
        y.set(1.0)
        cg.solve(op, x, y)
        eig = cg.compute_eigenvalues()
        s = api.Chebyshev(ctx, sp.n_owned, sp.n_ghost, (0.1 * eig[-1], 1.1 * eig[-1]))
        s.set_max_iterations(NSMOOTH)
        ops.append(op)
        smoothers.append(s)
        eigs.append(float(eig[-1]))
        del cg, x, y
    interps = []
    for a, b in zip(lv[:-1], lv[1:]):
        interps.append(api.Interpolator(ctx, a["P"], b["P"], a["dofmap"], b["dofmap"],
                                        a["sp"].n_owned + a["sp"].n_ghost, b["sp"].n_owned + b["sp"].n_ghost,
                                        mesh.lcells, mesh.bcells, a["halo"], b["halo"]))
    A0 = ops[0].to_csr()
    coarse = api.CoarseSolverType(ctx, A0, COARSE_ITS, COARSE_RTOL, amg=not os.environ.get("PMGX_BENCH_JACOBI_COARSE"))
    pmg = api.MultigridPreconditioner(ctx, [d["bc"] for d in lv])
    pmg.set_solvers(smoothers)
    pmg.set_operators(ops)
    pmg.set_interpolators(interps)
    pmg.set_coarse_solver(coarse)
    top = lv[-1]
    sp = top["sp"]
    X = sp.coords
    kx, ky, kz, kap = 2, 3, 4, 2.0
    f = (kap * np.pi ** 2 * (kx * kx + ky * ky + kz * kz) * np.sin(kx * np.pi * X[:, 0]) * np.sin(ky * np.pi * X[:, 1])
         * np.sin(kz * np.pi * X[:, 2]))
    b = api.Vector(ctx, sp.n_owned, sp.n_ghost, top["halo"])
    ops[-1].assemble_rhs(ctx.to_device(f), 0.0, b)
    sp.coords = None
    keep = (lv, xgeom, gdm, kappa, A0, coarse, interps, smoothers)
    return pmg, ops, b, eigs, keep


def run_gpu(args):
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torchrun --nproc-per-node N for --gpus N > 1")
    torch.cuda.set_device(local)
    numa = bind_to_gpu_numa_node(local) if world > 1 else None
    from pmg_dolfinx_b200 import api
    nccl_id = None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        box = [api.Context.nccl_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        nccl_id = box[0]
    ctx = api.Context(local, rank, world, nccl_id)

    # Parity gate in the same process, on the same ranks and transport as the timed run: a small
    # perturbed box partitioned like the benchmark mesh, apply / diagonal / CG / Chebyshev / 3 V-cycles
    # gathered to rank 0 and compared with the single-domain oracle (1e-12 / 1e-10 / identical CG
    # counts).  The oracle is the checker only; nothing of it runs inside the timed region.
    parity = {"checked": False}
    if not args.no_parity:
        import importlib.util
        spec = importlib.util.spec_from_file_location("mgpu_check", os.path.join(ROOT, "scripts", "mgpu_check.py"))
        mc = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mc)
        res = mc.run_check(api, ctx, rank, world, log=lambda m: sys.stderr.write(m + "\n"))
        res2 = mc.run_check(api, ctx, rank, world, perturb=0.0, log=lambda m: sys.stderr.write(m + "\n"))
        parity = {"checked": True, "ok": bool(res["ok"] and res2["ok"]), "max_rel": max(res["max_rel"], res2["max_rel"]),
                  "max_err_over_tol": max(res["max_err_over_tol"], res2["max_err_over_tol"]),
                  "transport": res["transport"], "ranks": world, "mesh_cells": res["mesh"],
                  "cases": "perturbed (streamed-G kernels) + uniform (affine kernel): P1/P2/P4 apply 1e-12, diag 1e-13, "
                           "CG history 1e-10 + identical iteration counts, 3 V-cycles stage residuals 1e-9 vs single-domain oracle",
                  "cg_iterations": {k: v for k, v in res["checks"].items() if "iterations" in k}}
        if not parity["ok"]:
            if rank == 0:
                print(json.dumps({"metric": METRIC, "error": "parity check failed", "parity": parity}), flush=True)
            raise SystemExit(3)

    def barrier():
        ctx.sync()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    Ptop = DEGREES[-1]
    n = api.boxmesh_fit(args.ndofs * world, Ptop)
    mesh = api.BoxMesh(n, PGRID[world], rank)
    pmg, ops, b, eigs, keep = build_problem(ctx, api, torch, mesh, world > 1)
    sp = keep[0][-1]["sp"]
    n_owned = sp.n_owned
    nd_global = sp.n_global
    u = api.Vector(ctx, sp.n_owned, sp.n_ghost)
    rn0 = api.norm(b)
    # warm-up
    for _ in range(args.warmup):
        pmg.apply(b, u)
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    l0 = ctx.launch_count()
    api.check(api.lib.pmgx_ctx_profile(ctx.h, 1))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record(ctx.stream)
    for _ in range(args.steps):
        pmg.apply(b, u)
    e1.record(ctx.stream)
    barrier()
    ms = e0.elapsed_time(e1)
    if args.dump_outputs:
        dump_output(torch, u.data[:n_owned], args.dump_outputs, "u" if world == 1 else f"u_rank{rank}",
                    DUMP_SAMPLE // world)
    import ctypes
    kms, kl = ctypes.c_double(), ctypes.c_longlong()
    api.check(api.lib.pmgx_ctx_profile_read(ctx.h, Ptop, ctypes.addressof(kms), ctypes.addressof(kl)))
    api.check(api.lib.pmgx_ctx_profile(ctx.h, 0))
    launches = ctx.launch_count() - l0
    rn = pmg.apply(b, u, verbose=True)  # residual after warmup+steps+1 cycles (untimed)
    t = torch.tensor([ms], dtype=torch.float64, device=ctx.device)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    ms_per_step = ms_max / args.steps

    # fine-level operator apply alone (the kernel the roofline is quoted on), incl. zero fill
    x, y = api.Vector(ctx, sp.n_owned, sp.n_ghost, keep[0][-1]["halo"]), api.Vector(ctx, sp.n_owned, sp.n_ghost)
    x.set(1.0)
    for _ in range(3):
        ops[-1](x, y)
    barrier()
    reps = 20
    a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a0.record(ctx.stream)
    for _ in range(reps):
        ops[-1](x, y)
    a1.record(ctx.stream)
    barrier()
    ta = torch.tensor([a0.elapsed_time(a1) / reps], dtype=torch.float64, device=ctx.device)
    if world > 1:
        dist.all_reduce(ta, op=dist.ReduceOp.MAX)
    apply_ms = float(ta.item())

    # the same apply with the reference's data flow (per-quadrature-point G streamed from HBM): the
    # kernel the B_apply roofline model describes; built only to be timed next to the default
    affine = ops[-1].is_affine()
    sg_ms, sg_kms, sg_kl = None, ctypes.c_double(), ctypes.c_longlong()
    if affine:
        lvt = keep[0][-1]
        op_s = api.MatFreeLaplacian(ctx, Ptop, keep[3], lvt["dofmap"], keep[1], keep[2], mesh.lcells, mesh.bcells,
                                    lvt["bc"], sp.n_owned, sp.n_ghost, lvt["halo"], flags=2 | 4)
        for _ in range(3):
            op_s(x, y)
        barrier()
        api.check(api.lib.pmgx_ctx_profile(ctx.h, 1))
        a0.record(ctx.stream)
        for _ in range(reps):
            op_s(x, y)
        a1.record(ctx.stream)
        barrier()
        api.check(api.lib.pmgx_ctx_profile_read(ctx.h, Ptop, ctypes.addressof(sg_kms), ctypes.addressof(sg_kl)))
        api.check(api.lib.pmgx_ctx_profile(ctx.h, 0))
        ts = torch.tensor([a0.elapsed_time(a1) / reps], dtype=torch.float64, device=ctx.device)
        if world > 1:
            dist.all_reduce(ts, op=dist.ReduceOp.MAX)
        sg_ms = float(ts.item())
        op_s.destroy()
        del op_s
        torch.cuda.empty_cache()

    # end-to-end through the public API with HOST buffers: every step uploads its right-hand side
    # from pinned host memory, runs the V-cycle and reads the solution back to pinned host memory.
    # The copies run on their own streams (PCIe is full duplex): step i's upload overlaps step
    # i-1's V-cycle and step i-2's read-back; b is double-buffered on the device, u is snapshotted
    # (D2D) before the read-back because the cycle updates it in place.
    hb = torch.empty(n_owned, dtype=torch.float64).pin_memory()
    hu = [torch.empty(n_owned, dtype=torch.float64).pin_memory() for _ in range(2)]
    hb.copy_(b.data[:n_owned])
    halo_top = keep[0][-1]["halo"]
    bb = [b, api.Vector(ctx, sp.n_owned, sp.n_ghost, halo_top)]
    us = [torch.empty(n_owned, dtype=torch.float64, device=ctx.device) for _ in range(2)]
    s_up, s_down = torch.cuda.Stream(device=ctx.device), torch.cuda.Stream(device=ctx.device)
    e2e_steps = args.steps

    def e2e_loop(nsteps, e_begin=None, e_end=None):
        trace = bool(os.environ.get("PMGX_E2E_TRACE")) and e_begin is not None
        up = [torch.cuda.Event(enable_timing=trace) for _ in range(nsteps)]      # b of step i is on the device
        used = [torch.cuda.Event(enable_timing=trace) for _ in range(nsteps)]    # V-cycle i done with b, u snapshot taken
        down = [torch.cuda.Event(enable_timing=trace) for _ in range(nsteps)]    # u of step i is on the host
        if e_begin is not None:
            e_begin.record(ctx.stream)
        s_up.wait_stream(ctx.stream)
        s_down.wait_stream(ctx.stream)
        def upload(i):
            with torch.cuda.stream(s_up):
                if i >= 2:
                    s_up.wait_event(used[i - 2])               # buffer i%2 is free again
                bb[i % 2].data[:n_owned].copy_(hb, non_blocking=True)
                up[i].record(s_up)

        upload(0)
        for i in range(nsteps):
            if i + 1 < nsteps:
                upload(i + 1)   # enqueued before apply(i): the host blocks inside the cycle (coarse-solve checks)
            ctx.stream.wait_event(up[i])
            pmg.apply(bb[i % 2], u)
            if i >= 2:
                ctx.stream.wait_event(down[i - 2])            # snapshot i%2 has left the device
            us[i % 2].copy_(u.data[:n_owned], non_blocking=True)
            used[i].record(ctx.stream)
            with torch.cuda.stream(s_down):
                s_down.wait_event(used[i])
                hu[i % 2].copy_(us[i % 2], non_blocking=True)
                down[i].record(s_down)
        ctx.stream.wait_event(down[-1])
        if nsteps > 1:
            ctx.stream.wait_event(down[-2])
        if e_end is not None:
            e_end.record(ctx.stream)
        if trace and rank == 0:
            ctx.sync()
            torch.cuda.synchronize()
            for i in range(nsteps):
                sys.stderr.write(f"e2e step {i}: b on device {e_begin.elapsed_time(up[i]):8.2f}  cycle done "
                                 f"{e_begin.elapsed_time(used[i]):8.2f}  u on host {e_begin.elapsed_time(down[i]):8.2f} ms\n")

    # same cycles as the device-resident measurement: restart from u = 0, W untimed cycles, K timed
    # (the cost of a cycle depends on how far the solve has converged: the coarse PCG stops early
    # on the first cycles and runs into its 60-iteration cap later)
    u.set(0.0)
    e2e_loop(max(args.warmup, 2))
    barrier()
    s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if os.environ.get("PMGX_E2E_TRACE"):
        api.check(api.lib.pmgx_ctx_profile(ctx.h, 1))
    e2e_loop(e2e_steps, s0, s1)
    barrier()
    if os.environ.get("PMGX_E2E_TRACE"):
        tms, tl = ctypes.c_double(), ctypes.c_longlong()
        api.check(api.lib.pmgx_ctx_profile_read(ctx.h, Ptop, ctypes.addressof(tms), ctypes.addressof(tl)))
        api.check(api.lib.pmgx_ctx_profile(ctx.h, 0))
        if rank == 0:
            sys.stderr.write(f"e2e: P{Ptop} apply launches {tl.value}, avg {tms.value / max(tl.value, 1):.3f} ms\n")
    te = torch.tensor([s0.elapsed_time(s1) / e2e_steps], dtype=torch.float64, device=ctx.device)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_ms = float(te.item())
    torch.cuda.set_stream(ctx.stream)
    # sampled from before the timed V-cycles until here: the timed region, the apply loops and the
    # end-to-end loop are all GPU-loaded (100 ms sampling period: the timed region alone yields 1-2 samples)
    clocks = sampler.stop() if rank == 0 else None

    if rank == 0:
        peak, peak_src = measured_peak()
        n_own_cells = mesh.n_owned_cells
        # the timed launches are the interior-cell launches on the compute stream (all cells at N = 1;
        # the boundary-cell launch of a multi-rank apply overlaps their tail on the halo stream)
        n_applies = kl.value
        frac_int = len(mesh.lcells) / max(n_own_cells, 1)
        B = b_apply(Ptop, n_own_cells, n_owned)
        B_launch = b_apply(Ptop, len(mesh.lcells), n_owned * frac_int)
        kname = ops[-1].kernel_name()
        traffic, traffic_src = measured_traffic(Ptop, len(mesh.lcells), f"{Ptop}_affine" if affine else str(Ptop))
        B_own = own_bytes(Ptop, len(mesh.lcells), n_owned * frac_int) if affine else B_launch
        t_launch = kms.value * 1e-3 / max(n_applies, 1)            # s, CUDA events around each interior launch
        flops_launch = len(mesh.lcells) * (Ptop + 1) ** 3 * (12 * (Ptop + 1) + 20)   # SURVEY 8d, secondary
        fp64_peak = 148 * 128 * 1.965e9 / 1e12                    # nominal: 64 FP64 FMA/clk/SM at the 1965 MHz max clock
        B_kernel = B_own if affine else B_launch
        roofline = {
            "bound": "hbm", "kernel": kname, "unit": "GB/s", "peak": peak, "peak_source": peak_src,
            # achieved = the bytes THIS kernel has to move per launch (its own algorithmic model) / launch time
            "achieved": B_kernel / t_launch / 1e9 if n_applies else None,
            "frac": B_kernel / t_launch / 1e9 / peak if n_applies else None,
            "algorithmic_bytes_per_launch": B_kernel,
            "bytes_model": ("affine geometry, G(q) = w_q Gc: dofmap 4 B per cell dof + 48 B Gc + 8 B kappa per cell + "
                            "17 B per dof (x, y, BC marker)") if affine else
                           "SURVEY 8d: (P+1)^3 * 52 B + 8 B per cell + 17 B per dof",
            "traffic": traffic, "traffic_source": traffic_src,
            "frac_dram_measured": (traffic / t_launch / 1e9 / peak) if (traffic and n_applies) else None,
            "fp64": {"tflops": flops_launch / t_launch / 1e12 if n_applies else None, "peak_tflops_nominal": fp64_peak,
                     "frac": flops_launch / t_launch / 1e12 / fp64_peak if n_applies else None,
                     "flops_per_launch": flops_launch},
            "launches_timed": kl.value, "cells_per_launch": len(mesh.lcells), "avg_launch_ms": t_launch * 1e3,
            # the SURVEY 8d model charges 48 B of G per quadrature point; the affine kernel does not stream
            # them, so this ratio is NOT a roofline fraction (it exceeds 1 by construction) -- it is the
            # speed-up over a kernel that streams G at the full HBM peak
            "streamed_model_8d": ({"bytes_per_launch": B_launch, "effective_gbs": B_launch / t_launch / 1e9,
                                   "times_hbm_peak": B_launch / t_launch / 1e9 / peak} if affine and n_applies else None),
            # the kernel that follows the 8d data flow (per-quadrature-point G streamed through the TMA ring),
            # timed in the same run on the same mesh: this is the HBM-roofline number of the path
            "streamed_G": ({"kernel": f"k_apply_tma<{Ptop},128,2>", "apply_ms": sg_ms,
                            "avg_launch_ms": sg_kms.value / max(sg_kl.value, 1),
                            "achieved": B_launch * sg_kl.value / (sg_kms.value * 1e-3) / 1e9,
                            "frac": B_launch * sg_kl.value / (sg_kms.value * 1e-3) / 1e9 / peak,
                            "traffic": measured_traffic(Ptop, len(mesh.lcells), str(Ptop))[0]}
                           if affine and sg_kms.value > 0 else None),
        }
        if roofline["frac"] is not None:
            assert roofline["frac"] <= 1.2, f"roofline.frac {roofline['frac']} is not a fraction of a roofline"
        cb = None
        if world == 1 and not args.no_cpu:
            try:
                cb = cpu_baseline(**cpu_baseline_args(args))
            except Exception as e:  # the CPU leg must never take the GPU line down with it
                sys.stderr.write(f"cpu_baseline failed: {e}\n")
        line = {
            "metric": METRIC, "value": nd_global / ms_per_step / 1e6, "unit": "Gdof/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "examples/pmg: P4->P2->P1 V-cycle, ~100M P4 dofs per GPU (BASELINE configs[4])",
                       "mesh_cells": list(n), "partition": list(PGRID[world]), "dofs_global": nd_global,
                       "dofs_per_level_rank0": [d["sp"].n_owned for d in keep[0]], "degrees": list(DEGREES),
                       "smoother": f"Chebyshev-4 Jacobi, {NSMOOTH} its", "lambda_max": eigs,
                       "coarse": (f"CSR PCG <= {COARSE_ITS} its, rtol {COARSE_RTOL} (src/amg.hpp:36-40), preconditioner: "
                                  + ("smoothed-aggregation V(2,2) cycle, Chebyshev-4/Jacobi smoother" if keep[5].amg else "Jacobi")),
                       "coarse_levels_rank0": keep[5].levels(), "coarse_converged_last_cycle": keep[5].last_status()[0],
                       "coarse_rel_residual_last_cycle": keep[5].last_status()[1],
                       "l2": "working set >> 126 MB L2, no flush needed",
                       "coarse_iterations_last_cycle": int(api.lib.pmgx_coarse_last_iterations(keep[5].h)),
                       "halo": "nvlink-p2p" if api.lib.pmgx_ctx_uses_p2p(ctx.h) else ("nccl" if world > 1 else "none"),
                       "residual_reduction_after_cycles": [args.warmup + args.steps + 1, rn / rn0]},
            "apply": {"degree": Ptop, "ms": apply_ms, "gdofs": nd_global / apply_ms / 1e6,
                      "gbs_algorithmic": B / apply_ms / 1e6, "frac_of_hbm_peak": B / apply_ms / 1e6 / peak,
                      "geometry": "affine: one 6-vector per cell" if affine else "streamed per quadrature point",
                      "note": "operator()(x,y) incl. zero fill of y and halo; max over ranks"},
            "roofline": roofline,
            "e2e": {"value": nd_global / e2e_ms / 1e6, "unit": "Gdof/s", "ms_per_step": e2e_ms, "steps": e2e_steps,
                    "note": "per step: H2D of b from pinned host memory, V-cycle, D2H of u; copies on their "
                            "own streams overlap the neighbouring steps' compute (pipeline fill and drain "
                            "are inside the timed region)",
                    "h2d_bytes_per_step": n_owned * 8 * world, "d2h_bytes_per_step": n_owned * 8 * world,
                    "host_numa_binding_rank0": numa},
            "parity": parity, "gpu_launches": launches, "clocks": clocks,
        }
        if cb is not None:
            line["cpu_baseline"] = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")}
            line["cpu_baseline"]["apply_gdofs"] = cb["apply_gdofs"]
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--ndofs", type=float, default=1e8, help="P4 dofs per GPU (weak scaling)")
    ap.add_argument("--cpu-cells", type=int, default=0, help="cells per direction of the CPU sample (0: 64, or 48 for long runs)")
    ap.add_argument("--no-parity", action="store_true", help="skip the in-process parity check before the timed region")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write a sample of the last timed V-cycle's solution to DIR")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the GPU path's solution; it needs --impl b200")
    args.ndofs = int(args.ndofs)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
