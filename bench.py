#!/usr/bin/env python
"""bench.py - the north-star hot path on synthetic refined P1 meshes (BASELINE.json config 4/5).

A *step* is one CONVERGED Newton-iteration pass of the hot path over one mesh, all inputs resident in HBM:
    strain E = B u  ->  Drucker-Prager return map  ->  K_tangent assembly + internal force (one pass)
      ->  CG + geometric multigrid V-cycle on K_tangent[Q,Q] to rtol 1e-10  ->  energy-norm criterion
(--solver jacobi: round 1's fixed number of Jacobi-PCG iterations instead; a fixed-iteration Jacobi run is still timed
beside the step for the per-iteration roofline of the SpMV/PCG kernels)
`value` is the first component of BASELINE.json's metric, K_tangent assembly throughput in Melem/s
(elements of all ranks / CUDA-event time of the assembly kernel inside the timed steps, max over ranks);
`parts` carries the other two components (DP return map Mpts/s, PCG-Newton s/step with ms/iteration) and
`rooflines` the achieved HBM bandwidth of every kernel against MEASURED_PEAKS.json.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--nx 2828] [--pcg-iters 20] [--dump-outputs DIR]
    python bench.py --impl reference      # the oracle port of the reference's CPU path on a bounded sample
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
METRIC = "K_tangent assembly Melem/s + DP return-map Mpts/s + PCG-Newton s/step; %HBM roof"


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 100 ms; samples inside the timed region are reported
    (plus, flagged, the ones taken under load during warm-up when the region is too short to catch three)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None
        self.t_begin = self.t_end = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def region_begin(self):
        self.t_begin = time.time()

    def region_end(self):
        self.t_end = time.time()

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"], "samples": 0}
        time.sleep(0.15)
        self.proc.terminate()
        ok = [(t, r) for t, r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        inside = [r for t, r in ok if self.t_begin is not None and self.t_begin <= t <= self.t_end + 0.1]
        note = "samples inside the timed region"
        if len(inside) < 3:
            inside = [r for t, r in ok if float(r[3]) > 250.0] if ok and all(x[1][3].replace(".", "").isdigit() for x in ok) else [r for _, r in ok]
            note = "timed region shorter than 3 sampling periods: samples under load (>250 W) from warm-up + timed region"
        sm = [float(r[1]) for r in inside]
        mx = [float(r[2]) for r in inside]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in inside for n, v in zip(names, r[5:9]) if v.lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm), "power_w_max": max([float(r[3]) for r in inside], default=None), "note": note}


# ------------------------------------------------------------------------------------------------
# CPU side: the oracle port of the reference path (NumPy/SciPy, single-threaded like the reference)
# ------------------------------------------------------------------------------------------------
def cpu_reference_pass(nx, pcg_iters, steps, warmup, seed=0):
    """Times the reference's statements (restated in oracle/fem_oracle.py) on an nx x nx P1 mesh."""
    import scipy.sparse.linalg as spla
    from oracle import fem_oracle as fo
    et = fo.ElementType.P1
    xi, wf = fo.quadrature_volume(et)
    _, d1, d2 = fo.local_basis_volume(et, xi)
    m = fo.square_mesh_p1(nx, nx, 10.0, 10.0)
    n_e = m["elements"].shape[1]
    G0, K0, eta0, c0, _ = fo.footing_constants()
    G, Kb, eta, c = (v * np.ones(n_e) for v in (G0, K0, eta0, c0))
    t0 = time.perf_counter()
    K, B, w, i_d, j_d, D = fo.elastic_stiffness(m["elements"], m["coordinates"], G, Kb, d1, d2, wf)
    t_elastic = time.perf_counter() - t0
    rng = np.random.default_rng(seed)
    E0 = np.array([[-3e-4], [-3e-4], [0.0]]) + 2e-4 * rng.standard_normal((3, n_e))
    U = 1e-3 * rng.standard_normal(m["coordinates"].shape)
    qf = m["Q"].flatten(order="F")
    t = {"strain": [], "return_map": [], "tangent": [], "force": [], "pcg": [], "criterion": [], "step": []}
    for s in range(warmup + steps):
        a = time.perf_counter()
        fo.strain(B, U)
        b = time.perf_counter()
        cp = fo.constitutive_problem(E0.copy(), np.zeros((4, n_e)), G, Kb, eta, c)
        c_ = time.perf_counter()
        Kt = fo.tangent_stiffness(K, B, D, w, cp["ds"], i_d, j_d)
        d = time.perf_counter()
        F = fo.internal_force(B, w, cp["s"])
        e = time.perf_counter()
        Kqq = Kt.tocsr()[qf][:, qf]
        dinv = 1.0 / Kqq.diagonal()
        e2 = time.perf_counter()                                  # the extraction is not counted as PCG time
        spla.cg(Kqq, -F[qf], rtol=0.0, atol=0.0, maxiter=pcg_iters, M=spla.LinearOperator(Kqq.shape, lambda v: dinv * v))
        f = time.perf_counter()
        u = U.flatten(order="F")
        fo.newton_criterion(K, u, u, u)
        g = time.perf_counter()
        if s >= warmup:
            for k, v in zip(("strain", "return_map", "tangent", "force", "pcg", "criterion"), (b - a, c_ - b, d - c_, e - d, f - e2, g - f)):
                t[k].append(v)
            t["step"].append((g - a) - (e2 - e))
    mean = {k: float(np.mean(v)) for k, v in t.items()}
    return {"n_e": n_e, "n_dof": int(2 * m["coordinates"].shape[1]), "nnz": int(K.nnz), "t": mean, "t_elastic": t_elastic}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    nx = args.cpu_nx
    r = cpu_reference_pass(nx, args.pcg_iters, args.steps, args.warmup)
    melem = r["n_e"] / r["t"]["tangent"] / 1e6
    sample = (f"oracle port (NumPy/SciPy restatement of Plasticity2D_DP/pythonFEM.py:1043-1075) on a {nx}x{nx} P1 mesh = "
              f"{r['n_e']} elements, {args.pcg_iters} SciPy-CG iterations/step; /root/reference is pure Python and does not travel")
    line = {"impl": "reference", "metric": METRIC, "value": melem, "unit": "Melem/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * r["t"]["step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"P1 uniform mesh {nx}x{nx} cells ({r['n_e']} elements): bounded sample of config 4", "pcg_iters": args.pcg_iters},
            "parts": {"return_map_mpts_s": r["n_e"] / r["t"]["return_map"] / 1e6, "pcg_ms_per_iter": 1e3 * r["t"]["pcg"] / max(args.pcg_iters, 1),
                      "newton_step_s": r["t"]["step"], "strain_ms": 1e3 * r["t"]["strain"], "force_ms": 1e3 * r["t"]["force"],
                      "elastic_assembly_melem_s": r["n_e"] / r["t_elastic"] / 1e6},
            "cpu_baseline": {"value": melem, "unit": "Melem/s", "cores": 1, "kind": "port", "sample": sample},
            "e2e": {"value": melem, "unit": "Melem/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


def multi_gpu_checks(args, P, part, mesh, pcg, k_tan, rhs, rm, d1, d2, wf, dev):
    """Correctness carried by an N > 1 run itself (every rank raises on failure):
    (a) the ghost cell row of rank r holds the same tangent operators as the first owned cell row of rank r+1;
    (b) the owned interface rows of K_tangent equal, bit for bit, a stand-alone single-GPU assembly of the two cell rows
        around the interface (same cells, same data, no partition);
    (c) the partitioned matrix is symmetric as ONE global operator: y'(K x) == x'(K y) over all ranks;
    (d) the fused iteration (exchanges inside the kernels over NVLink peer memory) reproduces the NCCL variant: same r'r
        after the step's fixed number of iterations."""
    import torch
    import torch.distributed as dist
    from fem_elastoplasticity_b200 import distributed as fdist, meshgen
    from fem_elastoplasticity_b200.plan import FemPlan
    nx, world, rank = part.nx, part.world, part.rank
    out = {}
    ds = rm["ds"]
    row = 2 * nx                                                     # elements per cell row
    # (a) checksums of the shared cell rows
    sums = torch.zeros(2 * world, dtype=torch.float64, device=dev)
    sums[2 * rank] = ds[:, :row].sum()                               # first owned cell row (local cell row 0)
    if part.has_upper:
        sums[2 * rank + 1] = ds[:, part.ny_loc * row:(part.ny_loc + 1) * row].sum()    # ghost cell row
    dist.all_reduce(sums)
    h = sums.cpu().numpy()
    for r in range(world - 1):
        assert h[2 * r + 1] == h[2 * (r + 1)], f"ghost cell row of rank {r} differs from the owner's data"
    out["ghost_data_identical"] = True
    # (b) stand-alone assembly of the cell rows around the upper interface (rank 0 also checks its lower boundary rows)
    if part.has_upper:
        lo_cell = part.ny_loc - 1
        thin = meshgen.square_mesh_p1(nx, 2, part.size_x, part.size_y, device=dev, iy0=part.iy0 + lo_cell, n_y_global=part.ny_global,
                                      size_y_global=part.size_y)
        Pt = FemPlan(thin["elements"], thin["coordinates"], d1, d2, wf, device=dev)
        kt = Pt.assemble_tangent(ds[:, lo_cell * row:(lo_cell + 2) * row].contiguous())
        a0, a1 = int(Pt.row_ptr[2 * (nx + 1)]), int(Pt.row_ptr[4 * (nx + 1)])          # middle node row of the thin mesh
        n0 = part.ny_loc * (nx + 1)                                                    # the same nodes in the local mesh: top owned row
        b0, b1 = int(P.row_ptr[2 * n0]), int(P.row_ptr[2 * (n0 + nx + 1)])
        assert a1 - a0 == b1 - b0 and torch.equal(kt[a0:a1], k_tan[b0:b1]), "interface rows differ from the stand-alone assembly"
        del Pt, kt
    out["interface_rows_equal_standalone_assembly"] = True
    # (c) global symmetry
    g = torch.Generator(device=dev).manual_seed(1234 + rank)
    xs = torch.randn(P.n_dof, dtype=torch.float64, device=dev, generator=g)
    ys = torch.randn(P.n_dof, dtype=torch.float64, device=dev, generator=g)
    part.halo_exchange(xs, ys)
    own = part.owned_mask(dev)
    kx, ky = P.spmv(k_tan, xs, mask=own), P.spmv(k_tan, ys, mask=own)
    sy = torch.stack([torch.dot(ys, kx), torch.dot(xs, ky)])
    dist.all_reduce(sy)
    asym = abs(float(sy[0] - sy[1])) / abs(float(sy[0]))
    assert asym <= 1e-11, f"partitioned K_tangent is not symmetric: {asym:.2e}"
    out["global_symmetry_rel"] = asym
    # (d) fused vs NCCL iteration
    if getattr(pcg, "fused", False):
        ref = fdist.DistributedPCG(P, part, pcg.mask, peer=False, use_graph=False)
        ref.solve(k_tan, rhs, iters=args.pcg_iters)
        rr_ref = float(ref.scal[1].item())
        pcg.solve(k_tan, rhs, iters=args.pcg_iters)
        rr_fused = float(pcg.peer.comm.view(torch.float64)[pcg.WORD_OUT + 1].item())
        xd = torch.stack([(pcg.x - ref.x).abs().max(), ref.x.abs().max()])
        dist.all_reduce(xd, op=dist.ReduceOp.MAX)
        out["fused_vs_nccl_rr_rel"] = abs(rr_fused - rr_ref) / abs(rr_ref)
        out["fused_vs_nccl_x_rel"] = float(xd[0] / xd[1])
        assert out["fused_vs_nccl_rr_rel"] <= 1e-8 and out["fused_vs_nccl_x_rel"] <= 1e-8, out
        del ref
    return out


def strong_scaling_part(args, world, rank, dev, d1, d2, wf, pcg_one_gpu_ms=None):
    """The nx x nx mesh of config 4 split over the N GPUs (strong scaling), timed in the same run as the weak-scaling
    headline: step ms and PCG ms/iteration, max over ranks.  The one-GPU time of the same mesh is the N = 1 run's."""
    import torch
    import torch.distributed as dist
    from fem_elastoplasticity_b200 import distributed as fdist, meshgen
    from fem_elastoplasticity_b200.plan import FemPlan, axpby, dp_return_map
    nx = args.nx
    ny_global = -(-nx // world) * world
    part = fdist.StripPartition(nx, ny_global, rank, world, size_x=10.0, size_y=10.0 * ny_global / nx)
    mesh = part.local_mesh(dev)
    P = FemPlan(mesh["elements"], mesh["coordinates"], d1, d2, wf, device=dev)
    G, Kb, eta, c = meshgen.footing_materials(P.n_int, dev)
    Es = meshgen.synthetic_strain_global(P.n_int, 2 * nx * part.iy0, dev)
    u = meshgen.synthetic_nodal_global(P.n_n, (nx + 1) * part.iy0, dev)
    mask = part.free_owned_mask(P, mesh)
    ep_old = torch.zeros((4, P.n_int), dtype=torch.float64, device=dev)
    E, k_tan, F, rhs, rm = P.empty(3, P.n_int), P.empty(P.nnz), P.empty(P.n_dof), P.empty(P.n_dof), {}
    k_el = P.assemble_elastic(G, Kb)
    pcg = fdist.DistributedPCG(P, part, mask, peer={"auto": "auto", "nccl": False, "peer": True, "fused": "fused"}[args.halo], use_graph=not args.no_graph)
    mgs = None
    if args.solver == "multigrid":
        from fem_elastoplasticity_b200.mg import MultigridPCG
        mgs = MultigridPCG(P, mask, part=part, free_mask=P.mask_u8(mesh["Q"]), degree=args.mg_degree, ratio=args.mg_ratio, **({} if args.mg_replicate_below is None else {"replicate_below": args.mg_replicate_below})).setup(k_el)
    evs, info = [], {"its": args.pcg_iters}

    def step(rec):
        e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        e[0].record()
        P.strain(u, out=E)
        dp_return_map(Es, ep_old, G, Kb, eta, c, want_ep=False, out=rm)
        P.assemble_tangent_force(rm["ds"], rm["s"], out_k=k_tan, out_f=F)
        axpby(-1.0, F, 0.0, F, out=rhs)
        e[1].record()
        if mgs is not None:
            x, info["its"], _ = mgs.solve(k_tan, rhs, rtol=args.rtol, maxit=args.converged_maxit)
        else:
            x, _ = pcg.solve(k_tan, rhs, iters=args.pcg_iters)
        e[2].record()
        pcg.energy_norms(k_el, x, u, rhs)
        if rec:
            evs.append(e)

    for _ in range(max(args.warmup, 3)):
        step(False)
    torch.cuda.synchronize()
    dist.barrier()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    n_steps = max(5, min(args.steps, 20))
    for _ in range(n_steps):
        step(True)
    t1.record()
    torch.cuda.synchronize()
    dist.barrier()
    v = torch.tensor([t0.elapsed_time(t1) / n_steps, float(np.mean([e[1].elapsed_time(e[2]) for e in evs])) / max(int(info["its"]), 1)],
                     dtype=torch.float64, device=dev)
    dist.all_reduce(v, op=dist.ReduceOp.MAX)
    return {"strong_n_elements": 2 * nx * ny_global, "strong_step_ms": float(v[0]), "strong_pcg_ms_per_iter": float(v[1]),
            "strong_pcg_iterations": int(info["its"]),
            "strong_note": f"config 4 mesh ({nx}x{ny_global} cells) split over {world} GPUs, the same converged step as the headline "
                           f"({'multigrid' if mgs is not None else 'jacobi'} PCG); the one-GPU time of this mesh is ms_per_step of the N=1 run"}


def bind_to_gpu_numa_node(index):
    """Pin this process to the CPU cores NVML reports as local to GPU ``index`` (first-touch then places the pinned host
    buffers on that NUMA node: with every rank on node 0 the end-to-end leg of round 1 did not scale past 1.5x at 8 GPUs)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = {64 * w + b for w, v in enumerate(words) for b in range(64) if (int(v) >> b) & 1}
        cpus &= set(os.sched_getaffinity(0))
        if cpus:
            os.sched_setaffinity(0, cpus)
            return f"{len(cpus)} cores local to GPU {index}"
    except Exception as e:  # noqa: BLE001
        return f"not bound ({type(e).__name__})"
    return "not bound"


DUMP_SAMPLE = 1 << 18   # entries kept along the last axis of an output: at most 41 MB for all outputs of a step


def dump_outputs(out_dir, arrays, rank, world):
    """Writes each tensor as out_dir/<name>.npy (<name>_rank<r>.npy when several ranks run).  Along its last axis an array
    longer than DUMP_SAMPLE / world keeps the entries at a fixed seeded sample of indices, the same in every run of the same
    size, so that the outputs of two builds can be compared entry for entry.  Integer outputs are written as floats."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    cap = DUMP_SAMPLE // world
    for name, t in arrays.items():
        n = t.shape[-1]
        if n > cap:
            idx = np.sort(np.random.default_rng(0).choice(n, cap, replace=False))
            t = t.index_select(t.dim() - 1, torch.as_tensor(idx, device=t.device))
        a = t.cpu().numpy()
        a = a.astype(np.float64 if a.dtype.itemsize == 8 else np.float32)      # int64 counts are exact in float64
        np.save(os.path.join(out_dir, name + (f"_rank{rank}" if world > 1 else "") + ".npy"), a)


# ------------------------------------------------------------------------------------------------
# GPU side
# ------------------------------------------------------------------------------------------------
def run_gpu(args):
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = bind_to_gpu_numa_node(local)   # pinned host buffers of the end-to-end leg are then allocated next to this GPU
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"      # keep NCCL's version banner off stdout: rank 0 prints ONE JSON line
        dist.init_process_group("nccl", device_id=dev)
    from fem_elastoplasticity_b200 import meshgen, distributed as fdist
    from fem_elastoplasticity_b200 import pythonFEM as api
    from fem_elastoplasticity_b200.plan import FemPlan, dp_return_map

    nx = args.nx
    et = api.LagrangeElementType.P1
    xi, wf = api.get_quadrature_volume(et)
    _, d1, d2 = api.get_local_basis_volume(et, xi)
    # weak scaling: rank r owns cell rows [r*nx, (r+1)*nx) of an nx x (nx*world) mesh plus one ghost cell row per neighbour
    if args.scaling == "strong":   # fixed total mesh (~nx x nx cells, rows rounded up to a multiple of the rank count)
        ny_global = -(-nx // world) * world
    else:                          # weak: nx x nx cells per GPU
        ny_global = nx * world
    part = fdist.StripPartition(nx, ny_global, rank, world, size_x=10.0, size_y=10.0 * ny_global / nx)
    mesh = part.local_mesh(dev)
    t_plan0 = time.perf_counter()
    P = FemPlan(mesh["elements"], mesh["coordinates"], d1, d2, wf, device=dev)
    torch.cuda.synchronize()
    t_plan = time.perf_counter() - t_plan0
    n_e_owned = part.n_e_owned
    G, Kb, eta, c = meshgen.footing_materials(P.n_int, dev)
    # synthetic state as a function of the GLOBAL element / node id: the ghost cell row a rank keeps carries its owner's
    # values, so the ranks' owned rows form ONE symmetric global matrix (per-rank seeds made K unsymmetric across the
    # interfaces in round 1 - the reason its partitioned converged solve stalled)
    Es = meshgen.synthetic_strain_global(P.n_int, 2 * nx * part.iy0, dev)
    u = meshgen.synthetic_nodal_global(P.n_n, (nx + 1) * part.iy0, dev)
    mask = part.free_owned_mask(P, mesh)
    E = P.empty(3, P.n_int)
    ep_old = torch.zeros((4, P.n_int), dtype=torch.float64, device=dev)
    rm = {}
    k_tan, F = P.empty(P.nnz), P.empty(P.n_dof)
    k_el = P.assemble_elastic(G, Kb)
    pcg = fdist.DistributedPCG(P, part, mask, peer={"auto": "auto", "nccl": False, "peer": True, "fused": "fused"}[args.halo], use_graph=not args.no_graph)
    rhs = P.empty(P.n_dof)
    from fem_elastoplasticity_b200.plan import axpby
    # the step's linear solve: CG preconditioned by a geometric multigrid V-cycle, driven to rtol (coarse operators of K_elast,
    # built once per mesh as in the Newton loop); --solver jacobi restores round 1's fixed number of Jacobi iterations
    mgs, solver_note = None, None
    if args.solver == "multigrid":
        from fem_elastoplasticity_b200.mg import MultigridPCG
        try:
            mgs = MultigridPCG(P, mask, part=part if world > 1 else None, free_mask=P.mask_u8(mesh["Q"]), degree=args.mg_degree, ratio=args.mg_ratio, **({} if args.mg_replicate_below is None else {"replicate_below": args.mg_replicate_below})).setup(k_el)
        except Exception as e:  # noqa: BLE001  (e.g. no symmetric memory on this box: every rank fails at the same collective)
            mgs, solver_note = None, f"multigrid unavailable ({type(e).__name__}: {e}); step timed with {args.pcg_iters} fixed Jacobi-PCG iterations"
            print(solver_note, file=sys.stderr)
    solve_info, last = {}, {}

    def ev():
        return torch.cuda.Event(enable_timing=True)

    phases = ("strain", "return_map", "assembly", "pcg", "criterion")
    launches = {"n": 0}

    def step(record=None):
        evs = [ev() for _ in range(len(phases) + 1)]
        evs[0].record()
        P.strain(u, out=E)
        evs[1].record()
        dp_return_map(Es, ep_old, G, Kb, eta, c, want_ep=False, out=rm)   # Ep_old is read (32 B/pt) as in the reference's Newton loop
        evs[2].record()
        P.assemble_tangent_force(rm["ds"], rm["s"], out_k=k_tan, out_f=F)
        evs[3].record()
        axpby(-1.0, F, 0.0, F, out=rhs)
        if mgs is not None:
            x, its, rel = mgs.solve(k_tan, rhs, rtol=args.rtol, maxit=args.converged_maxit)
            solve_info.update(iterations=its, relres=rel)
            n_launch = 5 + its * mgs.launches_per_iteration()
        else:
            x, its = pcg.solve(k_tan, rhs, iters=args.pcg_iters)
            n_launch = pcg.launches_last
        evs[4].record()
        last["solution"], last["energy_norms"] = x, pcg.energy_norms(k_el, x, u, rhs)
        evs[5].record()
        launches["n"] = 1 + 1 + 1 + 1 + n_launch + 3
        if record is not None:
            record.append(evs)

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for _ in range(args.warmup):
        step()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    sampler.region_begin()
    rec = []
    torch.cuda.synchronize()
    t0 = ev()
    t1 = ev()
    t0.record()
    for _ in range(args.steps):
        step(rec)
    t1.record()
    torch.cuda.synchronize()
    sampler.region_end()
    if world > 1:
        dist.barrier()
    clocks = sampler.stop() if rank == 0 else None
    total_ms = t0.elapsed_time(t1)
    per = {p: float(np.mean([e[i].elapsed_time(e[i + 1]) for e in rec])) for i, p in enumerate(phases)}
    if args.dump_outputs:                                # before anything below overwrites the step's buffers
        dump_outputs(args.dump_outputs, {"strain": E, "stress": rm["s"], "tangent_operator": rm["ds"], "plastic": rm["ind_p"],
                                         "plastic_counts": rm["counts"], "k_tangent": k_tan, "internal_force": F, **last},
                     rank, world)
    # ---- isolated kernels (same inputs, outside the step): K_tangent alone and K_elast
    def iso(fn, reps=5):
        fn()
        torch.cuda.synchronize()
        b0, b1 = ev(), ev()
        b0.record()
        for _ in range(reps):
            fn()
        b1.record()
        torch.cuda.synchronize()
        return b0.elapsed_time(b1) / reps
    true_rel = None
    if mgs is not None:                                  # true residual of the last step's solution, over all ranks
        kx = P.spmv(k_tan, mgs.x, mask=mask)
        tr = torch.stack([((rhs - kx) * mask).square().sum(), (rhs * mask).square().sum()])
        if world > 1:
            dist.all_reduce(tr)
        true_rel = float((tr[0] / tr[1]).sqrt().item())
        assert true_rel <= 10 * args.rtol, f"multigrid solve: true residual {true_rel:.2e}"
    # fixed number of Jacobi-PCG iterations on the same system: the per-iteration roofline figure of K7-K9
    t_jac = iso(lambda: pcg.solve(k_tan, rhs, iters=args.pcg_iters), reps=3)
    t_mg_cheb = t_mg_resid = t_spmv = 0.0
    if mgs is not None:                                  # the level-0 kernels of the V-cycle and the CG's SpMV, on their own
        xa, xb = mgs.v0["xa"], mgs.v0["xb"]
        xa.copy_(mgs.x)
        t_mg_cheb = iso(lambda: mgs.fine_step(k_tan, rhs, xa, xb, mode=2, step=1), reps=10)
        t_mg_resid = iso(lambda: mgs.fine_step(k_tan, rhs, xa, mgs.v0["r"], mode=1), reps=10)
        t_spmv = iso(lambda: P.spmv(k_tan, mgs.x, mask=mask, out=mgs.q), reps=10)
    t_tan_only = iso(lambda: P.assemble_tangent(rm["ds"], out=k_tan))
    t_el_only = iso(lambda: P.assemble_elastic(G, Kb, out=k_el))
    # ---- correctness carried by the run itself (N > 1): see multi_gpu_checks
    checks = multi_gpu_checks(args, P, part, mesh, pcg, k_tan, rhs, rm, d1, d2, wf, dev) if world > 1 else None
    # ---- (optional, --two-level) the same system with round 1's two-level preconditioner, for comparison
    tl_conv = None
    if args.two_level:
        from fem_elastoplasticity_b200.distributed import PCGNotConverged
        from fem_elastoplasticity_b200.twolevel import TwoLevelPCG
        tl = TwoLevelPCG(P, mask, nc=args.coarse_cells, part=part if world > 1 else None, free_mask=P.mask_u8(mesh["Q"])).setup(k_el)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        c0 = time.perf_counter()
        converged = True
        try:
            _, c_its, c_rel = tl.solve(k_tan, rhs, rtol=args.rtol, maxit=50000, check_every=50)
        except PCGNotConverged as e:
            converged, c_its, c_rel = False, e.iters, e.relres
        torch.cuda.synchronize()
        c_s = time.perf_counter() - c0
        tl_conv = {"preconditioner": f"two-level: Jacobi + {tl.grid[4]}x{tl.grid[5]} bilinear coarse grid ({tl.ncd} coarse DOFs, dense inverse)",
                   "converged": converged, "rtol": args.rtol, "iterations": c_its, "relres": c_rel, "seconds": c_s,
                   "coarse_setup_seconds": tl.setup_seconds}
        del tl
    # ---- strong scaling in the same run (N > 1): the nx x nx mesh of config 4 split over the N GPUs, same step
    strong = strong_scaling_part(args, world, rank, dev, d1, d2, wf, pcg_one_gpu_ms=None) if (world > 1 and args.scaling == "weak" and not args.no_strong) else None
    # ---- end-to-end leg: tangent assembly through the public API with HOST buffers (pinned); every step uploads its DS
    # (H2D) and downloads its K values (D2H) inside the timed region.  Two steps are in flight on two streams with
    # double-buffered device arrays, so the upload of step i+1 overlaps the download of step i (PCIe is full duplex).
    ds_host = torch.empty((9, P.n_int), dtype=torch.float64, pin_memory=True)
    ds_host.copy_(rm["ds"])
    k_host = [torch.empty(P.nnz, dtype=torch.float64, pin_memory=True) for _ in range(2)]
    ds_dev = [torch.empty((9, P.n_int), dtype=torch.float64, device=dev) for _ in range(2)]
    k_dev = [P.empty(P.nnz) for _ in range(2)]
    streams = [torch.cuda.Stream(device=dev) for _ in range(2)]
    e2e_steps = max(4, min(args.steps, 8))

    def e2e_step(i):
        j = i & 1
        with torch.cuda.stream(streams[j]):
            ds_dev[j].copy_(ds_host, non_blocking=True)
            P.assemble_tangent(ds_dev[j], out=k_dev[j])
            k_host[j].copy_(k_dev[j], non_blocking=True)

    for i in range(2):                                   # warm-up of both buffers
        e2e_step(i)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    w0 = time.perf_counter()
    for i in range(e2e_steps):
        e2e_step(i)
    torch.cuda.synchronize()
    e2e_ms = (time.perf_counter() - w0) * 1e3 / e2e_steps
    assert torch.equal(k_host[0], k_host[1]) and bool((k_host[0] == k_tan.cpu()).all())   # the downloaded result is the K_tangent
    # ---- the whole Newton step through the reference-facing facade (pythonFEM.py names, NumPy arrays in and out of every
    # call, so every stage pays its host<->device copies; the matrix stays on the device behind a DeviceMatrix handle).  One GPU.
    facade = None
    if world == 1 and not args.no_facade_step:
        U_np = u.cpu().numpy().reshape((2, -1), order="F")
        mats = [t.cpu().numpy() for t in (G, Kb, eta, c)]
        ep_np, q_np = np.zeros((4, P.n_int)), mesh["Q"].cpu().numpy()
        Kel_h = api.DeviceMatrix(P, k_el)
        e_syn = Es.cpu().numpy()

        def facade_step():
            E_np = api.strain(Kel_h, U_np)                                     # (3, n_int) NumPy out
            cp = api.construct_constitutive_problem(e_syn if args.facade_synthetic_strain else E_np, ep_np, *mats)
            Kt = api.assemble_tangent(Kel_h, cp["ds"], mode="direct", host_matrix=False)
            F_np = api.internal_force(Kel_h, cp["s"])
            dU = api.solve_increment(Kt, F_np, q_np, rtol=args.rtol, K_elast=Kel_h)
            return api.stopping_criterion(Kel_h, dU, U_np, U_np + dU), cp

        facade_step()                                                          # warm-up: multigrid set-up, graph capture
        torch.cuda.synchronize()
        f0 = time.perf_counter()
        crit, cp = facade_step()
        torch.cuda.synchronize()
        f_s = time.perf_counter() - f0
        assert np.isfinite(crit) and np.array_equal(cp["ind_p"], rm["ind_p"].cpu().numpy().astype(bool))
        nb = 8 * P.n_int
        facade = {"seconds": f_s, "melem_s": P.n_e / f_s / 1e6, "criterion": float(crit),
                  "h2d_bytes": int(2 * 8 * P.n_dof + 3 * nb + 4 * nb + 4 * nb + 9 * nb + 3 * nb + 8 * P.n_dof + 3 * 8 * P.n_dof),
                  "d2h_bytes": int(3 * nb + (4 + 9 + 4 + 1) * nb + P.n_int + 2 * 8 * P.n_dof),
                  "what": "pythonFEM facade, NumPy in/out per call: strain -> construct_constitutive_problem -> assemble_tangent(direct, DeviceMatrix) "
                          "-> internal_force -> solve_increment (multigrid CG to rtol) -> stopping_criterion; the caller's arrays (U, materials, Ep, strain) are pageable, "
                          "the arrays the facade returns (and gets back as the next call's input) are page-locked"}
        del Kel_h, cp
    # ---- reduce over ranks (max time)
    vec = torch.tensor([total_ms, per["strain"], per["return_map"], per["assembly"], per["pcg"], per["criterion"], e2e_ms,
                        t_tan_only, t_el_only, t_jac, t_mg_cheb, t_mg_resid, t_spmv], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(vec, op=dist.ReduceOp.MAX)
    total_ms, t_strain, t_rm, t_asm, t_pcg, t_crit, e2e_ms, t_tan_only, t_el_only, t_jac, t_mg_cheb, t_mg_resid, t_spmv = [float(v) for v in vec.cpu()]
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    n_e_tot = n_e_owned * world
    n_int_tot = n_e_tot
    n_dof_rank, nnz_rank = P.n_dof, P.nnz
    peak, peak_src = measured_peak()
    ms_step = total_ms / args.steps
    gbs = lambda nbytes, ms: nbytes / (ms * 1e-3) / 1e9  # noqa: E731
    algo = {
        "tangent_only": 212.0 * P.n_e, "elastic": 156.0 * P.n_e,
        "assembly": 212.0 * P.n_e + 24.0 * P.n_int + 8.0 * P.n_dof,
        "return_map": 193.0 * P.n_int,
        "strain": 12.0 * P.n_e + 8.0 * P.n_dof + 24.0 * P.n_int,
        "pcg_iter": 12.0 * nnz_rank + 148.0 * n_dof_rank,
        "spmv": 12.0 * nnz_rank + 4.0 * (n_dof_rank + 1) + 16.0 * n_dof_rank,
        # bytes THIS implementation has to move (block pattern: 8 B/nnz of values + one 16-bit block position per 4 values,
        # node pointers, x once, y once, mask; Jacobi-PCG vector kernels: 10 vector passes) - ncu agrees within 4 % (profiles/r2c)
        "spmv_own": 8.5 * nnz_rank + (4.0 + 16.0 + 16.0 + 2.0) * P.n_n,
        "pcg_iter_own": 8.5 * nnz_rank + 38.0 * P.n_n + 80.0 * n_dof_rank,
        # level-0 multigrid step: FP32 values (4 B/nnz) + block positions + node pointers + b, D^-1 (2x2 blocks), d, x in, d, x out
        "mg_cheb": (4.5 if (mgs is not None and mgs.k32 is not None) else 8.5) * nnz_rank + 4.0 * P.n_n + 56.0 * n_dof_rank,
        "mg_resid": (4.5 if (mgs is not None and mgs.k32 is not None) else 8.5) * nnz_rank + 6.0 * P.n_n + 24.0 * n_dof_rank,
    }
    pcg_ms_iter = t_jac / max(args.pcg_iters, 1)
    conv = None
    if mgs is not None:
        its = int(solve_info["iterations"])
        conv = {"preconditioner": f"geometric multigrid V-cycle: {mgs.n_levels + 1} levels, Chebyshev smoother of degree {mgs.degree} on block Jacobi (2x2 node blocks; interval lambda_max/{mgs.ratio:g}), "
                                  f"Galerkin coarse operators of K_elast, dense solve on {2 * mgs.lv[-1]['n']} DOFs",
                "converged": True, "rtol": args.rtol, "iterations": its, "relres": solve_info["relres"], "true_relres": true_rel,
                "seconds": t_pcg * 1e-3, "ms_per_iteration": t_pcg / max(its, 1), "setup_seconds": mgs.setup_seconds,
                "levels": [[mgs.lattice[4], mgs.lattice[5]]] + [[lv["nxn"], lv["N"]] for lv in mgs.lv],
                "distributed_levels": int(sum(1 for lv in mgs.lv if not lv["rep"])) if world > 1 else 0,
                "cuda_graph": bool(mgs._graph is not None),
                "history": "point-Jacobi 57 500 iterations / 41.7 s, two-level 1 900 iterations / 1.77 s on the same 16M-element system (round 1 / profiles/r2j)",
                "two_level": tl_conv}
    ncu_traffic = {}
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            ncu_traffic = json.load(f)
    except Exception:
        pass
    asm_roof = {"kernel": "assemble_rows_tmap_kernel<TANGENT,FORCE> (K_tangent + internal force, one pass, TMA-staged)",
                "achieved": gbs(algo["assembly"], t_asm), "frac": gbs(algo["assembly"], t_asm) / peak, "ms": t_asm,
                "algorithmic_bytes": algo["assembly"], "traffic": ncu_traffic.get("assemble_rows_kernel"),
                "share_of_step": t_asm / ms_step}
    if mgs is not None:
        # the dominant kernel of the converged step: the level-0 Chebyshev step of the V-cycle (2*degree - 1 launches per CG
        # iteration), the smoother's vector updates fused into the epilogue of the block-CSR SpMV
        n_cheb = (2 * mgs.degree - 1) * int(solve_info["iterations"]) + 2 * mgs.degree - 1
        roof = {"bound": "hbm", "kernel": "mg_fine_stream_kernel<CHEB> (level-0 Chebyshev smoothing step of the multigrid V-cycle: block-CSR SpMV streamed through shared memory by a producer warp, "
                                          f"{'FP32' if mgs.k32 is not None else 'FP64'} matrix copy + fused vector updates)",
                "achieved": gbs(algo["mg_cheb"], t_mg_cheb), "peak": peak, "unit": "GB/s", "frac": gbs(algo["mg_cheb"], t_mg_cheb) / peak,
                "traffic": ncu_traffic.get("mg_fine_stream_kernel_cheb"), "peak_source": peak_src, "algorithmic_bytes_per_launch": algo["mg_cheb"],
                "ms_per_launch": t_mg_cheb, "launches_per_step": n_cheb, "share_of_step": n_cheb * t_mg_cheb / ms_step,
                "frac_of_8TBs_nominal": gbs(algo["mg_cheb"], t_mg_cheb) / 8000.0,
                "assembly": asm_roof}
    else:
        roof = {"bound": "hbm", "kernel": asm_roof["kernel"], "achieved": asm_roof["achieved"], "peak": peak, "unit": "GB/s", "frac": asm_roof["frac"],
                "traffic": asm_roof["traffic"], "peak_source": peak_src, "algorithmic_bytes_per_launch": algo["assembly"],
                "frac_of_8TBs_nominal": asm_roof["achieved"] / 8000.0}
    rooflines = {k: {"achieved": gbs(algo[a], ms), "frac": gbs(algo[a], ms) / peak, "ms": ms, "algorithmic_bytes": algo[a]}
                 for k, a, ms in (("dp_return_map", "return_map", t_rm), ("strain", "strain", t_strain),
                                  ("assemble_tangent_force(in step)", "assembly", t_asm),
                                  ("assemble_tangent_only(isolated)", "tangent_only", t_tan_only),
                                  ("assemble_elastic(isolated)", "elastic", t_el_only),
                                  ("pcg_iteration(spmv+2 vector kernels)", "pcg_iter", pcg_ms_iter),
                                  ("pcg_iteration, bytes of this implementation", "pcg_iter_own", pcg_ms_iter),
                                  ("criterion(3 spmv)", "spmv", t_crit / 3.0)) if ms > 0}
    if mgs is not None:
        rooflines.update({k: {"achieved": gbs(algo[a], ms), "frac": gbs(algo[a], ms) / peak, "ms": ms, "algorithmic_bytes": algo[a]}
                          for k, a, ms in (("mg_fine_step_cheb(isolated)", "mg_cheb", t_mg_cheb), ("mg_fine_step_residual(isolated)", "mg_resid", t_mg_resid),
                                           ("spmv(isolated), CSR bytes", "spmv", t_spmv), ("spmv(isolated), bytes of this implementation", "spmv_own", t_spmv))})
    line = {
        "metric": METRIC, "value": n_e_tot / (t_asm * 1e-3) / 1e6, "unit": "Melem/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"config {4 if (world == 1 or args.scaling == 'strong') else 5}: synthetic uniform P1 mesh {nx}x{ny_global} cells, {n_e_tot} elements "
                               f"({n_e_owned} per GPU, strip partition), DP return map + tangent assembly + PCG",
                   "n_elements": n_e_tot, "n_dof_per_gpu": n_dof_rank, "nnz_per_gpu": nnz_rank,
                   "step_solver": (f"CG + geometric multigrid V-cycle to rtol {args.rtol:g} ({int(solve_info['iterations'])} iterations)" if mgs is not None
                                   else f"{args.pcg_iters} fixed Jacobi-PCG iterations (truncated solve)"),
                   "pcg_iters_per_step": int(solve_info["iterations"]) if mgs is not None else args.pcg_iters,
                   "jacobi_iterations_timed_for_the_roofline": args.pcg_iters,
                   "preconditioner": "multigrid" if mgs is not None else "jacobi", "pcg_cuda_graph": bool(pcg._graph is not None),
                   "halo": ("fused iteration: halo + both reductions as nvlink peer stores/flags inside the 3 PCG kernels (symmetric memory)" if getattr(pcg, "fused", False)
                            else "nvlink peer stores fused into the p-update kernel (symmetric memory), nccl all-reduces" if pcg.peer is not None
                            else ("none (1 GPU)" if world == 1 else "nccl send/recv + all-reduces")), "plastic_fraction": float(rm["ind_p"].double().mean().item()),
                   "l2": "inputs larger than L2 (>=1 GB per array vs 126 MB), no flush needed",
                   "plan_build_s": t_plan, "plan_bytes": P.bytes},
        "parts": {"tangent_assembly_melem_s": n_e_tot / (t_asm * 1e-3) / 1e6, "return_map_mpts_s": n_int_tot / (t_rm * 1e-3) / 1e6,
                  "pcg_newton_s_per_step": ms_step * 1e-3, "pcg_ms_per_iter": pcg_ms_iter, "strain_ms": t_strain, "criterion_ms": t_crit,
                  "assembly_ms": t_asm, "return_map_ms": t_rm, "tangent_only_isolated_ms": t_tan_only,
                  "tangent_only_isolated_melem_s": n_e_tot / (t_tan_only * 1e-3) / 1e6,
                  "elastic_isolated_melem_s": n_e_tot / (t_el_only * 1e-3) / 1e6, "newton_step_melem_s": n_e_tot / (ms_step * 1e-3) / 1e6,
                  **({} if strong is None else dict(strong, strong_speedup_vs_weak_step=ms_step / strong["strong_step_ms"]))},
        "pcg_converged_solve": conv, "multi_gpu_checks": checks,
        "newton_step_converged_s": (None if conv is None else ms_step * 1e-3),
        "roofline": roof, "rooflines": rooflines, "clocks": clocks,
        "e2e": {"value": n_e_tot / (e2e_ms * 1e-3) / 1e6, "unit": "Melem/s", "h2d_bytes_per_step": int(72 * P.n_int),
                "d2h_bytes_per_step": int(8 * P.nnz), "what": "FemPlan.assemble_tangent: pinned host DS -> device -> kernel -> pinned host K values, every step; two steps in flight "
                        "(double-buffered, H2D of step i+1 overlaps D2H of step i)", "steps": e2e_steps},
        "e2e_step": facade, "host_numa_binding": numa, "solver_note": solver_note,
        "gpu_launches": int(launches["n"] * args.steps),
    }
    if world == 1 and not args.no_cpu_baseline:
        # SURVEY 8(d): 100 k elements (config 1's size), 0.5 M and 1 M; rates are per element, the largest sample is the headline
        sizes = []
        for cnx in sorted({224, args.cpu_nx, 707}):
            r = cpu_reference_pass(cnx, args.pcg_iters, 1, 0)
            sizes.append({"n_elements": r["n_e"], "tangent_assembly_melem_s": r["n_e"] / r["t"]["tangent"] / 1e6,
                          "elastic_assembly_melem_s": r["n_e"] / r["t_elastic"] / 1e6, "return_map_mpts_s": r["n_e"] / r["t"]["return_map"] / 1e6,
                          "pcg_ms_per_iter": 1e3 * r["t"]["pcg"] / max(args.pcg_iters, 1),
                          "newton_step_fixed_iterations_s": r["t"]["step"]})
        line["cpu_baseline"] = {"value": sizes[-1]["tangent_assembly_melem_s"], "unit": "Melem/s", "cores": 1, "kind": "port",
                                "sample": f"oracle port of Plasticity2D_DP/pythonFEM.py:1047-1050 on {sizes[-1]['n_elements']} elements "
                                          f"(1/{max(1, n_e_tot // sizes[-1]['n_elements'])} of the workload; the reference's assembly needs ~2.1 KB "
                                          f"of host memory per element, 34 GB at 16M); host has {os.cpu_count()} cores, the reference path is "
                                          "single-threaded; port vs the reference itself (build container, 204 800 elements): tangent 1.23 vs 1.28 "
                                          "Melem/s, return map 1.09 vs 1.65 Mpts/s (BASELINE.md)",
                                "return_map_mpts_s": sizes[-1]["return_map_mpts_s"], "pcg_ms_per_iter": sizes[-1]["pcg_ms_per_iter"],
                                "newton_step_s": sizes[-1]["newton_step_fixed_iterations_s"], "sizes": sizes}
    emit(line)
    if world > 1:
        dist.destroy_process_group()


_JSON_FD = 1


def emit(line):
    """The ONE JSON line, on the real stdout (see main)."""
    os.write(_JSON_FD, (json.dumps(line) + "\n").encode())


def main():
    # stdout carries exactly one JSON line: anything libraries print there (NCCL's version banner comes from C code, at
    # the WARN level too) is sent to stderr by pointing fd 1 at fd 2 for the duration of the run
    global _JSON_FD
    sys.stdout.flush()
    _JSON_FD = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--nx", type=int, default=2828, help="cells per side per GPU (2828 -> 15 995 168 elements, config 4)")
    ap.add_argument("--pcg-iters", type=int, default=50)
    ap.add_argument("--cpu-nx", type=int, default=500, help="mesh side of the bounded CPU sample")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: nx x nx cells per GPU (config 5 at 8 GPUs); strong: one nx x nx mesh split over the GPUs")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--solver", default="multigrid", choices=["multigrid", "jacobi"],
                    help="linear solve of the step: multigrid = CG + V-cycle to --rtol (a converged Newton step); jacobi = --pcg-iters fixed iterations")
    ap.add_argument("--rtol", type=float, default=1e-10)
    ap.add_argument("--mg-degree", type=int, default=2)
    ap.add_argument("--mg-ratio", type=float, default=16.0)
    ap.add_argument("--mg-replicate-below", type=int, default=None, help="multigrid levels with at most this many nodes are replicated on every rank (default: mg.py's)")
    ap.add_argument("--no-facade-step", action="store_true", help="skip the whole-step timing through the pythonFEM facade (one GPU)")
    ap.add_argument("--facade-synthetic-strain", action="store_true", default=True, help=argparse.SUPPRESS)
    ap.add_argument("--two-level", action="store_true", help="also solve the step's system with the two-level preconditioner of round 1")
    ap.add_argument("--coarse-cells", type=int, default=64)
    ap.add_argument("--converged-maxit", type=int, default=400, help="iteration cap of the multigrid solve")
    ap.add_argument("--no-strong", action="store_true", help="skip the strong-scaling part of an N > 1 run")
    ap.add_argument("--halo", default="auto", choices=["auto", "nccl", "peer", "fused"], help="multi-GPU exchanges of the PCG: fused = inside the kernels over NVLink peer memory; auto = fused, NCCL if symmetric memory is unavailable")
    ap.add_argument("--no-graph", action="store_true", help="launch the PCG iterations eagerly instead of replaying a CUDA graph")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the arrays the last one computed as DIR/<name>.npy "
                                                           "(float64, or float32 for flags; a fixed sample of each larger array, 41 MB at most)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl b200)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
