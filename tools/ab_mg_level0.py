"""A/B of the multigrid V-cycle's level 0 on the bench's 16M-element system (nx = 2828, one GPU): the FP32 block-CSR copy
streamed through shared memory (mg_fine_stream_kernel) against the symmetric FP32 lattice stencil (mg_fine_lattice_kernel).

    python tools/ab_mg_level0.py [--nx 2828] [--reps 25] [--solves 4] [--out results/ab_mg_level0.json]

Prints, per variant: ms of one Chebyshev step and one residual step (CUDA events, batches of 10 launches, the variants
alternating rep by rep), the bytes per pass computed from the shapes, the achieved GB/s; ms, iterations and ms per
iteration of whole solves to rtol 1e-10 (alternating); the largest relative difference of the solutions; and, as a probe of
what one thread per node sustains on this card, the level-1 smoother kernel mg_stencil_kernel<MG_CHEB, float, SYM> timed
with torch.profiler inside V-cycles.  The working set (> 1.4 GB per pass) is far larger than the 126 MB L2."""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from fem_elastoplasticity_b200 import _lib, meshgen, mg, pythonFEM as api  # noqa: E402
from fem_elastoplasticity_b200 import distributed as fdist  # noqa: E402
from fem_elastoplasticity_b200.plan import FemPlan, dp_return_map  # noqa: E402


def card():
    props = torch.cuda.get_device_properties(0)
    try:
        smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()
    except (OSError, subprocess.SubprocessError) as e:
        smi = [f"nvidia-smi unavailable: {e}"]
    return {"name": props.name, "sm_count": props.multi_processor_count, "nvidia_smi": smi[0] if smi else ""}


def lattice(on):
    _lib.call("fem_set_tuning", b"mg_fine_lattice", 0 if on else 2)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nx", type=int, default=2828)
    ap.add_argument("--reps", type=int, default=25)
    ap.add_argument("--solves", type=int, default=4)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("ab_mg_level0.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    res = {"card": card(), "nx": args.nx}
    print("card:", res["card"], flush=True)

    et = api.LagrangeElementType.P1
    xi, wf = api.get_quadrature_volume(et)
    _, d1, d2 = api.get_local_basis_volume(et, xi)
    part = fdist.StripPartition(args.nx, args.nx, 0, 1, size_x=10.0, size_y=10.0)
    mesh = part.local_mesh(dev)
    P = FemPlan(mesh["elements"], mesh["coordinates"], d1, d2, wf, device=dev)
    G, Kb, eta, c = meshgen.footing_materials(P.n_int, dev)
    k_el = P.assemble_elastic(G, Kb)
    r = dp_return_map(meshgen.synthetic_strain_global(P.n_int, 0, dev), None, G, Kb, eta, c)
    k_tan, F = P.assemble_tangent_force(r["ds"], r["s"])
    rhs = -F
    mask = part.free_owned_mask(P, mesh)
    M = mg.MultigridPCG(P, mask, free_mask=P.mask_u8(mesh["Q"])).setup(k_el)
    res["fine_lattice"] = M.fine_lattice
    print(f"n_n {P.n_n}  nnz {P.nnz}  levels {M.n_levels + 1}  level 0 on the lattice: {M.fine_lattice}", flush=True)
    if not M.fine_lattice:
        raise SystemExit("the bench mesh did not qualify for the lattice stencil")

    # ---- whole solves, alternating (each variant captures its own CUDA graph)
    sols, solves = {}, {"csr": [], "lattice": []}
    graphs = {}
    for rep in range(args.solves + 1):
        for name in ("csr", "lattice"):
            lattice(name == "lattice")
            M._graph = graphs.get(name)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            x, its, rel = M.solve(k_tan, rhs, rtol=1e-10)
            e1.record()
            torch.cuda.synchronize()
            graphs[name] = M._graph
            if rep == 0:                                  # warm-up (graph capture, module loads)
                sols[name] = (x.clone(), its, rel)
                continue
            solves[name].append((e0.elapsed_time(e1), its))
    lattice(True)
    xc, xl = sols["csr"][0], sols["lattice"][0]
    diff = float((xl - xc).abs().max() / xc.abs().max())
    kx = P.spmv(k_tan, xl, mask=mask)
    true_rel = float(((rhs - kx) * mask).norm() / (rhs * mask).norm())
    res["solve"] = {}
    for name in ("csr", "lattice"):
        ms = [t for t, _ in solves[name]]
        its = solves[name][0][1]
        res["solve"][name] = {"ms_median": statistics.median(ms), "ms_min": min(ms), "ms_max": max(ms), "iterations": its,
                              "ms_per_iteration": statistics.median(ms) / its, "relres": sols[name][2]}
        print(f"solve {name:8s}: {statistics.median(ms):8.3f} ms (min {min(ms):.3f}, max {max(ms):.3f}), {its} iterations, "
              f"{statistics.median(ms) / its:.4f} ms/iteration", flush=True)
    res["solution_max_rel_diff"], res["lattice_true_relres"] = diff, true_rel
    print(f"max |x_lattice - x_csr| / max |x_csr| = {diff:.3e}; true relative residual of the lattice solution {true_rel:.3e}", flush=True)

    # ---- single level-0 steps (the planes and k32 hold k_tan after the solves)
    xa, xb, rr = M.v0["xa"], M.v0["xb"], M.v0["r"]
    xa.copy_(M.x)
    steps = {
        ("cheb", "csr"): lambda: M.fine_step(k_tan, rhs, xa, xb, mode=2, step=1),
        ("cheb", "lattice"): lambda: M.fine_step_lattice(rhs, xa, xb, mode=2, step=1),
        ("resid", "csr"): lambda: M.fine_step(k_tan, rhs, xa, rr, mode=1),
        ("resid", "lattice"): lambda: M.fine_step_lattice(rhs, xa, rr, mode=1),
    }
    n_n, n_dof, nnz = P.n_n, P.n_dof, P.nnz
    # bytes from the shapes: block-CSR values 4 B + block positions 0.5 B per nonzero, row pointers 4 B per node; planes 64 B
    # per node; vectors per DOF: b, D^-1 (2), d, x read and d, out written (Chebyshev), b, x read and r written (residual)
    bytes_ = {("cheb", "csr"): 4.5 * nnz + 4.0 * n_n + 56.0 * n_dof, ("cheb", "lattice"): 64.0 * n_n + 56.0 * n_dof,
              ("resid", "csr"): 4.5 * nnz + 6.0 * n_n + 24.0 * n_dof, ("resid", "lattice"): 66.0 * n_n + 24.0 * n_dof}
    for fn in steps.values():
        fn()
    torch.cuda.synchronize()
    times = {k: [] for k in steps}
    batch = 10
    for _ in range(args.reps):
        for k, fn in steps.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(batch):
                fn()
            e1.record()
            torch.cuda.synchronize()
            times[k].append(e0.elapsed_time(e1) / batch)
    res["steps"] = {}
    for k, ts in times.items():
        med = statistics.median(ts)
        gbs = bytes_[k] / (med * 1e-3) / 1e9
        res["steps"][f"{k[0]}_{k[1]}"] = {"ms_median": med, "ms_min": min(ts), "ms_max": max(ts), "bytes": bytes_[k], "GB_per_s": gbs,
                                          "bytes_per_node": bytes_[k] / n_n}
        print(f"{k[0]:5s} {k[1]:8s}: {med:.4f} ms (min {min(ts):.4f}, max {max(ts):.4f})  {bytes_[k] / 1e9:.3f} GB "
              f"({bytes_[k] / n_n:.0f} B/node)  {gbs:7.0f} GB/s", flush=True)

    # ---- level-1 probe: mg_stencil_kernel<MG_CHEB, float, SYM> (one thread per node, 19 FP32 planes) inside V-cycles
    from torch.profiler import ProfilerActivity, profile
    z = torch.zeros_like(rhs)
    nv = 5
    M.vcycle(k_tan, M.r, z)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(nv):
            M.vcycle(k_tan, M.r, z)
        torch.cuda.synchronize()
    durs = {}
    for e in prof.events():
        if e.device_type.name == "CUDA":
            durs.setdefault(e.name, []).append(e.device_time_total)
    st = sorted((d for n, ds in durs.items() if "mg_stencil_kernel<2, float, true>" in n for d in ds), reverse=True)
    l1 = M.lv[0]
    if len(st) >= 3 * nv:
        us = statistics.median(st[:3 * nv])              # level 1: three Chebyshev sweeps per V-cycle, the longest ones
        b1 = 76.0 * l1["n"] + 112.0 * l1["n"]
        res["level1_probe"] = {"nodes": l1["n"], "us_median": us, "bytes": b1, "GB_per_s": b1 / (us * 1e-6) / 1e9}
        print(f"level-1 probe mg_stencil_kernel<CHEB, float, SYM>: {l1['n']} nodes, {us:.1f} us, {b1 / 1e6:.1f} MB, "
              f"{b1 / (us * 1e-6) / 1e9:.0f} GB/s", flush=True)
    else:
        print("level-1 probe: kernel not found in the trace:", sorted(durs)[:40], flush=True)
    for n, ds in sorted(durs.items(), key=lambda kv: -sum(kv[1]))[:12]:
        print(f"  {sum(ds) / nv:9.1f} us per V-cycle  {len(ds) // nv:3d}x  {n[:120]}")
    if args.out:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
