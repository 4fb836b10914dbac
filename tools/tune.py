"""On-GPU launch-shape sweep (CUDA events, inputs >> L2): python tools/tune.py [--nx 2828] > gpurun_out/tune.json"""
import argparse
import ctypes as C
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from fem_elastoplasticity_b200 import _lib, meshgen  # noqa: E402
from fem_elastoplasticity_b200 import pythonFEM as api  # noqa: E402
from fem_elastoplasticity_b200.plan import FemPlan, dp_return_map  # noqa: E402


def knob(key, val):
    _lib.call("fem_set_tuning", key.encode(), int(val))


def timeit(fn, reps=10, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nx", type=int, default=2828)
    args = ap.parse_args()
    et = api.LagrangeElementType.P1
    xi, wf = api.get_quadrature_volume(et)
    _, d1, d2 = api.get_local_basis_volume(et, xi)
    m = meshgen.square_mesh_p1(args.nx, args.nx)
    P = FemPlan(m["elements"], m["coordinates"], d1, d2, wf)
    G, Kb, eta, c = meshgen.footing_materials(P.n_int)
    Es = meshgen.synthetic_strain(P.n_int)
    ep = torch.zeros((4, P.n_int), dtype=torch.float64, device="cuda")
    out = {"n_e": P.n_e, "nnz": P.nnz, "n_dof": P.n_dof, "max_degree": P.max_degree, "stage": P.stage_info()}
    rm = {}
    res = {}
    res["return_map_ms"] = timeit(lambda: dp_return_map(Es, ep, G, Kb, eta, c, want_ep=False, want_counts=True, out=rm))
    r = dp_return_map(Es, ep, G, Kb, eta, c, want_ep=False, out=rm)
    kel_ref = None
    k, F = P.empty(P.nnz), P.empty(P.n_dof)
    for v, name in ((2, "reg"), (6, "tmapipe"), (0, "default")):
        knob("assemble_variant", v)
        res[f"assemble_elastic_{name}_ms"] = timeit(lambda: P.assemble_elastic(G, Kb, out=k))
        kel = k.clone()
        res[f"assemble_tangent_{name}_ms"] = timeit(lambda: P.assemble_tangent(r["ds"], out=k))
        kt = k.clone()
        res[f"assemble_tangent_force_{name}_ms"] = timeit(lambda: P.assemble_tangent_force(r["ds"], r["s"], out_k=k, out_f=F))
        res[f"assemble_tangent_ref_{name}_ms"] = timeit(lambda: P.assemble_tangent_ref(r["ds"], G, Kb, kel, out=k))
        if kel_ref is None:
            kel_ref, kt_ref, F_ref = kel, kt, F.clone()
        else:
            res[f"{name}_equals_reg_bits"] = bool(torch.equal(kel, kel_ref) and torch.equal(kt, kt_ref) and torch.equal(F, F_ref))
    knob("assemble_variant", 0)
    res["internal_force_ms"] = timeit(lambda: P.internal_force(r["s"], out=F))
    u = torch.randn(P.n_dof, dtype=torch.float64, device="cuda")
    E = P.empty(3, P.n_int)
    res["strain_ms"] = timeit(lambda: P.strain(u, out=E))
    y = P.empty(P.n_dof)
    mask = P.mask_u8(m["Q"])
    dot = torch.zeros(1, dtype=torch.float64, device="cuda")
    y_ref = None
    # 1: round-1 kernel (x gathered through L1/L2); 2: x staged in shared memory, matrix through registers; 0: every operand
    # streamed through shared memory by bulk async copies (one persistent CTA per SM)
    for staged, name, bpss in ((1, "gather", (8,)), (2, "staged", (2,)), (0, "stream", (1,))):
        knob("spmv_staged", staged)
        for bps in bpss:
            knob("spmv_blocks_per_sm", bps)
            res[f"spmv_{name}_b{bps}_ms"] = timeit(lambda: P.spmv(kel_ref, u, mask=mask, out=y, dot=dot))
            if y_ref is None:
                y_ref = y.clone()
            else:
                res[f"spmv_{name}_b{bps}_maxdiff"] = float((y - y_ref).abs().max() / y_ref.abs().max())
    knob("spmv_staged", 0), knob("spmv_blocks_per_sm", 0)
    out["results"] = res
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
