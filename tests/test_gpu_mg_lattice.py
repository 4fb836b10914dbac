"""Level 0 of the multigrid V-cycle on the lattice (csrc/mg.cu: mg_to_f32_lattice_kernel, mg_fine_lattice_kernel): the
symmetric FP32 stencil against the FP32 block-CSR copy it replaces in the smoother and the residual, the V-cycle built on
it, and the fallback to the block-CSR path on meshes that do not qualify."""
import os

import numpy as np
import pytest

from oracle import fem_oracle as fo

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def fem():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device")
    from fem_elastoplasticity_b200 import _lib, meshgen, mg, plan
    return {"torch": torch, "plan": plan, "mg": mg, "meshgen": meshgen, "lib": _lib}


def p1_tables():
    xi, wf = fo.quadrature_volume(fo.ElementType.P1)
    _, d1, d2 = fo.local_basis_volume(fo.ElementType.P1, xi)
    return d1, d2, wf


def system(fem, nx, ny, size_y=10.0, tangent=True):
    from fem_elastoplasticity_b200.plan import dp_return_map
    d1, d2, wf = p1_tables()
    m = fem["meshgen"].square_mesh_p1(nx, ny, 10.0, size_y)
    P = fem["plan"].FemPlan(m["elements"], m["coordinates"], d1, d2, wf)
    G, Kb, eta, c = fem["meshgen"].footing_materials(P.n_int)
    k_el = P.assemble_elastic(G, Kb)
    r = dp_return_map(fem["meshgen"].synthetic_strain(P.n_int), None, G, Kb, eta, c)
    k_tan, F = P.assemble_tangent_force(r["ds"], r["s"])
    return P, m, k_el, (k_tan if tangent else k_el), F, P.mask_u8(m["Q"])


def set_lattice(fem, on):
    fem["lib"].call("fem_set_tuning", b"mg_fine_lattice", 0 if on else 2)


def test_planes_equal_the_block_csr_copy(fem):
    torch, mg = fem["torch"], fem["mg"]
    P, m, k_el, k, _, mask = system(fem, 333, 211, 6.0)
    M = mg.MultigridPCG(P, mask).setup(k_el)
    assert M.fine_lattice and M.lat32_nw == 1              # square_mesh_p1: diagonals from (ix+1, iy) to (ix, iy+1)
    M.k32.fill_(float("nan"))
    M.to_f32(k)
    assert torch.equal(M.k32, k.to(torch.float32))          # the block-CSR copy is what fem_mg_to_f32 writes
    LX, n, st = 334, P.n_n, M.lat32_stride
    A = P.to_scipy_csr(k).tocsr()
    a = np.arange(n)
    planes = M.k32s.view(16, st)[:, :n].cpu().numpy()
    for slot, off in enumerate((0, 1, LX, LX - 1)):
        b = a + off
        ok = b < n
        bb = np.where(ok, b, 0)
        for q in range(4):
            want = np.asarray(A[2 * a + q // 2, 2 * bb + q % 2]).ravel()
            want = np.where(ok, want, 0.0).astype(np.float32)
            got = planes[4 * slot + q]
            assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), (slot, q)


def test_lattice_steps_agree_with_block_csr(fem):
    torch, mg = fem["torch"], fem["mg"]
    for tangent in (False, True):
        P, m, k_el, k, _, mask = system(fem, 333, 211, 6.0, tangent)
        M = mg.MultigridPCG(P, mask).setup(k_el)
        assert M.fine_lattice
        M.block_jacobi(k)
        M.to_f32(k)
        g = torch.Generator(device="cuda").manual_seed(4)
        rnd = lambda: torch.randn(P.n_dof, dtype=torch.float64, device="cuda", generator=g) * mask  # noqa: E731
        b, x, d0 = rnd(), rnd(), rnd()
        outs = []
        for lat in (False, True):
            M.v0["d"].copy_(d0)
            out, res, dot = torch.zeros_like(x), torch.zeros_like(x), torch.zeros(1, dtype=torch.float64, device="cuda")
            if lat:
                M.fine_step_lattice(b, x, out, mode=2, step=1, dot=dot)
                M.fine_step_lattice(b, x, res, mode=1)
            else:
                M.fine_step(k, b, x, out, mode=2, step=1, dot=dot)
                M.fine_step(k, b, x, res, mode=1)
            outs.append((out.clone(), M.v0["d"].clone(), res.clone(), float(dot.item())))
        for u, v in zip(outs[0][:3], outs[1][:3]):
            assert float((u - v).abs().max()) <= 1e-6 * float(u.abs().max())
        assert abs(outs[0][3] - outs[1][3]) <= 1e-6 * abs(outs[0][3])
        r_ref = (b - P.spmv(k, x)) * mask
        d_ref = M.desc.c1[1] * d0 + M.desc.c2[1] * M.block_apply(M.minv, r_ref)
        out, d, res, dot = outs[1]
        assert float((res - r_ref).abs().max()) <= 1e-6 * float(r_ref.abs().max())
        assert float((d - d_ref).abs().max()) <= 1e-6 * float(d_ref.abs().max())
        assert float((out - (x + d_ref)).abs().max()) <= 1e-6 * float((x + d_ref).abs().max())
        assert abs(dot - float(b @ (x + d_ref))) <= 1e-6 * abs(float(b @ (x + d_ref)))
        # masked DOFs stay zero; the step is reproducible bit for bit
        assert not bool(((out != 0) & (mask == 0)).any())
        M.v0["d"].copy_(d0)
        out2, dot2 = torch.zeros_like(x), torch.zeros(1, dtype=torch.float64, device="cuda")
        M.fine_step_lattice(b, x, out2, mode=2, step=1, dot=dot2)
        assert torch.equal(out2, out) and float(dot2.item()) == dot


def test_lattice_vcycle_is_symmetric(fem):
    torch, mg = fem["torch"], fem["mg"]
    P, m, k_el, k, _, mask = system(fem, 120, 90, 7.5)
    M = mg.MultigridPCG(P, mask).setup(k_el)
    assert M.fine_lattice
    M.block_jacobi(k)
    M.to_f32(k)
    g = torch.Generator(device="cuda").manual_seed(9)
    u, v = (torch.randn(P.n_dof, dtype=torch.float64, device="cuda", generator=g) * mask for _ in range(2))
    zu, zv = torch.zeros_like(u), torch.zeros_like(v)
    M.vcycle(k, u, zu)
    M.vcycle(k, v, zv)
    a, b = float(u @ zv), float(v @ zu)
    assert abs(a - b) <= 1e-10 * abs(a)


@pytest.mark.parametrize("nx", [96, 384])
def test_lattice_solve_converges_like_block_csr(fem, nx):
    torch, mg = fem["torch"], fem["mg"]
    P, m, k_el, k, F, mask = system(fem, nx, nx)
    M = mg.MultigridPCG(P, mask).setup(k_el)
    assert M.fine_lattice
    its = {}
    try:
        for lat in (False, True):
            set_lattice(fem, lat)
            M._graph = None
            x, its[lat], rel = M.solve(k, -F, rtol=1e-10)
            x = x.clone()
            true = float(((-F - P.spmv(k, x)) * mask).norm() / (F * mask).norm())
            assert rel <= 1e-10 and true <= 2e-10, (lat, rel, true)
        x2, n2, _ = M.solve(k, -F, rtol=1e-10)
        assert n2 == its[True] and torch.equal(x2, x)        # two solves, the same bits
    finally:
        set_lattice(fem, True)
    assert abs(its[True] - its[False]) <= 1, its


def test_fallback_to_block_csr(fem):
    """A node numbering that is not the lattice's keeps the block-CSR level 0 (switching the stencil on changes nothing);
    the unstructured tsx mesh is still refused."""
    torch, mg = fem["torch"], fem["mg"]
    d1, d2, wf = p1_tables()
    m = fem["meshgen"].square_mesh_p1(64, 48, 10.0, 7.5)
    n = m["coordinates"].shape[1]
    perm = torch.randperm(n, generator=torch.Generator().manual_seed(5)).cuda()   # new id -> old id
    inv = torch.empty_like(perm)
    inv[perm] = torch.arange(n, device="cuda")
    elem = inv[m["elements"].long()].to(torch.int32)
    coord, q = m["coordinates"][:, perm].contiguous(), m["Q"][:, perm].contiguous()
    P = fem["plan"].FemPlan(elem, coord, d1, d2, wf)
    G, Kb, _, _ = fem["meshgen"].footing_materials(P.n_int)
    k = P.assemble_elastic(G, Kb)
    mask = P.mask_u8(q)
    M = mg.MultigridPCG(P, mask).setup(k)
    assert not M.fine_lattice and M.desc.lat32 is None
    F = torch.randn(P.n_dof, dtype=torch.float64, device="cuda", generator=torch.Generator(device="cuda").manual_seed(2)) * mask
    xs = []
    try:
        for lat in (False, True):
            set_lattice(fem, lat)
            M._graph = None
            x, its, rel = M.solve(k, F, rtol=1e-10)
            assert rel <= 1e-10
            xs.append((x.clone(), its))
    finally:
        set_lattice(fem, True)
    assert xs[0][1] == xs[1][1] and torch.equal(xs[0][0], xs[1][0])
    # tsx: not on a uniform lattice
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "assembly_tsx_p1.npz"))
    el = torch.as_tensor(g["elements"].astype(np.int32)).cuda()
    co = torch.as_tensor(g["coordinates"]).cuda()
    Pt = fem["plan"].FemPlan(el, co, d1, d2, wf)
    with pytest.raises(mg.MultigridUnsupported):
        mg.MultigridPCG(Pt, Pt.mask_u8(torch.as_tensor(fo.tsx_q_mask(g["coordinates"])).cuda()))
