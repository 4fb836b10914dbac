"""GPU parity tests: the CUDA path (through the C ABI) against the oracle and the fixtures generated
from the reference.  Bars (BASELINE.json north_star): CSR row_ptr/col_idx and plastic flags bit-exact;
matrix values, stresses within rtol 1e-12 (assembly, strain and force are in fact bit-exact)."""
import numpy as np
import pytest
import scipy.sparse as sp

from conftest import csr_from
from oracle import fem_oracle as fo

pytestmark = pytest.mark.gpu

RTOL = 1e-12   # north_star tolerance for floating-point results


@pytest.fixture(scope="module")
def fem():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device")
    import fem_elastoplasticity_b200 as pkg
    from fem_elastoplasticity_b200 import plan, pythonFEM
    return {"torch": torch, "plan": plan, "api": pythonFEM, "pkg": pkg}


def tables(et):
    xi, wf = fo.quadrature_volume(et)
    _, d1, d2 = fo.local_basis_volume(et, xi)
    return d1, d2, wf


def canon(K):
    return fo.canonical_csr(K)


def assert_csr_bits(K_gpu_csr, ref, prune=True):
    K = sp.csr_matrix(K_gpu_csr).copy()
    if prune:
        K.eliminate_zeros()
    K.sort_indices()
    assert np.array_equal(K.indptr, ref.indptr), "row_ptr differs"
    assert np.array_equal(K.indices, ref.indices), "col_idx differs"
    bad = np.flatnonzero(K.data != ref.data)
    assert bad.size == 0, f"{bad.size} values differ; max rel {np.abs(K.data[bad] - ref.data[bad]).max() / np.abs(ref.data).max():.3e}"


@pytest.mark.parametrize("name", ["assembly_tsx_p1.npz", "assembly_footing_p1_l1.npz"])
def test_pattern_and_elastic_values_bit_exact(fem, golden, name):
    g = golden(name)
    d1, d2, wf = tables(fo.ElementType.P1)
    P = fem["plan"].FemPlan(g["elements"], g["coordinates"], d1, d2, wf)
    n_e = g["elements"].shape[1]
    rp, ci = P.pattern_host()
    assert np.array_equal(rp.astype(np.int64), g["S_indptr"]), "structural row_ptr"
    assert np.array_equal(ci, g["S_indices"]), "structural col_idx"
    assert np.array_equal(P.weight.cpu().numpy(), g["weight"].ravel())
    vals = P.assemble_elastic(float(g["shear"]) * np.ones(n_e), float(g["bulk"]) * np.ones(n_e))
    assert_csr_bits(P.to_scipy_csr(vals), csr_from(g, "K"))       # pruned pattern + values, bit-exact
    if "B_data" in g.files:                                        # stored values of the reference's B
        B = fem["api"]._host_B(P, g["elements"])
        assert np.array_equal(canon(B).data, g["B_data"])


@pytest.mark.parametrize("name", ["P1", "P2", "Q1", "Q2"])
def test_all_element_types(fem, golden, name):
    g = golden("assembly_all_types_l0.npz")
    et = fo.ElementType[name]
    d1, d2, wf = tables(et)
    elem, coord = g[f"{name}_elements"], g[f"{name}_coordinates"]
    P = fem["plan"].FemPlan(elem, coord, d1, d2, wf)
    rp, ci = P.pattern_host()
    assert np.array_equal(rp.astype(np.int64), g[f"{name}_S_indptr"]) and np.array_equal(ci, g[f"{name}_S_indices"])
    assert np.array_equal(P.weight.cpu().numpy(), g[f"{name}_weight"].ravel())
    G0, K0 = fo.footing_constants()[:2]
    vals = P.assemble_elastic(G0 * np.ones(P.n_int), K0 * np.ones(P.n_int))
    # the gather reproduces scipy's accumulation order for every element type, so even the reference's
    # value-dependent pruned pattern (exact cancellations, SURVEY H1) must come out identical
    assert_csr_bits(P.to_scipy_csr(vals), csr_from(g, f"{name}_K"))


def test_config1_elasticity2d_facade(fem, golden):
    """comparison_assembly_P1_2D_elasticity.py:74-80 protocol: 1-based float elements, (K, weight) result, in-place shift."""
    g = golden("assembly_elasticity2d_n16.npz")
    d1, d2, wf = tables(fo.ElementType.P1)
    el = g["elements_1based"].copy()
    n_e = el.shape[1]
    K, w = fem["api"].get_elastic_stiffness_matrix(el, g["coordinates"], float(g["shear"]) * np.ones(n_e),
                                                   float(g["bulk"]) * np.ones(n_e), d1, d2, wf, variant="elasticity2d")
    assert np.array_equal(el, g["elements_1based"] - 1)              # Elasticity2D/pythonFEM.py:389
    assert sp.isspmatrix_csc(K)
    assert_csr_bits(K.tocsr(), csr_from(g, "K"), prune=False)
    assert np.array_equal(w, g["weight"])


def test_facade_plasticity_signature(fem, golden):
    g = golden("assembly_footing_p1_l1.npz")
    d1, d2, wf = tables(fo.ElementType.P1)
    n_e = g["elements"].shape[1]
    G, Kb = float(g["shear"]) * np.ones(n_e), float(g["bulk"]) * np.ones(n_e)
    K, B, w, i_d, j_d, D = fem["api"].get_elastic_stiffness_matrix(g["elements"], g["coordinates"], G, Kb, d1, d2, wf)
    Ko, Bo, wo, io, jo, Do = fo.elastic_stiffness(g["elements"], g["coordinates"], G, Kb, d1, d2, wf)
    assert_csr_bits(K.tocsr(), canon(Ko), prune=False)
    assert np.array_equal(canon(B).data, canon(Bo).data) and np.array_equal(canon(B).indices, canon(Bo).indices)
    assert np.array_equal(canon(D).data, canon(Do).data) and np.array_equal(canon(D).indptr, canon(Do).indptr)
    assert np.array_equal(w, wo) and np.array_equal(i_d, io) and np.array_equal(j_d, jo)


def check_return_map(r, ref, keys=("s", "ds", "ep")):
    assert np.array_equal(r["ind_p"].astype(bool), ref["ind_p"]), "plastic flags must be bit-exact"
    for k in keys:
        scale = np.abs(ref[k]).max(axis=1, keepdims=True) + 1e-300
        err = np.abs(r[k] - ref[k]) / np.maximum(np.abs(ref[k]), 1e-3 * scale)
        assert err.max() <= RTOL, (k, err.max())


def test_return_map_golden(fem, golden):
    g = golden("return_map.npz")
    api = fem["api"]
    args = (g["shear"], g["bulk"], g["eta"], g["c"])
    for apply in (False, True):
        ep_prev = g["Ep"].copy()
        r = api.construct_constitutive_problem(g["E"].copy(), ep_prev, *args, apply_plastic_strain=apply)
        ref = {k: g[f"pl{int(apply)}_{k}"] for k in ("s", "ds", "ind_p", "ep")}
        check_return_map(r, ref)
        assert r["lambda_final"] is None and r["n_apex"] > 0 and r["n_smooth"] > 0
        if apply:
            assert r["ep"] is ep_prev                                # mutated in place and returned (:751)
        else:
            assert np.array_equal(ep_prev, g["Ep"]) and not r["ep"].any()
    for tag in ("tsx1", "tsx0"):                                     # tsx0: early-out quirk (tsx-tunnel/pythonFEM.py:1103)
        r = api.construct_constitutive_problem(g["E"].copy(), g[f"{tag}_e0"], g["Ep"].copy(), *args, apply_plastic_strain=True)
        check_return_map(r, {k: g[f"{tag}_{k}"] for k in ("s", "ds", "ind_p", "ep")})


def test_return_map_random_vs_oracle(fem):
    G0, K0, eta0, c0, _ = fo.footing_constants()
    rng = np.random.default_rng(7)
    for n in (1, 2, 3, 255, 100001):                                 # odd sizes exercise the scalar kernel
        E = np.array([[-3e-4], [-3e-4], [0]]) + 2e-4 * rng.standard_normal((3, n))
        E[:, : max(1, n // 20)] *= 6
        Ep = 1e-5 * rng.standard_normal((4, n))
        G, K = G0 * (1 + 0.1 * rng.random(n)), K0 * (1 + 0.1 * rng.random(n))
        eta, c = eta0 * np.ones(n), c0 * np.ones(n)
        ref = fo.constitutive_problem(E.copy(), Ep.copy(), G, K, eta, c, True)
        r = fem["api"].construct_constitutive_problem(E.copy(), Ep.copy(), G, K, eta, c, True)
        check_return_map(r, ref)
        assert r["n_smooth"] == ref["n_smooth"] and r["n_apex"] == ref["n_apex"]
        lam_ref = ref["lambda_final"][0]
        sm = ~np.isnan(lam_ref) & (lam_ref != 0)
        np.testing.assert_allclose(r["lambda_apex_intended"][0][sm], lam_ref[sm], rtol=RTOL)


def test_return_map_empty_and_elastic(fem):
    G0, K0, eta0, c0, _ = fo.footing_constants()
    n = 64
    z = np.zeros((3, n))
    r = fem["api"].construct_constitutive_problem(z, np.zeros((4, n)), G0 * np.ones(n), K0 * np.ones(n), eta0 * np.ones(n), c0 * np.ones(n))
    assert not r["ind_p"].any() and r["lambda_final"] is not None and not r["s"].any()
    ref = fo.constitutive_problem(z, np.zeros((4, n)), G0 * np.ones(n), K0 * np.ones(n), eta0 * np.ones(n), c0 * np.ones(n))
    assert np.array_equal(r["ds"], ref["ds"])                         # elastic tangent is bit-exact


def test_newton_glue_golden(fem, golden):
    g, m = golden("newton_glue_footing_l1.npz"), golden("assembly_footing_p1_l1.npz")
    d1, d2, wf = tables(fo.ElementType.P1)
    n_e = m["elements"].shape[1]
    G0, K0, eta0, c0, _ = fo.footing_constants()
    G, Kb = G0 * np.ones(n_e), K0 * np.ones(n_e)
    P = fem["plan"].FemPlan(m["elements"], m["coordinates"], d1, d2, wf)
    u = g["U"].reshape(-1, order="F")
    E = P.strain(u).cpu().numpy()
    assert np.array_equal(E, g["E"]), "strain must be bit-exact (csr_matvec order)"
    F = P.internal_force(g["s"]).cpu().numpy()
    assert np.array_equal(F, g["F"]), "internal force must be bit-exact (csc_matvec order)"
    kel = P.assemble_elastic(G, Kb)
    ref = csr_from(g, "Kt")
    kt_ref = P.assemble_tangent_ref(g["ds"], G, Kb, kel)
    assert_csr_bits(P.to_scipy_csr(kt_ref), ref)                      # reference operation order: bit-exact
    kt = P.assemble_tangent(g["ds"])
    Kd = P.to_scipy_csr(kt)
    diff = abs(Kd - ref).max()
    assert diff <= RTOL * abs(ref).max(), diff                        # direct one-pass form: within tolerance
    kt2, F2 = P.assemble_tangent_force(g["ds"], g["s"])
    assert np.array_equal(kt2.cpu().numpy(), kt.cpu().numpy()) and np.array_equal(F2.cpu().numpy(), g["F"])
    # tangent of an all-elastic state equals K_elast bit-for-bit
    cp = fo.constitutive_problem(np.zeros((3, n_e)), np.zeros((4, n_e)), G, Kb, eta0 * np.ones(n_e), c0 * np.ones(n_e))
    assert np.array_equal(P.assemble_tangent(cp["ds"]).cpu().numpy(), kel.cpu().numpy())


def test_spmv_and_pcg_vs_dense(fem, golden):
    torch = fem["torch"]
    for name in ("assembly_tsx_p1.npz", "assembly_footing_p1_l1.npz"):
        g = golden(name)
        d1, d2, wf = tables(fo.ElementType.P1)
        n_e = g["elements"].shape[1]
        P = fem["plan"].FemPlan(g["elements"], g["coordinates"], d1, d2, wf)
        vals = P.assemble_elastic(float(g["shear"]) * np.ones(n_e), float(g["bulk"]) * np.ones(n_e))
        K = csr_from(g, "K", shape=(P.n_dof, P.n_dof))
        rng = np.random.default_rng(11)
        x = rng.standard_normal(P.n_dof)
        y = P.spmv(vals, x).cpu().numpy()
        np.testing.assert_allclose(y, K @ x, rtol=1e-12, atol=1e-12 * np.abs(K @ x).max())
        q = g["Q"] if "Q" in g.files else fo.tsx_q_mask(g["coordinates"])
        mask = P.mask_u8(q)
        qf = q.flatten(order="F")
        ym = P.spmv(vals, x, mask=mask).cpu().numpy()
        assert not ym[~qf].any()
        rhs = rng.standard_normal(P.n_dof)
        sol, its, rel = P.pcg(vals, rhs, mask, rtol=1e-14, maxit=20000, check_every=20)
        ref = fo.masked_dense_solve(K, rhs, q)
        assert rel <= 1e-13 and its > 0
        np.testing.assert_allclose(sol.cpu().numpy(), ref, rtol=1e-9, atol=1e-11 * np.abs(ref).max())
        # energy products of the stopping criterion
        v = [torch.as_tensor(rng.standard_normal(P.n_dof)).cuda() for _ in range(3)]
        en = P.energy_norms(vals, *v).cpu().numpy()
        np.testing.assert_allclose(en, [vi.cpu().numpy() @ (K @ vi.cpu().numpy()) for vi in v], rtol=1e-12)


def test_error_paths(fem):
    from fem_elastoplasticity_b200 import FemError, NonFiniteJacobian
    d1, d2, wf = tables(fo.ElementType.P1)
    coord = np.array([[0.0, 1.0, 0.0], [0.0, 0.0, 1.0]])
    with pytest.raises(FemError):                                     # node id out of range
        fem["plan"].FemPlan(np.array([[0], [1], [5]]), coord, d1, d2, wf)
    flat = np.array([[0.0, 1.0, 2.0], [0.0, 0.0, 0.0]])               # collinear triangle: det = 0
    with pytest.raises(NonFiniteJacobian):
        fem["plan"].FemPlan(np.array([[0], [1], [2]]), flat, d1, d2, wf)
    with pytest.raises(FemError):                                     # unsupported (n_p, n_q)
        fem["plan"].FemPlan(np.array([[0], [1], [2]]), coord, np.ones((3, 2)), np.ones((3, 2)), np.ones((1, 2)))


def test_large_mesh_properties(fem):
    """Size-independent properties at a size the oracle cannot reach quickly (2M elements)."""
    torch = fem["torch"]
    from fem_elastoplasticity_b200 import meshgen
    n = 1000
    m = meshgen.square_mesh_p1(n, n)
    d1, d2, wf = tables(fo.ElementType.P1)
    P = fem["plan"].FemPlan(m["elements"], m["coordinates"], d1, d2, wf)
    assert P.nnz == 28 * n * n + 24 * n + 4                           # SURVEY section 8 closed form
    G, Kb, eta, c = meshgen.footing_materials(P.n_int)
    kel = P.assemble_elastic(G, Kb)
    # rigid-body translations are in the null space; K symmetric
    tx = torch.zeros(P.n_dof, dtype=torch.float64, device="cuda")
    tx[0::2] = 1.0
    scale = kel.abs().max().item()
    assert P.spmv(kel, tx).abs().max().item() <= 1e-9 * scale
    g = torch.Generator(device="cuda").manual_seed(1)
    a = torch.randn(P.n_dof, generator=g, dtype=torch.float64, device="cuda")
    b = torch.randn(P.n_dof, generator=g, dtype=torch.float64, device="cuda")
    ab, ba = torch.dot(b, P.spmv(kel, a)).item(), torch.dot(a, P.spmv(kel, b)).item()
    assert abs(ab - ba) <= 1e-10 * abs(ab)
    # patch test: a linear displacement field has a constant strain
    u = torch.empty(P.n_dof, dtype=torch.float64, device="cuda")
    u[0::2] = 1e-3 * m["coordinates"][0] + 2e-3 * m["coordinates"][1]
    u[1::2] = -3e-3 * m["coordinates"][0] + 5e-4 * m["coordinates"][1]
    E = P.strain(u)
    for row, val in zip(E, (1e-3, 5e-4, 2e-3 - 3e-3)):
        assert (row - val).abs().max().item() <= 1e-12
    # elastic state: tangent == elastic stiffness bit-for-bit; plastic state flags match the oracle on a sample
    from fem_elastoplasticity_b200.plan import dp_return_map
    r = dp_return_map(torch.zeros((3, P.n_int), dtype=torch.float64, device="cuda"), None, G, Kb, eta, c)
    assert torch.equal(P.assemble_tangent(r["ds"]), kel)
    Es = meshgen.synthetic_strain(P.n_int)
    r = dp_return_map(Es, None, G, Kb, eta, c)
    idx = slice(0, 200000)
    ref = fo.constitutive_problem(Es[:, idx].cpu().numpy(), np.zeros((4, 200000)), G[idx].cpu().numpy(), Kb[idx].cpu().numpy(),
                                  eta[idx].cpu().numpy(), c[idx].cpu().numpy())
    assert np.array_equal(r["ind_p"][idx].cpu().numpy().astype(bool), ref["ind_p"])
    assert int(r["counts"].sum().item()) == int(r["ind_p"].sum().item())
    frac = r["ind_p"].double().mean().item()
    assert 0.005 < frac < 0.08
    # the TMA-staged kernel is the one that ran (structured mesh -> staging plan valid) and equals the other variants bit-for-bit
    from fem_elastoplasticity_b200 import _lib
    assert P.stage_info()[0] == 1 and 32 <= P.stage_info()[1] <= 96      # (stage_ok, TMA box width in elements)
    S4 = torch.randn((4, P.n_int), dtype=torch.float64, device="cuda", generator=g)
    ref = None
    try:
        for v in (6, 2, 1):
            _lib.call("fem_set_tuning", b"assemble_variant", v)
            got = (P.assemble_elastic(G, Kb), *P.assemble_tangent_force(r["ds"], S4), P.assemble_tangent_ref(r["ds"], G, Kb, kel))
            if ref is None:
                ref = got
            else:
                assert all(torch.equal(x, y) for x, y in zip(ref, got)), v
    finally:
        _lib.call("fem_set_tuning", b"assemble_variant", 0)
    assert torch.equal(ref[0], kel)
    # internal force of a constant stress field vanishes at interior nodes (divergence-free)
    S = torch.ones((4, P.n_int), dtype=torch.float64, device="cuda")
    F = P.internal_force(S).reshape(-1, 2)
    interior = (m["coordinates"][0] > 0) & (m["coordinates"][0] < 10) & (m["coordinates"][1] > 0) & (m["coordinates"][1] < 10)
    assert F[interior].abs().max().item() <= 1e-12


def test_assembly_variants_agree_bitwise(fem, golden):
    """Shared-memory and register accumulators run the same arithmetic in the same order."""
    from fem_elastoplasticity_b200 import _lib
    g, m = golden("newton_glue_footing_l1.npz"), golden("assembly_footing_p1_l1.npz")
    d1, d2, wf = tables(fo.ElementType.P1)
    n_e = m["elements"].shape[1]
    G0, K0 = fo.footing_constants()[:2]
    G, Kb = G0 * np.ones(n_e), K0 * np.ones(n_e)
    P = fem["plan"].FemPlan(m["elements"], m["coordinates"], d1, d2, wf)
    res = {}
    try:
        for v in (6, 2, 1):
            _lib.call("fem_set_tuning", b"assemble_variant", v)
            kel = P.assemble_elastic(G, Kb)
            kt, F = P.assemble_tangent_force(g["ds"], g["s"])
            ktr = P.assemble_tangent_ref(g["ds"], G, Kb, kel)
            res[v] = [t.cpu().numpy() for t in (kel, kt, F, ktr)]
    finally:
        _lib.call("fem_set_tuning", b"assemble_variant", 0)
    for v in (2, 6):
        for a, b in zip(res[1], res[v]):
            assert np.array_equal(a, b), v
    assert_csr_bits(P.to_scipy_csr(fem["torch"].as_tensor(res[2][3]).cuda()), csr_from(g, "Kt"))


def test_canonical_row_stores_any_alignment(fem):
    """The straight-line path of the regular triangulation writes a node's two rows as seven 256-bit stores when K is
    32-byte aligned and as 16-byte stores otherwise; with the path off (assemble_canon = 2) the generic kernel runs.  All
    three must give the same bits, and the oracle's."""
    torch = fem["torch"]
    from fem_elastoplasticity_b200 import _lib
    m = fo.square_mesh_p1(200, 150, 10.0, 7.5)
    d1, d2, wf = tables(fo.ElementType.P1)
    n_e = m["elements"].shape[1]
    G0, K0 = fo.footing_constants()[:2]
    G, Kb = G0 * np.ones(n_e), K0 * np.ones(n_e)
    P = fem["plan"].FemPlan(m["elements"], m["coordinates"], d1, d2, wf)
    assert P.stage_info()[0] == 1
    rng = np.random.default_rng(5)
    ds = rng.standard_normal((9, P.n_int))
    s = rng.standard_normal((4, P.n_int))
    big = torch.zeros(P.nnz + 8, dtype=torch.float64, device="cuda")
    assert big.data_ptr() % 32 == 0
    res = {}
    try:
        for name, canon, off in (("wide", 0, 0), ("wide_misaligned", 0, 2), ("generic", 2, 0)):
            _lib.call("fem_set_tuning", b"assemble_canon", canon)
            k = big[off:off + P.nnz]
            assert k.data_ptr() % 32 == (16 if off else 0)
            P.assemble_elastic(G, Kb, out=k)
            kel = k.clone()
            k.zero_()
            kt, F = P.assemble_tangent_force(ds, s, out_k=k)
            res[name] = [t.cpu().numpy() for t in (kel, kt.clone(), F)]
            k.zero_()
    finally:
        _lib.call("fem_set_tuning", b"assemble_canon", 0)
    for name in ("wide_misaligned", "generic"):
        for a, b in zip(res["wide"], res[name]):
            assert np.array_equal(a, b), name
    Ko = fo.elastic_stiffness(m["elements"], m["coordinates"], G, Kb, d1, d2, wf)[0]
    Kg = P.to_scipy_csr(torch.as_tensor(res["wide"][0]).cuda())
    Kg.eliminate_zeros()
    assert_csr_bits(Kg, fo.canonical_csr(Ko))


def test_full_size_config4_properties(fem):
    """BASELINE.json config 4 (N=2828, 15 995 168 elements): size-independent properties at the benchmarked size."""
    torch = fem["torch"]
    from fem_elastoplasticity_b200 import _lib, meshgen
    from fem_elastoplasticity_b200.plan import dp_return_map
    n = 2828
    m = meshgen.square_mesh_p1(n, n)
    d1, d2, wf = tables(fo.ElementType.P1)
    P = fem["plan"].FemPlan(m["elements"], m["coordinates"], d1, d2, wf)
    assert (P.n_e, P.n_n, P.n_dof, P.nnz) == (15995168, 8003241, 16006482, 224000228)      # SURVEY section 8
    assert P.stage_info()[0] == 1
    # row_ptr of a uniform mesh: every interior node has 7 neighbours
    deg = (P.nbr_ptr[1:] - P.nbr_ptr[:-1])
    assert int(deg.max()) == 7 and int(deg.min()) == 3
    assert torch.equal(P.row_ptr[0::2][:-1].long(), 4 * P.nbr_ptr[:-1].long())
    G, Kb, eta, c = meshgen.footing_materials(P.n_int)
    kel = P.assemble_elastic(G, Kb)
    # the oracle on the first rows of the mesh: bit-exact values on a 2828 x 2 strip (same numbering, same coordinates)
    strip = fo.square_mesh_p1(n, 2, 10.0, 10.0 * 2 / n)
    coord = m["coordinates"][:, : 3 * (n + 1)].cpu().numpy()
    Ks = fo.canonical_csr(fo.elastic_stiffness(strip["elements"], coord, G[: 4 * n].cpu().numpy(), Kb[: 4 * n].cpu().numpy(), d1, d2, wf)[0])
    rows = 2 * 2 * (n + 1)                                  # node rows 0 and 1 are complete in the strip
    rp = P.row_ptr[: rows + 1].cpu().numpy()
    sub = sp.csr_matrix((kel[: rp[-1]].cpu().numpy(), P.col_idx[: rp[-1]].cpu().numpy(), rp), shape=(rows, P.n_dof))
    sub.eliminate_zeros()
    ref = Ks[:rows]
    assert np.array_equal(sub.indptr, ref.indptr) and np.array_equal(sub.indices, ref.indices) and np.array_equal(sub.data, ref.data)
    # null space, symmetry, elastic-tangent identity, variant equality at full size
    tx = torch.zeros(P.n_dof, dtype=torch.float64, device="cuda")
    tx[1::2] = 1.0
    assert P.spmv(kel, tx).abs().max().item() <= 1e-9 * kel.abs().max().item()
    g = torch.Generator(device="cuda").manual_seed(3)
    a = torch.randn(P.n_dof, generator=g, dtype=torch.float64, device="cuda")
    b = torch.randn(P.n_dof, generator=g, dtype=torch.float64, device="cuda")
    ab, ba = torch.dot(b, P.spmv(kel, a)).item(), torch.dot(a, P.spmv(kel, b)).item()
    assert abs(ab - ba) <= 1e-10 * abs(ab)
    Es = meshgen.synthetic_strain(P.n_int)
    r = dp_return_map(Es, None, G, Kb, eta, c)
    counts = r["counts"].cpu().numpy()
    assert counts.sum() == int(r["ind_p"].sum().item()) and counts[0] > 0 and counts[1] > 0
    idx = slice(8000000, 8100000)
    ref = fo.constitutive_problem(Es[:, idx].cpu().numpy(), np.zeros((4, 100000)), G[idx].cpu().numpy(), Kb[idx].cpu().numpy(),
                                  eta[idx].cpu().numpy(), c[idx].cpu().numpy())
    assert np.array_equal(r["ind_p"][idx].cpu().numpy().astype(bool), ref["ind_p"])
    err = np.abs(r["s"][:, idx].cpu().numpy() - ref["s"]) / np.maximum(np.abs(ref["s"]), 1e-3 * np.abs(ref["s"]).max(axis=1, keepdims=True))
    assert err.max() <= RTOL
    kt = P.assemble_tangent(r["ds"])
    try:
        _lib.call("fem_set_tuning", b"assemble_variant", 2)
        assert torch.equal(P.assemble_tangent(r["ds"]), kt)
    finally:
        _lib.call("fem_set_tuning", b"assemble_variant", 0)
    r0 = dp_return_map(torch.zeros_like(Es), None, G, Kb, eta, c)
    assert torch.equal(P.assemble_tangent(r0["ds"]), kel)


def test_empty_and_ragged_inputs(fem):
    """Edge cases: zero Gauss points, a single element, an isolated node, a node of valence > 8 (shared-memory kernel)."""
    torch = fem["torch"]
    api = fem["api"]
    r = api.construct_constitutive_problem(np.zeros((3, 0)), np.zeros((4, 0)), np.zeros(0), np.zeros(0), np.zeros(0), np.zeros(0))
    assert r["s"].shape == (4, 0) and r["ds"].shape == (9, 0) and r["ind_p"].shape == (0,)
    d1, d2, wf = tables(fo.ElementType.P1)
    # one triangle + one node that belongs to no element (empty rows, as in the reference's B^T D B)
    coord = np.array([[0.0, 1.0, 0.0, 5.0], [0.0, 0.0, 1.0, 5.0]])
    elem = np.array([[0], [1], [2]])
    P = fem["plan"].FemPlan(elem, coord, d1, d2, wf)
    Ko = fo.canonical_csr(fo.elastic_stiffness(elem, coord, np.ones(1), 2 * np.ones(1), d1, d2, wf)[0])
    K = P.to_scipy_csr(P.assemble_elastic(np.ones(1), 2 * np.ones(1)))
    K.eliminate_zeros()
    assert np.array_equal(K.indptr, Ko.indptr) and np.array_equal(K.indices, Ko.indices) and np.array_equal(K.data, Ko.data)
    assert K.indptr[-1] == K.indptr[6]                      # rows of the isolated node are empty
    # a fan of 12 triangles around one node: valence 13 > 12 -> shared-memory accumulators
    k = 12
    ang = 2 * np.pi * np.arange(k) / k
    coord = np.concatenate([[[0.0], [0.0]], np.array([np.cos(ang), np.sin(ang)]) * (1 + 0.1 * np.arange(k))], axis=1)
    elem = np.array([[0] * k, list(range(1, k + 1)), [i % k + 1 for i in range(1, k + 1)]])
    P = fem["plan"].FemPlan(elem, coord, d1, d2, wf)
    assert P.max_degree == 13 and P.stage_info()[0] == 0
    rng = np.random.default_rng(0)
    G, Kb = 1 + rng.random(k), 2 + rng.random(k)
    Ko = fo.canonical_csr(fo.elastic_stiffness(elem, coord, G, Kb, d1, d2, wf)[0])
    K = P.to_scipy_csr(P.assemble_elastic(G, Kb))
    K.eliminate_zeros()
    assert np.array_equal(K.indptr, Ko.indptr) and np.array_equal(K.indices, Ko.indices) and np.array_equal(K.data, Ko.data)


def test_transform_and_csv_fixture_io(fem, golden, tmp_path):
    """SURVEY 8(f)-3/4: transform() on the device; CSV mesh reader and the golden *_qq.csv / fq.csv layout."""
    from fem_elastoplasticity_b200 import fixture_io
    m, g = golden("assembly_tsx_p1.npz"), golden("tsx_csv_golden.npz")
    np.savetxt(tmp_path / "coord.csv", m["coordinates"], delimiter=",", fmt="%.17g")
    np.savetxt(tmp_path / "elem.csv", m["elements"] + 1, delimiter=",", fmt="%d")
    coords, elem = fixture_io.read_mesh_csv(tmp_path / "coord.csv", tmp_path / "elem.csv")
    assert np.array_equal(coords, m["coordinates"]) and np.array_equal(elem, m["elements"])
    d1, d2, wf = tables(fo.ElementType.P1)
    n_e = elem.shape[1]
    G, Kb = float(m["shear"]) * np.ones(n_e), float(m["bulk"]) * np.ones(n_e)
    K, B, w, i_d, j_d, D = fem["api"].get_elastic_stiffness_matrix(elem, coords, G, Kb, d1, d2, wf)
    q = fixture_io.tsx_dirichlet_mask(coords)
    assert np.array_equal(q, fo.tsx_q_mask(coords))
    # regenerate the missing kelast_qq.csv and read it back; for P1 it must carry k_tangent_qq.csv's pattern
    fixture_io.write_qq_csv(tmp_path / "kelast_qq.csv", K, q)
    kqq = fixture_io.read_qq_csv(tmp_path / "kelast_qq.csv")
    assert kqq.shape == tuple(g["kqq_shape"]) == (908, 908)
    assert np.array_equal(kqq, fixture_io.free_block(K, q))           # %.17g round-trips doubles
    ref = csr_from(g, "kqq", shape=(908, 908))
    got = sp.csr_matrix(kqq)
    got.sort_indices()
    assert np.array_equal(got.indptr, ref.indptr) and np.array_equal(got.indices, ref.indices)
    assert np.abs(got.data - ref.data).max() <= 2e-4 * np.abs(ref.data).max()
    # F[Q] export layout
    _, _, _, _, s0, _ = fo.tsx_constants()
    F0 = fem["api"].internal_force(B, np.tile(s0, (1, n_e)))
    fixture_io.write_fq_csv(tmp_path / "f0q.csv", F0, q)
    back = np.genfromtxt(tmp_path / "f0q.csv", delimiter=",")
    assert back.shape == (908,) and np.array_equal(back, F0.ravel()[q.flatten(order="F")])
    # transform(): integration-point -> nodal weighted average (Plasticity2D_DP/pythonFEM.py:760-816)
    P = K._fem_plan
    rng = np.random.default_rng(2)
    qi = rng.standard_normal(n_e)
    got = P.transform(qi).cpu().numpy()
    np.testing.assert_allclose(got, fo.transform(qi, elem, w), rtol=1e-13)


def test_tsx_p2_unstructured(fem, golden):
    """P2 kernels (6 nodes, 7 points, shared-memory accumulators) on the unstructured tsx mesh: K bit-exact vs the reference,
    F0 = B^T (w sigma0) bit-exact, and F0[Q] against the reference's own f0q.csv."""
    g, c = golden("assembly_tsx_p2.npz"), golden("tsx_csv_golden.npz")
    et = fo.ElementType.P2
    d1, d2, wf = tables(et)
    P = fem["plan"].FemPlan(g["elements"], g["coordinates"], d1, d2, wf)
    assert (P.n_p, P.n_q, P.n_n) == (6, 7, 1839) and P.max_degree > 12
    assert np.array_equal(P.weight.cpu().numpy(), g["weight"].flatten(order="F"))
    vals = P.assemble_elastic(float(g["shear"]) * np.ones(P.n_int), float(g["bulk"]) * np.ones(P.n_int))
    assert_csr_bits(P.to_scipy_csr(vals), csr_from(g, "K"))
    s0 = fo.tsx_constants()[4]
    F0 = P.internal_force(np.tile(s0, (1, P.n_int))).cpu().numpy()
    assert np.array_equal(F0, g["F0"])
    qf = fo.tsx_q_mask(g["coordinates"]).flatten(order="F")
    assert np.abs(F0[qf] - c["f0q"]).max() < 2e-3
    # strain of a linear field is constant on quadratic elements too
    u = np.empty(P.n_dof)
    u[0::2] = 1e-3 * g["coordinates"][0] - 2e-3 * g["coordinates"][1]
    u[1::2] = 4e-3 * g["coordinates"][0] + 5e-4 * g["coordinates"][1]
    E = P.strain(u).cpu().numpy()
    for row, val in zip(E, (1e-3, 5e-4, -2e-3 + 4e-3)):
        assert np.abs(row - val).max() <= 1e-11


def test_two_level_pcg(fem, golden):
    """Two-level preconditioned CG (Jacobi + coarse-grid correction): same solution as the dense solve, far fewer iterations."""
    from fem_elastoplasticity_b200 import meshgen
    from fem_elastoplasticity_b200.twolevel import TwoLevelPCG
    torch = fem["torch"]
    d1, d2, wf = tables(fo.ElementType.P1)
    # (a) unstructured tsx mesh (domain with a hole: some coarse nodes have no support) against the dense solve
    g = golden("assembly_tsx_p1.npz")
    n_e = g["elements"].shape[1]
    P = fem["plan"].FemPlan(g["elements"], g["coordinates"], d1, d2, wf)
    vals = P.assemble_elastic(float(g["shear"]) * np.ones(n_e), float(g["bulk"]) * np.ones(n_e))
    q = fo.tsx_q_mask(g["coordinates"])
    mask = P.mask_u8(q)
    rhs = np.random.default_rng(5).standard_normal(P.n_dof)
    tl = TwoLevelPCG(P, mask, nc=6)
    x, its, rel = tl.solve(vals, P._f64(rhs), rtol=1e-13, maxit=5000, check_every=5)
    ref = fo.masked_dense_solve(csr_from(g, "K", shape=(P.n_dof, P.n_dof)), rhs, q)
    assert rel <= 1e-13
    np.testing.assert_allclose(x.cpu().numpy(), ref, rtol=1e-8, atol=1e-10 * np.abs(ref).max())
    _, its_j, _ = P.pcg(vals, rhs, mask, rtol=1e-13, maxit=20000, check_every=5)
    assert its < its_j
    # (b) footing problem, 160 x 160 cells: the CPU prototype needs 3551 Jacobi / 430 two-level iterations (H/h = 10)
    m = meshgen.square_mesh_p1(160, 160)
    P = fem["plan"].FemPlan(m["elements"], m["coordinates"], d1, d2, wf)
    G, Kb, _, _ = meshgen.footing_materials(P.n_int)
    k = P.assemble_elastic(G, Kb)
    mask = P.mask_u8(m["Q"])
    ud = (-1e-3 * m["dirichlet_nodes"]).t().reshape(-1).contiguous()
    f = -P.spmv(k, ud)
    xj, its_j, _ = P.pcg(k, f, mask, rtol=1e-10, maxit=20000, check_every=25)
    tl = TwoLevelPCG(P, mask, nc=16)
    xt, its_t, rel = tl.solve(k, f, rtol=1e-10, maxit=20000, check_every=5)
    print("jacobi", its_j, "two-level", its_t)
    assert 3000 < its_j < 4200 and 300 < its_t < 600
    assert float((xt - xj).abs().max() / xj.abs().max()) < 1e-6
