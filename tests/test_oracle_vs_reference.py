"""The oracle's mesh generator and assembly against stored outputs of the original project (tests/golden, written by
oracle/make_golden.py from the original's assemble_mesh and get_elastic_stiffness_matrix).  Everything is bit-exact."""
import numpy as np
import pytest

from oracle import fem_oracle as fo
from conftest import csr_from


def same(a, b):
    a, b = fo.canonical_csr(a), fo.canonical_csr(b)
    return (a.shape == b.shape and np.array_equal(a.indptr, b.indptr) and np.array_equal(a.indices, b.indices)
            and np.array_equal(a.data, b.data))


@pytest.mark.parametrize("name,level", [("P1", 0), ("Q1", 0), ("P2", 0), ("Q2", 0), ("P1", 1)])
def test_assembly_bit_exact(golden, name, level):
    """K and the weights on the original's footing mesh; for P1/Q1 the oracle's generator reproduces that mesh."""
    g, pre = (golden("assembly_footing_p1_l1.npz"), "") if level == 1 else (golden("assembly_all_types_l0.npz"), f"{name}_")
    et = fo.ElementType[name]
    xi, wf = fo.quadrature_volume(et)
    _, d1, d2 = fo.local_basis_volume(et, xi)
    elem, coord = g[pre + "elements"], g[pre + "coordinates"]
    n_int = elem.shape[1] * np.size(wf)
    G0, K0 = fo.footing_constants()[:2]
    K, _, w, _, _, _ = fo.elastic_stiffness(elem, coord, G0 * np.ones(n_int), K0 * np.ones(n_int), d1, d2, wf)
    assert same(K, csr_from(g, pre + "K")) and np.array_equal(w, g[pre + "weight"])
    if name in ("P1", "Q1"):
        m = fo.footing_mesh(level, et)
        keys = ("coordinates", "elements", "Q") + (("dirichlet_nodes",) if "dirichlet_nodes" in g.files else ())
        assert all(np.array_equal(m[k], g[pre + k]) for k in keys)


def test_material_constants():
    # the constants are literals inside elasticity_fem (:910-933); restated values must reproduce eta, c
    phi = np.pi / 9
    assert fo.footing_constants()[2] == 3 * np.tan(phi) / np.sqrt(9 + 12 * (np.tan(phi)) ** 2)
    assert fo.ElementType.P1.value == 1                       # the original's LagrangeElementType.P1
