"""Core-valence-separated X-TDA plans (plan.build_xtda_plan(p, core)) executed by the NumPy interpreter against the oracle's
P A P, the core set checks, the CVS so2st and the Davidson solver with nstates close to the dimension.  CPU only."""
import numpy as np
import pytest

from numpy_vectors import NumpyVectors
from oracle import amat
from oracle import sigma as osig
from plan_interp import PlanInterpreter
from xtddft_b200 import davidson as pdav
from xtddft_b200 import plan as planmod
from xtddft_b200 import utils
from xtddft_b200.synth import make_problem

FUNCTIONALS = {"LDA": dict(xctype="LDA", hyb=0.0), "GGA": dict(xctype="GGA", hyb=0.2), "MGGA": dict(xctype="MGGA", hyb=0.25),
               "HF": dict(xctype="HF", hyb=1.0), "RSH_GGA": dict(xctype="GGA", hyb=0.2, omega=0.33, alpha=0.65)}


def _problem(restricted, func, nc=4, no=2, nv=6, seed=700):
    return make_problem(nc + no + nv, nc, no, nv, 17, 40, restricted=restricted, seed=seed, **FUNCTIONALS[func])


def _dense_a(p):
    """Full-space A in PySCF order: the oracle's dense builder on ROKS, the oracle sigma of the unit vectors where the dense
    builder does not reach (UKS references, the tau part of meta-GGA kernels)."""
    if p.restricted and p.xctype != "MGGA":
        return amat.xtda_amat(p)
    vind, hd = osig.xtda_gen_vind(p)
    return vind(np.eye(hd.size)).T


def _core_sets(p, ncore):
    core = np.arange(p.nc - ncore, p.nc)            # the highest closed orbitals: not the trivial leading block
    if p.restricted:
        return core, (core, core)
    core_a = np.concatenate([core, [p.nc]])         # UKS: one open alpha orbital in the core set as well
    return (core_a, core), (core_a, core)


def test_default_plan_is_the_full_plan():
    for restricted in (True, False):
        p = _problem(restricted, "GGA")
        a, b = planmod.build_xtda_plan(p), planmod.build_xtda_plan(p, core=None)
        assert len(a.channels) == len(b.channels)
        for ca, cb in zip(a.channels, b.channels):
            assert np.array_equal(ca.occ_idx, cb.occ_idx) and np.array_equal(ca.vir_idx, cb.vir_idx)
            assert ca.o_blocks == cb.o_blocks and ca.v_blocks == cb.v_blocks
        assert [(k.tensor, k.ch) for k in a.k_terms] == [(k.tensor, k.ch) for k in b.k_terms]
        assert all(np.array_equal(x.weights, y.weights) for x, y in zip(a.k_terms, b.k_terms))
        assert [vars(j) for j in a.j_blocks] == [vars(j) for j in b.j_blocks]
        assert len(a.local_gemms) == len(b.local_gemms) and len(a.diags) == len(b.diags)
        for x, y in zip(a.local_gemms, b.local_gemms):
            assert (x.side, x.dst, x.src, x.alpha) == (y.side, y.dst, y.src, y.alpha) and np.array_equal(x.mat, y.mat)
        for x, y in zip(a.diags, b.diags):
            assert x.ch == y.ch and np.array_equal(x.d, y.d)
        assert np.array_equal(a.layout_entries, b.layout_entries) and np.array_equal(a.layout_coefs, b.layout_coefs)
        assert np.array_equal(a.hdiag, b.hdiag) and a.ext_dim == b.ext_dim and a.meta == b.meta
        assert a.ext_dim == p.nocc_a * p.nvir_a + p.nocc_b * p.nvir_b


@pytest.mark.parametrize("func", list(FUNCTIONALS))
@pytest.mark.parametrize("restricted", [True, False])
@pytest.mark.parametrize("ncore", [1, 2, "closed"])
def test_cvs_plan_is_projected_a(restricted, func, ncore):
    p = _problem(restricted, func)
    ncore = p.nc if ncore == "closed" else ncore
    core, (core_a, core_b) = _core_sets(p, ncore)
    pl = planmod.build_xtda_plan(p, core=core)
    rows = utils.cvs_rows(p.nc, p.no, p.nv, core_a, core_b)
    assert pl.ext_dim == rows.size == len(core_a) * p.nvir_a + len(core_b) * p.nvir_b
    a = _dense_a(p)
    pap = a[np.ix_(rows, rows)]
    z = np.random.default_rng(3).standard_normal((3, rows.size))
    got = PlanInterpreter(pl, p).sigma(z)
    ref = z @ pap.T
    assert np.abs(got - ref).max() <= 1e-12 * max(1.0, np.abs(ref).max())
    if restricted:
        hd_full = osig.xtda_gen_vind(p)[1]
        assert np.abs(pl.hdiag - hd_full[rows]).max() < 1e-14
    else:
        ea, eb = p.mo_energy
        hd_full = np.hstack([(ea[p.nocc_a:] - ea[:p.nocc_a, None]).ravel(), (eb[p.nocc_b:] - eb[:p.nocc_b, None]).ravel()])
        assert np.array_equal(pl.hdiag, hd_full[rows])
    if restricted and ncore == p.nc:
        # every closed orbital: A without the open-occupied (OV(aa)) rows
        full = np.arange(a.shape[0])
        ov = p.nc * p.nv + np.arange(p.no * p.nv)
        assert np.array_equal(rows, np.setdiff1d(full, ov))


@pytest.mark.parametrize("restricted,core", [
    (True, [2, 1]), (True, [1, 1]), (True, []), (True, [4]), (True, [-1, 0]), (True, [0.0, 1.0]), (True, [[0, 1]]),
    (False, [0, 1]), (False, ([0], [4])), (False, ([6], [0])), (False, ([1, 0], [0])), (False, ([0], [])), (False, ([0],)),
])
def test_bad_core_raises(restricted, core):
    p = _problem(restricted, "LDA")
    with pytest.raises(ValueError):
        planmod.build_xtda_plan(p, core=core)


@pytest.mark.parametrize("restricted", [True, False])
def test_cvs_so2st_is_full_so2st_on_core_rows(restricted):
    p = _problem(restricted, "GGA")
    nc, no, nv = p.nc, p.no, p.nv
    core, (core_a, core_b) = _core_sets(p, 2)
    rows = utils.cvs_rows(nc, no, nv, core_a, core_b)
    dim = p.nocc_a * p.nvir_a + p.nocc_b * p.nvir_b
    x = np.random.default_rng(5).standard_normal((rows.size, 4))             # CVS vectors, PySCF order (what the Davidson returns)
    order, my_rows = utils.cvs_order_pyscf2my(nc, no, nv, core_a, core_b)
    full_my = utils.so2st(utils.cvs_embed(x, rows, dim)[utils.order_pyscf2my(nc, no, nv)], nc, no, nv)
    got = utils.so2st(x[order], nc, no, nv, core=(core_a, core_b))
    assert np.array_equal(got, full_my[my_rows])
    outside = np.setdiff1d(np.arange(dim), my_rows)
    assert np.abs(full_my[outside]).max() == 0.0
    # identical to the full-space result when the core set is every occupied orbital
    if restricted:
        xf = np.random.default_rng(6).standard_normal((dim, 2))
        allc = (np.arange(p.nocc_a), np.arange(p.nocc_b))
        with pytest.raises(ValueError):                # a ROKS core set holds closed orbitals only
            planmod.cvs_core(p, np.arange(p.nocc_a))
        o2, _ = utils.cvs_order_pyscf2my(nc, no, nv, *allc)
        assert np.array_equal(utils.so2st(xf[o2], nc, no, nv, core=allc), utils.so2st(xf[utils.order_pyscf2my(nc, no, nv)], nc, no, nv))


def test_cvs_so2st_rejects_unpaired_core():
    p = _problem(False, "GGA")
    with pytest.raises(ValueError):
        utils.so2st(np.zeros((2 * p.nv + 1 * (p.no + p.nv), 1)), p.nc, p.no, p.nv, core=(np.array([0, 1]), np.array([1])))


@pytest.mark.parametrize("nroots_from_dim", [0, 2, 6])
def test_davidson_nstates_close_to_dim(nroots_from_dim):
    """The CVS operator of a small problem (dim 28) with nstates = dim - k: the solver ends converged with the dense roots."""
    p = _problem(True, "GGA")
    pl = planmod.build_xtda_plan(p, core=[2, 3])
    it = PlanInterpreter(pl, p)
    a = it.sigma(np.eye(pl.ext_dim)).T
    a = 0.5 * (a + a.T)
    dim, k = pl.ext_dim, pl.ext_dim - nroots_from_dim
    x0 = pdav.init_guess(pl.hdiag, k, 1e-3)
    conv, e, x, info = pdav.davidson1(lambda xs: xs @ a, x0, pl.hdiag.copy(), tol=1e-12, tol_residual=1e-6, lindep=1e-12, max_cycle=50,
                                      nroots=k, level_shift=0.0, backend=NumpyVectors(dim))
    assert conv.all()
    assert np.abs(e - np.linalg.eigvalsh(a)[:k]).max() < 1e-8
    assert info[0] < 50
