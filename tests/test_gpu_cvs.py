"""Core-valence-separated X-TDA on the B200 engine: sigma of P A P against the oracle on the FP64 and the emulated exchange path
(small shapes and the config-4 orbital shape with 1 and 2 core orbitals, forced aux / grid chunks), aux / grid shards, Davidson
roots against a dense eigh of P A P (5 roots and nstates close to dim), oscillator strengths, and the driver classes with
`core_idx` on synthetic and stand-in mean-field objects.  Needs a B200."""
import ctypes as C

import numpy as np
import pytest

from adapter_fakes import fake_scf, packed_df
from oracle import amat
from oracle import properties as oprop
from oracle import sigma as osig
from xtddft_b200 import plan as planmod
from xtddft_b200 import utils
from xtddft_b200.adapters import SynthMF
from xtddft_b200.synth import make_problem

from golden.make_golden_properties import one_electron

pytestmark = pytest.mark.gpu
RTOL = 1e-9
FUNCTIONALS = {"LDA": dict(xctype="LDA", hyb=0.0), "GGA": dict(xctype="GGA", hyb=0.2), "MGGA": dict(xctype="MGGA", hyb=0.25),
               "HF": dict(xctype="HF", hyb=1.0), "RSH_GGA": dict(xctype="GGA", hyb=0.2, omega=0.33, alpha=0.65)}


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


def _rel(got, ref):
    return float(np.abs(got - ref).max() / max(1.0, np.abs(ref).max()))


def _core(p, ncore):
    """(core argument, (core_a, core_b)): the highest ncore closed orbitals; on UKS the alpha set also holds the first open orbital."""
    core = np.arange(p.nc - ncore, p.nc)
    if p.restricted:
        return core, (core, core)
    core_a = np.concatenate([core, [p.nc]])
    return (core_a, core), (core_a, core)


def _cvs_ref(p, core_ab, z):
    """P A P z from the oracle's full-space sigma of the zero-padded vectors."""
    rows = utils.cvs_rows(p.nc, p.no, p.nv, *core_ab)
    vind, hd = osig.xtda_gen_vind(p)
    return vind(utils.cvs_embed(z.T, rows, hd.size).T)[:, rows], hd[rows]


def _engine(p, pl, slices, **kw):
    from xtddft_b200.engine import SigmaEngine
    kw.setdefault("workspace_bytes", 256 << 20)
    kw.setdefault("max_nvec", 4)
    return SigmaEngine.from_problem(pl, p, exchange_slices=slices, **kw)


@pytest.mark.parametrize("slices", [0, 6])
@pytest.mark.parametrize("func", list(FUNCTIONALS))
@pytest.mark.parametrize("restricted", [True, False])
@pytest.mark.parametrize("ncore", [1, 2, 4])
def test_cvs_sigma_vs_oracle(torch_cuda, restricted, func, ncore, slices):
    p = make_problem(5 + 2 + 40, 5, 2, 40, 23, 300, restricted=restricted, seed=600 + ncore, **FUNCTIONALS[func])
    core, core_ab = _core(p, ncore)
    z = np.random.default_rng(ncore).standard_normal((3, utils.cvs_rows(p.nc, p.no, p.nv, *core_ab).size))
    ref, hd = _cvs_ref(p, core_ab, z)
    eng = _engine(p, planmod.build_xtda_plan(p, core=core), slices)
    try:
        assert eng.exchange_slices == slices
        assert _rel(eng.sigma_host(z), ref) < RTOL
        assert np.abs(eng.hdiag() - hd).max() < 1e-12
    finally:
        eng.close()


_CFG4 = {}


def _config4_case(nv, ncore):
    """(problem, z, oracle P A P z, hdiag), computed once per shape for both exchange paths."""
    if (nv, ncore) not in _CFG4:
        p = make_problem(136 + 1 + nv, 136, 1, nv, 6, 2048, xctype="GGA", hyb=0.2, seed=320)
        _, core_ab = _core(p, ncore)
        z = np.random.default_rng(5).standard_normal((2, utils.cvs_rows(p.nc, p.no, p.nv, *core_ab).size))
        _CFG4[(nv, ncore)] = (p, z) + _cvs_ref(p, core_ab, z)
    return _CFG4[(nv, ncore)]


@pytest.mark.parametrize("slices", [0, 6])
@pytest.mark.parametrize("ncore", [1, 2])
@pytest.mark.parametrize("nv", [821, 822])
def test_cvs_config4_orbital_shape(torch_cuda, monkeypatch, nv, ncore, slices):
    """Config-4 orbital counts (nc 136, no 1, nv 821 / 822) with few aux functions and grid points; several aux and grid chunks
    forced, the loop counts read back from the engine."""
    monkeypatch.setenv("XTD_CHUNK_AUX", "2")
    monkeypatch.setenv("XTD_CHUNK_GRID", "640")
    p, z, ref, hd = _config4_case(nv, ncore)
    core, _ = _core(p, ncore)
    eng = _engine(p, planmod.build_xtda_plan(p, core=core), slices, workspace_bytes=4 << 30, df_chunk=2)
    try:
        got = eng.sigma(torch_cuda.from_numpy(z).cuda()).cpu().numpy()
        ca, cg = eng.last_chunks()
        # FP64 path: 6 aux functions in chunks of 2, 2048 points in chunks of 640; the emulated path regroups the aux functions into
        # whole scale groups and runs its one-component grid GEMMs on its own point chunks
        assert (ca, cg) == (3, 4) if slices == 0 else ca >= 2, (ca, cg)
        assert _rel(got, ref) < RTOL
        assert np.abs(eng.hdiag() - hd).max() < 1e-10
    finally:
        eng.close()


@pytest.mark.parametrize("slices", [0, 6])
def test_cvs_shards_sum_to_whole(torch_cuda, slices):
    """world = 2 shards of the aux functions and grid points, one after the other on this GPU: the partial sigma buffers add up to
    the unsharded one, and the sharded result finished from the sum equals the unsharded sigma."""
    from xtddft_b200 import _lib
    from xtddft_b200.engine import _as_tensor
    torch = torch_cuda
    p = make_problem(3 + 2 + 60, 3, 2, 60, 37, 500, xctype="GGA", hyb=0.3, seed=610)
    pl = planmod.build_xtda_plan(p, core=[1])
    zt = torch.from_numpy(np.random.default_rng(9).standard_normal((3, pl.ext_dim))).cuda()

    def partial(eng):
        _lib.check(eng.lib.xtd_sigma_partial(eng._h, zt.shape[0], C.c_void_p(zt.data_ptr())), "partial")
        ptr, n = C.c_void_p(), C.c_long()
        _lib.check(eng.lib.xtd_partial_buffer(eng._h, zt.shape[0], C.byref(ptr), C.byref(n)), "buffer")
        return _as_tensor(torch, ptr.value, n.value, eng.device).clone()

    eng = _engine(p, pl, slices)
    whole = partial(eng)
    full = eng.sigma(zt).cpu().numpy()
    eng.close()
    acc = torch.zeros_like(whole)
    for r in range(2):
        e = _engine(p, planmod.build_xtda_plan(p, core=[1]), slices, rank=r, world=2)
        acc += partial(e)
        e.close()
    assert (acc - whole).abs().max().item() <= 1e-11 * max(1.0, whole.abs().max().item())
    vind_ref, _ = _cvs_ref(p, ([1], [1]), zt.cpu().numpy())
    assert _rel(full, vind_ref) < RTOL


def _pap(p, core_ab):
    rows = utils.cvs_rows(p.nc, p.no, p.nv, *core_ab)
    if p.restricted and p.xctype != "MGGA":                     # the dense builder has no tau part
        a = amat.xtda_amat(p)
    else:
        a = osig.xtda_gen_vind(p)[0](np.eye(p.nocc_a * p.nvir_a + p.nocc_b * p.nvir_b)).T
    return a[np.ix_(rows, rows)]


@pytest.mark.parametrize("restricted", [True, False])
@pytest.mark.parametrize("python_solver", [False, True])
def test_cvs_davidson_roots_vs_dense(torch_cuda, restricted, python_solver):
    """Five roots from the native and the Python solver loop against a dense eigh of P A P."""
    from xtddft_b200.drivers_common import make_engine, solve
    p = make_problem(4 + 2 + 30, 4, 2, 30, 27, 400, xctype="GGA", hyb=0.25, restricted=restricted, seed=620)
    core, core_ab = _core(p, 2)
    w = np.linalg.eigvalsh(_pap(p, core_ab))
    eng = make_engine(planmod.build_xtda_plan(p, core=core), p, distributed=False)
    try:
        conv, e, x, cyc, hd = solve(eng, 5, "xtda", python_solver=python_solver)
        assert conv.all()
        assert np.abs(e - w[w > 1e-3][:5]).max() < 1e-8
        assert x.shape == (hd.size, 5)
    finally:
        eng.close()


@pytest.mark.parametrize("gap", [0, 1, 3])
@pytest.mark.parametrize("python_solver", [False, True])
def test_cvs_davidson_nstates_close_to_dim(torch_cuda, gap, python_solver):
    """nstates = dim - gap on a CVS space of 21 unknowns: the solver ends converged with every dense root."""
    from xtddft_b200.drivers_common import make_engine, solve
    p = make_problem(3 + 1 + 10, 3, 1, 10, 15, 200, xctype="LDA", hyb=0.3, seed=630)
    pap = _pap(p, ([2], [2]))
    dim = pap.shape[0]
    assert dim == 21
    w = np.linalg.eigvalsh(pap)
    eng = make_engine(planmod.build_xtda_plan(p, core=[2]), p, distributed=False)
    try:
        conv, e, x, cyc, _ = solve(eng, dim - gap, "xtda", python_solver=python_solver)
        assert conv.all() and len(e) == dim - gap
        assert np.abs(e - w[:dim - gap]).max() < 1e-8
    finally:
        eng.close()


@pytest.mark.parametrize("restricted", [True, False])
def test_cvs_driver_and_oscillator_strengths(torch_cuda, restricted):
    """XTDA(core_idx=...) on a synthetic mean-field object: roots, the CVS layout of v, cvs_embed, so2st and the oscillator strengths
    against the oracle's moments of the zero-padded vectors."""
    from xtddft_b200.XTDA import XTDA
    p = make_problem(4 + 2 + 30, 4, 2, 30, 27, 400, xctype="GGA", hyb=0.25, restricted=restricted, seed=640)
    dip = one_electron(p.nao, 641)[0]
    p.meta = dict(p.meta or {}, one_electron={"int1e_r": dip})
    core, core_ab = _core(p, 2)
    mf = SynthMF(p)
    td = XTDA(mf.mol, mf, nstates=5, core_idx=core)
    e, v = td.kernel()
    assert td.converged.all()
    w = np.linalg.eigvalsh(_pap(p, core_ab))
    assert np.abs(e - w[w > 1e-3][:5]).max() < 1e-8
    rows = utils.cvs_rows(p.nc, p.no, p.nv, *core_ab)
    assert v.shape == (rows.size, 5)
    x_full = td.cvs_embed(td._x_rows.T)
    assert x_full.shape == (p.nocc_a * p.nvir_a + p.nocc_b * p.nvir_b, 5)
    ref_os = oprop.xtda_osc_str(p, e, x_full.T, dip)
    assert np.abs(td.os - ref_os).max() <= RTOL * max(1.0, np.abs(ref_os).max())
    v_full_my = x_full[utils.order_pyscf2my(p.nc, p.no, p.nv)]
    _, my_rows = utils.cvs_order_pyscf2my(p.nc, p.no, p.nv, *core_ab)
    assert np.allclose(v, utils.so2st(v_full_my, p.nc, p.no, p.nv)[my_rows], atol=1e-14)
    d = td.xycv_a - td.xycv_b
    assert np.allclose(td.dS2, np.einsum("ij,ij->i", d, d))


@pytest.mark.parametrize("tag", ["roks_gga_no1", "uks_gga_no1", "roks_mgga_no2"])
def test_cvs_driver_from_object(torch_cuda, tag):
    """The GPU-class driver built from the stand-in mean-field objects (adapters.from_pyscf, packed tensor) with core_idx: operator
    and roots against the oracle's P A P of the same problem."""
    import os
    from xtddft_b200.XTDA_GPU import XTDA
    here = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
    d = np.load(os.path.join(here, f"xtda_{tag}.npz"), allow_pickle=False)
    prm = d["params"]
    nc, no, nv, naux, ng, seed = [int(x) for x in prm[:6]]
    restricted = bool(prm[6]) if len(prm) > 6 else True
    p = make_problem(nc + no + nv, nc, no, nv, naux, ng, xctype=str(d["xctype"]), hyb=float(d["hyb"]), restricted=restricted, seed=seed)
    core, core_ab = _core(p, 1)
    rows = utils.cvs_rows(p.nc, p.no, p.nv, *core_ab)
    with fake_scf() as (FakeROKS, FakeUKS):
        mf = (FakeROKS if restricted else FakeUKS)(p)
        mf.with_df = packed_df(p)
        td = XTDA(mf.mol, mf, nstates=3, core_idx=core)
        vind, hd = td.gen_vind(mf)
        z = np.random.default_rng(1).standard_normal((2, rows.size))
        ref, hd_ref = _cvs_ref(p, core_ab, z)
        assert _rel(vind(z), ref) < RTOL
        assert np.abs(hd - hd_ref).max() < 1e-12
        e, v = td.kernel()
    w = np.linalg.eigvalsh(_pap(p, core_ab))
    assert np.abs(e - w[:3]).max() < 1e-8, (e, w[:3])
    assert v.shape == (rows.size, 3)
