"""SURVEY 8f row f3 on the B200: the Z-vector operator (engine plan with the transposed-density exchange term and the transposed local
couplings) against the fixtures of the reference's own `matvec` / `fvind` closures and against the oracle, through the C-ABI; the
device Krylov solve against dense solves of the oracle's operator.  Needs a B200."""
import numpy as np
import pytest

from oracle import zvector as ozv
from test_zvector_cpu import TAGS, load_case
from xtddft_b200 import plan as planmod
from xtddft_b200.synth import make_problem

pytestmark = pytest.mark.gpu

RTOL = 1e-9     # north_star tolerance on operator images


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


def _rel(got, ref):
    return float(np.abs(got - ref).max() / max(1.0, np.abs(ref).max()))


def _engine(p, with_diag=False, **kw):
    from xtddft_b200.engine import SigmaEngine
    pl = planmod.build_zvector_plan(p, with_diag=with_diag)
    return SigmaEngine.from_problem(pl, p, workspace_bytes=kw.pop("workspace_bytes", 512 << 20), max_nvec=kw.pop("max_nvec", 6), **kw), pl


@pytest.mark.parametrize("tag", TAGS)
def test_operator_golden(torch_cuda, golden_dir, tag):
    """The CUDA operator reproduces what the reference's own closures returned (tests/golden/make_golden_zvector.py)."""
    d, p = load_case(golden_dir, tag)
    eng, _ = _engine(p)
    got = eng.sigma(torch_cuda.from_numpy(d["x"]).cuda()).cpu().numpy()
    assert _rel(got, d["ax"]) < RTOL
    assert np.abs(eng.sigma_host(d["x"]) - got).max() == 0.0
    eng.close()


@pytest.mark.parametrize("xct,hyb,kw", [("GGA", 0.2, {}), ("LDA", 0.0, {}), ("HF", 1.0, {}), ("MGGA", 0.3, {}),
                                        ("GGA", 0.25, dict(omega=0.33, alpha=0.65))])
@pytest.mark.parametrize("no", [1, 2])
@pytest.mark.parametrize("restricted", [True, False])
def test_operator_oracle(torch_cuda, xct, hyb, kw, no, restricted):
    p = make_problem(22 + no, 5, no, 17, 23, 300, xctype=xct, hyb=hyb, restricted=restricted, seed=400 + no, **kw)
    eng, pl = _engine(p)
    op = ozv.roks_matvec(p) if restricted else ozv.uks_fvind(p)
    z = np.random.default_rng(3).standard_normal((4, pl.ext_dim))
    got = eng.sigma(torch_cuda.from_numpy(z).cuda()).cpu().numpy()
    assert _rel(got, np.stack([op(x) for x in z])) < RTOL
    eng.close()


@pytest.mark.parametrize("restricted", [True, False])
@pytest.mark.parametrize("slices", [0, 6])
def test_operator_many_tiles_and_aux_chunks(torch_cuda, monkeypatch, restricted, slices):
    """More than 16384 elements per block (the local couplings, transposed ones included, run as DMMA GEMMs instead of the one-launch
    small-problem kernel), several 128-tiles in every GEMM dimension, 9 auxiliary-function chunks in both exchange terms (direct and transposed), odd
    block sizes; slices = 6: the direct exchange and the grid GEMMs on the INT8-emulated path, the transposed term on FP64 DMMA."""
    monkeypatch.setenv("XTD_CHUNK_AUX", "8")
    monkeypatch.setenv("XTD_OZ_SHORT_K", "0")
    p = make_problem(343, 60, 3, 280, 68, 700, xctype="GGA", hyb=0.4, restricted=restricted, seed=410)
    eng, pl = _engine(p, workspace_bytes=(2 << 30) if slices else (256 << 20), exchange_slices=slices)
    op = ozv.roks_matvec(p) if restricted else ozv.uks_fvind(p)
    z = np.random.default_rng(4).standard_normal((5, pl.ext_dim))
    got = eng.sigma(torch_cuda.from_numpy(z).cuda()).cpu().numpy()
    assert eng.last_chunks()[0] == 9
    assert _rel(got, np.stack([op(x) for x in z])) < RTOL
    eng.close()


@pytest.mark.parametrize("restricted", [True, False])
def test_solve(torch_cuda, restricted):
    """`ZVector.solve` (Krylov vectors in HBM, `xtd_vec_*` subspace algebra) against LAPACK on the oracle's dense operator, with the
    right-hand side the oracle builds from a seeded amplitude vector (tdroks_sfu.py:207-274 / tduks_sfu.py:205-244)."""
    from xtddft_b200.zvector import ZVector
    p = make_problem(30, 5, 2, 23, 25, 320, xctype="GGA", hyb=0.25, restricted=restricted, seed=420)
    v = np.random.default_rng(6).standard_normal((p.nc, p.nv))
    v /= np.linalg.norm(v)
    zv = ZVector(p, workspace_bytes=512 << 20)
    if restricted:
        rhs = ozv.roks_rhs(p, v)
        ref = ozv.roks_solve(p, rhs)
        az = zv.matvec(ref)
        assert _rel(az, rhs) < 1e-9
    else:
        wa, wb = ozv.uks_rhs(p, v)
        rhs = np.hstack([wa.ravel(), wb.ravel()])
        ref = ozv.uks_solve(p, wa, wb)
    z = zv.solve(rhs, tol=1e-11, max_cycle=80)
    assert zv.converged and zv.cycles < 80
    assert np.abs(z - ref).max() < 1e-9 * max(1.0, np.abs(ref).max())
    blocks = zv.split(z)
    assert sum(b.size for b in blocks) == zv.dim
    zv.engine.close()


def test_workload_route_solves(torch_cuda):
    """The bench's route (device-generated BASELINE config-4 inputs at 1/8 scale, tensor streamed block by block): the device solve
    converges and the solution satisfies the equation under an independent application of the operator."""
    import dataclasses
    from xtddft_b200.synth_device import make_device_problem
    from xtddft_b200.workloads import engine_for_device_problem
    from xtddft_b200.zvector import solve_linear
    dp = dataclasses.replace(make_device_problem(4, 0.125), method="zvector")
    eng = engine_for_device_problem(dp, max_nvec=4, workspace_bytes=1 << 30)
    rhs = np.random.default_rng(9).standard_normal(eng.ext_dim)
    rhs /= np.linalg.norm(rhs)
    x, conv, cycles, res = solve_linear(eng.sigma, rhs, eng.plan.hdiag, tol=1e-9, max_cycle=60)
    assert conv and res < 1e-9
    ax = eng.sigma_host(x[None])[0]
    assert np.abs(ax - rhs).max() < 1e-8
    eng.close()


@pytest.mark.parametrize("tag", TAGS)
def test_rhs_and_w_matrix_on_device(torch_cuda, golden_dir, tag):
    """`ZVector.rhs` / `ZVector.w_matrix` (whole-MO-space engine plans) against the right-hand side and the W matrix the reference's own
    `grad_elec` built."""
    from xtddft_b200.zvector import ZVector
    d, p = load_case(golden_dir, tag)
    zv = ZVector(p, workspace_bytes=512 << 20)
    rhs = zv.rhs(d["amp"].reshape(p.nc, p.nv), workspace_bytes=512 << 20)
    assert _rel(rhs, d["rhs"]) < RTOL
    assert _rel(zv.w_matrix(d["z"]), d["im0"]) < RTOL
    z = zv.solve(rhs, tol=1e-11, max_cycle=zv.dim)
    assert np.abs(z - d["z"]).max() < 1e-8 * max(1.0, np.abs(d["z"]).max())
