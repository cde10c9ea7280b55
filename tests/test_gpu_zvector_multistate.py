"""Several Z-vector states at once on the B200: `xtd_block_response_batch` against single `xtd_block_response` calls (FP64 and emulated
exchange, forced aux / grid chunks, density batches split inside the call, two shards), the five fixtures as members of a batch,
`ZVector.solve_many` against `solve`, and the config-4 orbital shape."""
import numpy as np
import pytest

from test_zvector_cpu import TAGS, load_case
from xtddft_b200 import plan as planmod
from xtddft_b200.synth import make_problem

pytestmark = pytest.mark.gpu

RTOL = 1e-9


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


def _rel(got, ref):
    return float(np.abs(got - ref).max() / max(1.0, np.abs(ref).max()))


def _engine(p, **kw):
    from xtddft_b200.engine import SigmaEngine
    pl = planmod.build_zvector_plan(p)
    pl.block_response = True
    return SigmaEngine.from_problem(pl, p, workspace_bytes=kw.pop("workspace_bytes", 512 << 20), max_nvec=4, **kw)


def _inputs(pl, k, seed):
    """k random symmetric densities in the block layout and k mixed-spin X blocks."""
    rng = np.random.default_rng(seed)
    dens = []
    for _ in range(k):
        parts = []
        for c in pl.channels:
            n = c.no + c.nv
            m = rng.standard_normal((n, n))
            m = m + m.T
            parts += [m[:c.no, :c.no].ravel(), m[c.no:, c.no:].ravel(), m[:c.no, c.no:].ravel()]
        dens.append(np.concatenate(parts))
    x = rng.standard_normal((k, pl.channels[1].no, pl.channels[0].nv))
    return np.stack(dens), x


def _check_batch(eng, k, seed, coef, tol=1e-12):
    dens, x = _inputs(eng.plan, k, seed)
    out, xo = eng.block_response(dens, coef, x)
    counters = eng.last_chunks() + (eng.last_density_batches(),)      # of the batched call, before the single calls below
    assert out.shape[0] == k and xo.shape[0] == k
    for i in range(k):
        o1, x1 = eng.block_response(dens[i], coef, x[i])
        assert _rel(out[i], o1) < tol, (i, _rel(out[i], o1))
        assert _rel(xo[i], x1) < tol, (i, _rel(xo[i], x1))
    return counters


COEF = (1.0, -0.25, -0.4, 0.7, 1.3)


@pytest.mark.parametrize("slices", [0, 6])
@pytest.mark.parametrize("xct,hyb,kw", [("GGA", 0.2, {}), ("LDA", 0.0, {}), ("HF", 1.0, {}), ("MGGA", 0.3, {}),
                                        ("GGA", 0.25, dict(omega=0.33, alpha=0.65))])
@pytest.mark.parametrize("restricted", [True, False])
def test_batch_matches_single_calls(torch_cuda, slices, xct, hyb, kw, restricted):
    """k in {1, 2, 3, 5} densities in one call against k single calls on the same engine (FP64 DMMA or 6-plane emulated exchange)."""
    p = make_problem(40, 6, 2, 32, 30, 600, xctype=xct, hyb=hyb, restricted=restricted, seed=520, **kw)
    eng = _engine(p, exchange_slices=slices)
    coef = (1.0, -0.25 if p.hybrid else 0.0, -0.4 if p.omega != 0.0 else 0.0, 0.7, 1.3 if p.hybrid else 0.0)
    for k in (1, 2, 3, 5):
        assert _check_batch(eng, k, 600 + k, coef)[2] == 1
    eng.close()


@pytest.mark.parametrize("slices", [0, 6])
@pytest.mark.parametrize("restricted", [True, False])
def test_forced_chunks_and_split_batches(torch_cuda, monkeypatch, slices, restricted):
    """XTD_CHUNK_AUX / XTD_CHUNK_GRID force several aux and grid chunks; a workspace that cannot hold six densities makes the call
    split them into passes, which the counter reports, with the same results."""
    monkeypatch.setenv("XTD_CHUNK_AUX", "8")
    monkeypatch.setenv("XTD_CHUNK_GRID", "128")
    p = make_problem(135 + 3 + 331, 135, 3, 331, 29, 700, xctype="GGA", hyb=0.25, restricted=restricted, seed=530)
    split = False
    for mb in (64, 48, 40):
        eng = _engine(p, exchange_slices=slices, workspace_bytes=mb << 20)
        aux, grid, nb = _check_batch(eng, 6, 610, (1.0, -0.25, 0.0, 0.7, 1.3))
        eng.close()
        assert aux >= 4 and grid >= 5
        if nb > 1:
            split = True
            break
    assert split


@pytest.mark.parametrize("restricted", [True, False])
def test_shards_sum_to_whole(torch_cuda, restricted):
    """world = 2 shards of the aux functions and grid points, one after the other on this GPU: the batched partial outputs sum to the
    world = 1 batched outputs."""
    p = make_problem(30, 5, 2, 23, 27, 500, xctype="GGA", hyb=0.25, restricted=restricted, seed=540, omega=0.33, alpha=0.65)
    pl = planmod.build_zvector_plan(p)
    dens, x = _inputs(pl, 3, 620)

    def run(**kw):
        eng = _engine(p, exchange_slices=0, **kw)
        r = eng.block_response(dens, COEF, x)
        eng.close()
        return r
    whole = run()
    parts = [run(rank=r, world=2) for r in range(2)]
    for j in range(2):                          # the responses, then K[X]
        assert np.abs(parts[0][j] + parts[1][j] - whole[j]).max() <= 1e-11 * max(1.0, np.abs(whole[j]).max())


@pytest.mark.parametrize("tag", TAGS)
def test_fixtures_inside_a_batch(torch_cuda, golden_dir, tag):
    """Each fixture state in the middle of a batch of three gives its golden right-hand side, W matrix and (solve_many) solution;
    no further engine is built."""
    from xtddft_b200.zvector import ZVector
    d, p = load_case(golden_dir, tag)
    zv = ZVector(p, workspace_bytes=512 << 20)
    rng = np.random.default_rng(21)
    V = np.stack([rng.standard_normal((p.nc, p.nv)), d["amp"].reshape(p.nc, p.nv), rng.standard_normal((p.nc, p.nv))])
    rhs = zv.rhs_many(V)
    assert rhs.shape == (3, zv.dim)
    assert _rel(rhs[1], d["rhs"]) < RTOL
    Z = np.stack([rng.standard_normal(zv.dim), d["z"], rng.standard_normal(zv.dim)])
    w = zv.w_matrices(Z)
    assert _rel(w[1], d["im0"]) < RTOL
    z = zv.solve_many(rhs, tol=1e-11, max_cycle=zv.dim)
    assert zv.converged.all()
    assert np.abs(z[1] - d["z"]).max() < 1e-8 * max(1.0, np.abs(d["z"]).max())
    assert getattr(zv, "_rhs_engines", None) is None
    zv.engine.close()


@pytest.mark.parametrize("restricted", [True, False])
def test_solve_many_against_solve(torch_cuda, restricted):
    """k = 5 states with max_nvec = 4: every solution matches `solve` on that state to the solver tolerance, every residual is below
    tol, and the block solve makes fewer operator calls than the single solves' cycles added up."""
    from xtddft_b200.zvector import ZVector
    p = make_problem(40, 6, 2, 32, 30, 600, xctype="GGA", hyb=0.25, restricted=restricted, seed=550)
    zv = ZVector(p, workspace_bytes=512 << 20, max_nvec=4)
    rng = np.random.default_rng(23)
    V = rng.standard_normal((5, p.nc, p.nv))
    rhs = zv.rhs_many(V)
    tol = 1e-10
    z = zv.solve_many(rhs, tol=tol, max_cycle=60)
    calls, res = zv.aop_calls, zv.residual.copy()
    assert zv.converged.all() and (res < tol).all()
    single = []
    for i in range(5):
        zi = zv.solve(rhs[i], tol=tol, max_cycle=60)
        assert zv.converged
        single.append(zv.cycles)
        # both solutions leave residuals below tol, so they differ by at most ~ tol times the inverse's norm
        assert np.abs(z[i] - zi).max() < 1e3 * tol * max(1.0, np.abs(zi).max())
    assert calls < sum(single), (calls, single)
    zv.engine.close()


def test_config4_orbital_shape(torch_cuda):
    """k = 4 states at the orbital counts of config 4 (nc 136, nv 821) with few aux functions and grid points, on one engine and its
    workspace, against single-state calls."""
    from xtddft_b200.zvector import ZVector
    p = make_problem(136 + 1 + 821, 136, 1, 821, 12, 2000, xctype="GGA", hyb=0.2, restricted=True, seed=560)
    zv = ZVector(p, workspace_bytes=2 << 30)
    rng = np.random.default_rng(25)
    V = rng.standard_normal((4, p.nc, p.nv))
    V /= np.linalg.norm(V, axis=(1, 2), keepdims=True)
    Z = rng.standard_normal((4, zv.dim))
    rhs = zv.rhs_many(V)
    w = zv.w_matrices(Z)
    for i in range(4):
        assert _rel(rhs[i], zv.rhs(V[i])) < RTOL
        assert _rel(w[i], zv.w_matrix(Z[i])) < RTOL
    zv.engine.close()
