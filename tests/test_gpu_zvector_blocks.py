"""The Z-vector right-hand side and W matrix from `xtd_block_response` on the operator engine's resident blocks, on the B200 through
the C-ABI: against the fixtures of the reference's own `grad_elec`, the oracle, the FP64 path (emulated path), forced aux / grid chunks,
two shards and the whole-MO-space route."""
import numpy as np
import pytest

from oracle import zvector as ozv
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


def _rhs_w(p, eng, v, z):
    from xtddft_b200.zvector import assemble_rhs, assemble_w, block_callables, rhs_intermediates
    resp, sfx, full = block_callables(p, eng.plan, eng.block_response)
    inter = rhs_intermediates(p, v, resp, sfx)
    return assemble_rhs(p, v, None, None, inter=inter), assemble_w(p, z, inter, full)


def _ref(p, v, z):
    if p.restricted:
        return ozv.roks_rhs(p, v), ozv.roks_w_matrix(p, v, z)
    return np.hstack([w.ravel() for w in ozv.uks_rhs(p, v)]), ozv.uks_w_matrix(p, v, z)


@pytest.mark.parametrize("tag", TAGS)
def test_fixtures(torch_cuda, golden_dir, tag):
    """`ZVector.rhs` / `w_matrix` on the default route build no further engine and reproduce the reference; the solve as well."""
    from xtddft_b200.zvector import ZVector
    d, p = load_case(golden_dir, tag)
    zv = ZVector(p, workspace_bytes=512 << 20)
    rhs = zv.rhs(d["amp"].reshape(p.nc, p.nv))
    assert _rel(rhs, d["rhs"]) < RTOL
    assert _rel(zv.w_matrix(d["z"]), d["im0"]) < RTOL
    assert getattr(zv, "_rhs_engines", None) is None
    z = zv.solve(rhs, tol=1e-11, max_cycle=zv.dim)
    assert np.abs(z - d["z"]).max() < 1e-8 * max(1.0, np.abs(d["z"]).max())
    zv.engine.close()


@pytest.mark.parametrize("xct,hyb,kw", [("GGA", 0.2, {}), ("LDA", 0.0, {}), ("HF", 1.0, {}), ("MGGA", 0.3, {}),
                                        ("GGA", 0.25, dict(omega=0.33, alpha=0.65))])
@pytest.mark.parametrize("no", [1, 2])
@pytest.mark.parametrize("restricted", [True, False])
def test_oracle(torch_cuda, xct, hyb, kw, no, restricted):
    p = make_problem(22 + no, 5, no, 17, 23, 300, xctype=xct, hyb=hyb, restricted=restricted, seed=410 + no, **kw)
    rng = np.random.default_rng(7)
    v = rng.standard_normal((p.nc, p.nv))
    z = rng.standard_normal(planmod.build_zvector_plan(p).ext_dim)
    ref_rhs, ref_w = _ref(p, v, z)
    eng = _engine(p, exchange_slices=0)
    rhs, w = _rhs_w(p, eng, v, z)
    eng.close()
    assert _rel(rhs, ref_rhs) < RTOL and _rel(w, ref_w) < RTOL


@pytest.mark.parametrize("xct,hyb,kw", [("LDA", 0.3, {}), ("GGA", 0.2, {}), ("MGGA", 0.25, {}), ("LDA", 0.0, {}),
                                        ("GGA", 0.25, dict(omega=0.33, alpha=0.65))])
@pytest.mark.parametrize("restricted", [True, False])
def test_emulated_against_fp64(torch_cuda, xct, hyb, kw, restricted):
    """6 digit planes: Lvv decoded from its int8 image, the fp64 virtual MO values kept beside the grid planes."""
    p = make_problem(40, 6, 2, 32, 30, 600, xctype=xct, hyb=hyb, restricted=restricted, seed=420, **kw)
    rng = np.random.default_rng(8)
    v = rng.standard_normal((p.nc, p.nv))
    z = rng.standard_normal(planmod.build_zvector_plan(p).ext_dim)
    out = []
    for slices in (0, 6):
        eng = _engine(p, exchange_slices=slices)
        out.append(_rhs_w(p, eng, v, z))
        eng.close()
    assert _rel(out[1][0], out[0][0]) < RTOL and _rel(out[1][1], out[0][1]) < RTOL
    ref_rhs, ref_w = _ref(p, v, z)
    assert _rel(out[1][0], ref_rhs) < RTOL and _rel(out[1][1], ref_w) < RTOL


@pytest.mark.parametrize("slices", [0, 6])
@pytest.mark.parametrize("restricted", [True, False])
def test_forced_chunks_and_tail_tiles(torch_cuda, monkeypatch, slices, restricted):
    """XTD_CHUNK_AUX / XTD_CHUNK_GRID force several aux and grid chunks; occupied and virtual counts past 128 take the tail tiles."""
    monkeypatch.setenv("XTD_CHUNK_AUX", "8")
    monkeypatch.setenv("XTD_CHUNK_GRID", "128")
    p = make_problem(135 + 3 + 131, 135, 3, 131, 29, 700, xctype="GGA", hyb=0.25, restricted=restricted, seed=430)
    rng = np.random.default_rng(9)
    v = rng.standard_normal((p.nc, p.nv))
    z = rng.standard_normal(planmod.build_zvector_plan(p).ext_dim)
    eng = _engine(p, exchange_slices=slices)
    rhs, w = _rhs_w(p, eng, v, z)
    aux, grid = eng.last_chunks()
    eng.close()
    assert aux >= 4 and grid >= 5
    ref_rhs, ref_w = _ref(p, v, z)
    assert _rel(rhs, ref_rhs) < RTOL and _rel(w, ref_w) < RTOL


@pytest.mark.parametrize("restricted", [True, False])
def test_shards_sum_to_whole(torch_cuda, restricted):
    """world = 2 shards of the aux functions and grid points, one after the other on this GPU: the partial outputs (what the
    all-reduce adds) sum to the world = 1 outputs."""
    p = make_problem(30, 5, 2, 23, 27, 500, xctype="GGA", hyb=0.25, restricted=restricted, seed=440, omega=0.33, alpha=0.65)
    rng = np.random.default_rng(10)
    pl = planmod.build_zvector_plan(p)
    sizes = [c.no * c.no + c.nv * c.nv + c.no * c.nv for c in pl.channels]
    dens = rng.standard_normal(sum(sizes))
    x = rng.standard_normal(pl.channels[1].no * pl.channels[0].nv)
    coef = (1.0, -0.25, -0.4, 0.7, 1.3)

    def run(**kw):
        eng = _engine(p, exchange_slices=0, **kw)
        r = eng.block_response(dens, coef, x)
        eng.close()
        return r
    whole = run()
    parts = [run(rank=r, world=2) for r in range(2)]
    for k in range(2):
        assert np.abs(parts[0][k] + parts[1][k] - whole[k]).max() <= 1e-11 * max(1.0, np.abs(whole[k]).max())


def test_mo_space_route_at_config4_orbital_shape(torch_cuda):
    """The whole-MO-space route (three more engines) against the block route at the orbital counts of config 4 (nc 136, nv 821),
    with few aux functions and grid points; both on the engines' default (emulated) exchange at this size."""
    from xtddft_b200.zvector import ZVector
    p = make_problem(136 + 1 + 821, 136, 1, 821, 12, 2000, xctype="GGA", hyb=0.2, restricted=True, seed=450)
    rng = np.random.default_rng(11)
    v = rng.standard_normal((p.nc, p.nv))
    v /= np.linalg.norm(v)
    zv = ZVector(p, workspace_bytes=2 << 30)
    z = rng.standard_normal(zv.dim)
    rb = zv.rhs(v)
    wb = zv.w_matrix(z)
    assert getattr(zv, "_rhs_engines", None) is None
    rm = zv.rhs(v, workspace_bytes=2 << 30, route="mo_space")
    wm = zv.w_matrix(z)
    assert _rel(rb, rm) < RTOL and _rel(wb, wm) < RTOL
    for e in set(e for e in zv._rhs_engines if e is not None):
        e.close()
    zv.engine.close()
