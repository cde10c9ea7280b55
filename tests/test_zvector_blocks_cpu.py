"""The block bookkeeping of the Z-vector right-hand side and W matrix on the operator plan's index sets (`zvector.block_callables`),
fed by the NumPy restatement of `xtd_block_response`, against the reference's own `w` / `(wvoa, wvob)` and `im0`."""
import os

import numpy as np
import pytest

from block_response_ref import block_response_numpy
from oracle import zvector as ozv
from xtddft_b200 import plan as planmod
from xtddft_b200.synth import make_problem
from xtddft_b200.zvector import assemble_rhs, assemble_w, block_callables, mo_to_blocks, rhs_intermediates

TAGS = ["roks_gga_no2", "roks_lda_no3", "roks_hf_no2", "uks_gga_no2", "uks_lda_pure_no2"]


def _rel(a, b):
    return float(np.abs(a - b).max() / max(1.0, np.abs(b).max()))


def _rhs_w(p, v, z):
    plan = planmod.build_zvector_plan(p)
    resp, sfx, full = block_callables(p, plan, lambda d, c, x: block_response_numpy(p, plan, d, c, x))
    inter = rhs_intermediates(p, v, resp, sfx)
    return assemble_rhs(p, v, None, None, inter=inter), assemble_w(p, z, inter, full)


@pytest.mark.parametrize("tag", TAGS)
def test_blocks_reproduce_the_reference(golden_dir, tag):
    d = np.load(os.path.join(golden_dir, f"zvector_{tag}.npz"), allow_pickle=False)
    nc, no, nv, naux, ng, seed, restricted = [int(x) for x in d["params"]]
    p = make_problem(nc + no + nv, nc, no, nv, naux, ng, xctype=str(d["xctype"]), hyb=float(d["hyb"]), restricted=bool(restricted), seed=seed)
    rhs, im0 = _rhs_w(p, d["amp"].reshape(p.nc, p.nv), d["z"])
    assert _rel(rhs, d["rhs"]) < 1e-12
    assert _rel(im0, d["im0"]) < 1e-12


@pytest.mark.parametrize("xct,hyb,kw", [("MGGA", 0.2, {}), ("GGA", 0.25, dict(omega=0.33, alpha=0.65))])
@pytest.mark.parametrize("restricted", [True, False])
def test_blocks_against_oracle(xct, hyb, kw, restricted):
    """Meta-GGA (tau) and range-separated (long-range exchange in W only) cases the fixtures do not cover."""
    p = make_problem(11, 3, 2, 6, 9, 30, xctype=xct, hyb=hyb, restricted=restricted, seed=93, **kw)
    rng = np.random.default_rng(3)
    v = rng.standard_normal((p.nc, p.nv))
    dim = planmod.build_zvector_plan(p).ext_dim
    z = rng.standard_normal(dim)
    rhs, im0 = _rhs_w(p, v, z)
    ref = ozv.roks_rhs(p, v) if restricted else np.hstack([w.ravel() for w in ozv.uks_rhs(p, v)])
    ref_w = ozv.roks_w_matrix(p, v, z) if restricted else ozv.uks_w_matrix(p, v, z)
    assert _rel(rhs, ref) < 1e-12
    assert _rel(im0, ref_w) < 1e-12


def test_non_symmetric_density_is_rejected():
    p = make_problem(9, 3, 1, 5, 7, 0, xctype="HF", hyb=1.0, seed=4)
    t = np.zeros((2, p.nmo, p.nmo))
    t[0, 0, 5] = 1.0
    with pytest.raises(ValueError):
        mo_to_blocks(planmod.build_zvector_plan(p), t)
