"""Host-side pieces of the PRODUCT (not the oracle) against the fixtures the reference's own code produced:
initial guesses (row a4: XTDA.get_init_guess, SF_TDA.init_guess, XSF_TDA._build_initial_guess_from_gaps), amplitude layouts
(row a18: order_pyscf2my, so2st, st2so, deal_v_davidson, get_vect) -- and, where XTDDFT_REFERENCE names a checkout of the
original XTDDFT source (not part of this repository), a regeneration of every fixture into a temporary directory that must
reproduce the committed files bit for bit.  CPU only."""
import os
import subprocess
import sys

import numpy as np
import pytest

from xtddft_b200 import davidson as dav
from xtddft_b200 import plan as planmod
from xtddft_b200 import utils
from xtddft_b200.synth import make_problem


def _load(golden_dir, name):
    return np.load(os.path.join(golden_dir, name), allow_pickle=False)


def _problem(d):
    prm = d["params"]
    nc, no, nv, naux, ng, seed = [int(v) for v in prm[:6]]
    restricted = bool(prm[6]) if len(prm) > 6 else True
    return make_problem(nc + no + nv, nc, no, nv, naux, ng, xctype=str(d["xctype"]), hyb=float(d["hyb"]), restricted=restricted, seed=seed)


def test_product_layout_helpers(golden_dir):
    h = _load(golden_dir, "helpers.npz")
    for (nc, no, nv) in [(2, 1, 3), (3, 2, 4), (1, 3, 2), (4, 1, 1)]:
        assert np.array_equal(utils.order_pyscf2my(nc, no, nv), h[f"order_{nc}_{no}_{nv}"])
        dim = (nc + no) * nv + nc * (no + nv)
        v = np.random.default_rng(7).standard_normal((dim, 3))
        assert np.abs(utils.so2st(v, nc, no, nv) - h[f"so2st_{nc}_{no}_{nv}"]).max() < 1e-15
        assert np.abs(utils.st2so(v, nc, no, nv) - h[f"st2so_{nc}_{no}_{nv}"]).max() < 1e-15
    for no in (2, 3, 4):
        assert np.abs(utils.get_vect(no) - h[f"vects_{no}"]).max() < 1e-15


@pytest.mark.parametrize("tag", ["down_gga", "down_lda", "down_uks", "down_mgga"])
def test_product_deal_v_davidson(golden_dir, tag):
    d = _load(golden_dir, f"sf_{tag}.npz")
    p = _problem(d)
    assert np.array_equal(utils.deal_v_davidson(d["deal_in"], p.nc, p.no, p.nv), d["deal_out"])


@pytest.mark.parametrize("tag", ["roks_gga_no1", "roks_gga_no2", "roks_lda_no3", "roks_hf_no1", "uks_gga_no1", "roks_mgga_no2"])
def test_xtda_init_guess(golden_dir, tag):
    """XTDA.get_init_guess (XTDA.py:700-734) on the orbital-energy gaps, through the product driver class."""
    from xtddft_b200.XTDA import XTDA
    d = _load(golden_dir, f"xtda_{tag}.npz")
    p = _problem(d)
    obj = XTDA.__new__(XTDA)                      # no engine: only the host-side guess
    obj.problem, obj.nstates, obj.deg_eia_thresh = p, 3, 1e-3
    assert np.array_equal(obj.get_init_guess(None, 3), d["x0"])


@pytest.mark.parametrize("tag", ["down_gga", "up_gga", "down_lda", "down_uks", "down_mgga"])
def test_sf_init_guess(golden_dir, tag):
    """SF_TDA.init_guess (SF_TDA.py:348-380): the drivers seed the solver with init_guess(hdiag, nstates, 1e-5)."""
    d = _load(golden_dir, f"sf_{tag}.npz")
    x0 = dav.init_guess(d["hdiag"], 3, dav.SOLVER["sf_down"]["window"])
    assert np.array_equal(x0, d["x0"])


@pytest.mark.parametrize("tag", ["gga_no2", "lda_no3"])
def test_xsf_init_guess(golden_dir, tag):
    """XSF_TDA._build_initial_guess_from_gaps (XSF_TDA.py:964-982) on the compressed preconditioner diagonal."""
    d = _load(golden_dir, f"xsf_{tag}.npz")
    x0 = dav.init_guess(d["hdiag_sa3_re1"], 3, dav.SOLVER["xsf"]["window"])
    assert np.array_equal(x0, d["x0"])


REFERENCE = os.environ.get("XTDDFT_REFERENCE", "")


@pytest.mark.skipif(not (REFERENCE and os.path.isdir(os.path.join(REFERENCE, "xtddft"))),
                    reason="needs XTDDFT_REFERENCE: a checkout of the original XTDDFT source, which is not part of this repository")
def test_goldens_regenerate_bit_for_bit(golden_dir, tmp_path):
    """Re-run the reference's own code (make_golden.py, make_golden_properties.py, make_golden_zvector.py) and diff against the
    committed files."""
    env = dict(os.environ, XTD_GOLDEN_OUT=str(tmp_path), OMP_NUM_THREADS="1", OPENBLAS_NUM_THREADS="1")
    for script in ("make_golden.py", "make_golden_properties.py", "make_golden_zvector.py"):
        res = subprocess.run([sys.executable, os.path.join(golden_dir, script)], env=env, capture_output=True, text=True, timeout=900)
        assert res.returncode == 0, res.stderr[-2000:]
    made = sorted(f for f in os.listdir(tmp_path) if f.endswith(".npz"))
    committed = sorted(f for f in os.listdir(golden_dir) if f.endswith(".npz"))
    assert made == committed
    for f in made:
        a, b = np.load(os.path.join(tmp_path, f), allow_pickle=False), np.load(os.path.join(golden_dir, f), allow_pickle=False)
        assert sorted(a.files) == sorted(b.files), f
        for k in a.files:
            assert a[k].shape == b[k].shape and a[k].dtype == b[k].dtype, (f, k)
            if a[k].dtype.kind == "f":
                # same code, same seeds; BLAS reductions may differ in the last bits between thread counts
                assert np.abs(a[k] - b[k]).max() <= 1e-13 * max(1.0, np.abs(b[k]).max()), (f, k)
            else:
                assert np.array_equal(a[k], b[k]), (f, k)
