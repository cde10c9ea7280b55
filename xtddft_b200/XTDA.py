"""X-TDA driver (spin-conserving spin-adapted TDA for ROKS / UKS references) on the B200 sigma engine.

Same constructor, `kernel()` / `Davidson()` entry points, options and result attributes as the reference classes
`XTDA` in xtddft/XTDA.py:21-54,694-829 (CPU) and xtddft/XTDA_GPU.py:24-53,368-500 (GPU); the sigma build
`vind` (XTDA.py:615-690) runs in libxtdsigma.so, and so does the property pass after the solve (oscillator and
rotatory strengths, XTDA.py:838-890 -> xtddft_b200/properties.py).  The dense debug paths (`full_diag`, `X_TDA` tensor
basis) are outside the hot path and raise NotImplementedError.
"""
from __future__ import annotations

import functools

import numpy as np

from . import plan as planmod
from . import utils
from .adapters import is_chiral, one_electron_ints, problem_from_mf
from .drivers_common import TimeCounter, solve, timed_engine


class XTDA:
    core_idx = None
    cvs_rows = None                 # rows of the core-valence-separated layout inside the full PySCF order (None: full space)

    def __init__(self, mol, mf, nstates=10, basis="orbital", so2st=True, use_Davidson=True, core_idx=None):
        self.mol, self.mf = mol, mf
        self.nstates = nstates
        self.basis = basis
        self.so2st = so2st
        self.use_Davidson = use_Davidson
        # pyscf.tdscf.rhf.TDBase defaults the reference copies (XTDA.py:29-31)
        self.conv_tol, self.lindep, self.max_cycle = 1e-5, 1e-12, 100
        self.deg_eia_thresh, self.positive_eig_threshold = 1e-3, 1e-3
        self.problem = problem_from_mf(mf, kernel="uks")
        self.X = bool(self.problem.restricted)
        # core-valence separation (K-edge states): keep only excitations out of these occupied orbitals -- closed-shell indices
        # on a ROKS reference, a pair (core_a, core_b) of occupied indices per spin on a UKS reference
        self.core_idx = core_idx
        if core_idx is not None:
            p = self.problem
            self._core = planmod.cvs_core(p, core_idx)
            self.cvs_rows = utils.cvs_rows(p.nc, p.no, p.nv, *self._core)
        self.tc = TimeCounter()
        self._settings = "xtda"
        self._engine = None

    # ---- operator interface (XTDA.py:694-698) ----------------------------------------------------------
    def _get_engine(self):
        if self._engine is None:
            build = functools.partial(planmod.build_xtda_plan, core=self.core_idx)
            self._engine = timed_engine(self.tc, build, self.problem, max_nvec=40)
            self.plan = self._engine.plan
        return self._engine

    def gen_vind(self, mf=None):
        assert mf is None or mf is self.mf
        eng = self._get_engine()
        return eng.as_vind(), eng.hdiag()

    def get_init_guess(self, mf=None, nstates=None, wfnsym=None, return_symmetry=False):
        """Koopmans unit vectors on the lowest orbital-energy gaps (+1e-3 window), XTDA.py:700-734."""
        from .davidson import init_guess
        p = self.problem
        ea, eb = p.mo_energy
        e_a = ea[p.nocc_a:] - ea[:p.nocc_a, None]
        e_b = eb[p.nocc_b:] - eb[:p.nocc_b, None]
        gaps = np.append(e_a.ravel(), e_b.ravel())
        if self.cvs_rows is not None:
            gaps = gaps[self.cvs_rows]
        return init_guess(gaps, self.nstates if nstates is None else nstates, self.deg_eia_thresh)

    init_guess = get_init_guess

    def kernel(self, x0=None, nstates=None):
        if self.basis == "tensor":
            raise NotImplementedError("tensor-basis X_TDA is a dense O(N^4) reference path, outside the sigma hot path")
        if self.basis != "orbital":
            raise ValueError("basis must be tensor or orbital")
        if not self.use_Davidson:
            raise NotImplementedError("full_diag is a dense debug path, outside the sigma hot path")
        return self.Davidson(x0=x0, nstates=nstates), self.v

    def Davidson(self, x0=None, nstates=None):
        if nstates is not None:
            self.nstates = nstates
        p = self.problem
        eng = self._get_engine()
        if x0 is None:
            x0 = self.get_init_guess(self.mf, self.nstates)
        over = dict(tol_residual=self.conv_tol, lindep=self.lindep, max_cycle=self.max_cycle)
        self.converged, self.e, x1, self.Davidcyc, _ = solve(eng, self.nstates, self._settings, x0=x0, tc=self.tc, **over)
        nc, no, nv = p.nc, p.no, p.nv
        nocca, noccb, nvira = nc + no, nc, nv
        self.nc, self.no, self.nv = nc, no, nv
        self.order = utils.order_pyscf2my(nc, no, nv)
        self._x_rows = np.ascontiguousarray(x1.T)          # PySCF-order amplitude rows for the property pass
        if self.cvs_rows is None:
            self.v = x1[self.order, :]
            vfull = self.v
        else:
            # v: the core rows of the order_pyscf2my layout; the block attributes below are slices of the zero-padded full vectors
            order, _ = utils.cvs_order_pyscf2my(nc, no, nv, *self._core)
            self.v = x1[order, :]
            vfull = self.cvs_embed(x1)[self.order, :]
        self.xy_a = vfull.T[:, :nocca * nvira]
        self.xy_b = vfull.T[:, nocca * nvira:]
        self.xycv_a = vfull.T[:, :noccb * nvira]
        self.xyov_a = vfull.T[:, noccb * nvira:nocca * nvira]
        self.xyco_b = vfull.T[:, nocca * nvira:nocca * nvira + noccb * no]
        self.xycv_b = vfull.T[:, nocca * nvira + noccb * no:]
        self.dS2 = self.deltaS2()
        self.os = self.osc_str()                           # None when no dipole integrals are available
        self.rs = self.rot_str() if is_chiral(self.mf, p) else np.zeros(self.nstates)     # XTDA.py:818-821
        if self.so2st:
            self.v = utils.so2st(self.v, nc, no, nv, core=None if self.cvs_rows is None else self._core)
        return self.e

    def cvs_embed(self, v):
        """Core-valence-separated vectors (rows in the engine's PySCF order: alpha (core i, a), then beta (core i, a)) zero-padded
        into the full PySCF-order layout [alpha (i, a) | beta (i, a)], for tools that expect full-space amplitudes."""
        if self.cvs_rows is None:
            raise ValueError("cvs_embed: this object was built without core_idx")
        p = self.problem
        return utils.cvs_embed(v, self.cvs_rows, p.nocc_a * p.nvir_a + p.nocc_b * p.nvir_b)

    def deltaS2(self):
        """XTDA.py:831-836: |X_cv(aa) - X_cv(bb)|^2."""
        d = self.xycv_a - self.xycv_b
        return np.einsum("ij,ij->i", d, d)

    def _property_pass(self):
        from .properties import PropertyPass
        if getattr(self, "_pp", None) is None:
            self._pp = PropertyPass(self.problem)
        return self._pp

    def osc_str(self):
        """Length-form oscillator strengths f = 2/3 w |<0|r|n>|^2 (XTDA.py:838-858), on the device."""
        dip = one_electron_ints(self.mf, self.problem, "int1e_r")
        if dip is None:
            return None
        return self._property_pass().xtda_osc_str(self.e[:self.nstates], self._x_rows, dip, self.cvs_rows)

    def rot_str(self):
        """Rotatory strengths in cgs units (XTDA.py:860-890), on the device."""
        ipo = one_electron_ints(self.mf, self.problem, "int1e_ipovlp")
        rxp = one_electron_ints(self.mf, self.problem, "int1e_cg_irxp")
        if ipo is None or rxp is None:
            return None
        return self._property_pass().xtda_rot_str(self.e[:self.nstates], self._x_rows, ipo, rxp, self.cvs_rows)

    def full_diag(self):
        raise NotImplementedError("full_diag is a dense O(dim^2) debug path, outside the sigma hot path")
