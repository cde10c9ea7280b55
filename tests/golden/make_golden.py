#!/usr/bin/env python
"""Generate golden sigma vectors by executing the REFERENCE's own code (a checkout of the original XTDDFT source,
named by the XTDDFT_REFERENCE environment variable; it is not part of this repository) on seeded synthetic inputs.

What runs verbatim from the reference (after the two minimal Appendix-D fixes: the full-width comma at
XSF_TDA.py:1137 and the bare-module imports):
  * xtddft/XTDA.py          XTDA._gen_tda_operation (vind, hdiag), gen_response, get_init_guess
  * xtddft/SF_TDA.py        gen_tda_operation_sf, gen_response_sf, cache_xc_kernel_sf, nr_uks_fxc_sf_tda,
                            nr_uks_fxc_sf_tda_mc, init_guess, deal_v_davidson
  * xtddft/XSF_TDA.py       XSF_TDA.gen_tda_operation_sf (vind, hdiag incl. J diagonals), get_vect, get_Amat/remove
  * xtddft/XSF_TDA_GPU.py   XSF_TDA_GPU.gen_vind (PySCF-order, removed layout), with NumPy standing in for CuPy
  * xtddft/utils/utils.py   order_pyscf2my, so2st, st2so

What is NOT in the reference tree (third-party PySCF / gpu4pyscf, not installed, not vendored) and is
supplied by the stub below, coded independently of `oracle/` from the published definitions:
  get_jk / get_j / get_k  (J_kl = sum_ij (ij|kl) D_ji, K_il = sum_jk (ij|kl) D_jk, from a 4-index tensor),
  numint block_loop / rho evaluator / nr_uks_fxc / sparse AO helpers (dense loops), a Slater-exchange
  `eval_xc_eff`, SCF accessors (make_rdm1, get_veff, get_hcore) returning the synthetic Fock matrices.

Usage:  XTDDFT_REFERENCE=<checkout of the original XTDDFT> python tests/golden/make_golden.py
Writes tests/golden/*.npz.  Inputs are regenerated from the seed stored in each file.
"""
import importlib
import importlib.util
import math
import os
import sys
import types

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.environ.get("XTD_GOLDEN_OUT", HERE)      # tests regenerate into a temporary directory and diff
ROOT = os.path.dirname(os.path.dirname(HERE))
REF = os.environ.get("XTDDFT_REFERENCE", "")          # checkout of the original XTDDFT source
sys.path.insert(0, ROOT)

from xtddft_b200.synth import make_problem  # noqa: E402  (input generator, product side)


# =================================================================================================
# stub of the third-party API surface
# =================================================================================================
class TaggedArray(np.ndarray):
    pass


def tag(a, **kw):
    t = np.asarray(a).view(TaggedArray)
    for k, v in kw.items():
        setattr(t, k, v)
    return t


class FakeMol:
    def __init__(self, p):
        self.p = p
        self.spin = p.no
        self.symmetry = False
        self.natm = 1
        self.verbose = 0

    def nao_nr(self):
        return self.p.nao

    def ao_loc_nr(self):
        return np.arange(self.p.nao + 1)

    def get_overlap_cond(self):
        return np.zeros((self.p.nao, self.p.nao))


class FakeGrids:
    cutoff = 1e-15

    def __init__(self, p):
        self.weights = p.weights
        self.coords = None if p.weights is None else np.zeros((p.weights.size, 3))


class FakeLibxc:
    def __init__(self, p):
        self.p = p

    def test_deriv_order(self, *a, **k):
        return True

    def is_hybrid_xc(self, xc):
        return self.p.hybrid

    def is_nlc(self, xc):
        return False


CX = 0.75 * (3.0 / math.pi) ** (1.0 / 3.0)


class FakeNumInt:
    """Dense restatement of the pyscf.dft.numint pieces the reference touches."""
    cutoff = 1e-13

    def __init__(self, p, blocks=3):
        self.p = p
        self.libxc = FakeLibxc(p)
        self.blocks = blocks

    def _xc_type(self, xc):
        return self.p.xctype

    def rsh_and_hybrid_coeff(self, xc, spin=0):
        return self.p.omega, self.p.alpha, self.p.hyb

    def block_loop(self, mol, grids, nao=None, deriv=0, max_memory=2000, **kw):
        p = self.p
        ng = p.ng
        edges = np.linspace(0, ng, self.blocks + 1).astype(int)
        for b0, b1 in zip(edges[:-1], edges[1:]):
            ao = p.ao[:, b0:b1] if deriv > 0 else p.ao[0, b0:b1]
            yield ao, None, p.weights[b0:b1], None

    def _gen_rho_evaluator(self, mol, dms, hermi=0, with_lapl=False, grids=None):
        dms = np.asarray(dms)
        if dms.ndim == 2:
            dms = dms[None]
        ndms = len(dms)

        def make_rho(idm, ao, mask, xctype):
            dm = np.asarray(dms[idm])
            if xctype == "LDA" or ao.ndim == 2:
                a0 = ao if ao.ndim == 2 else ao[0]
                return np.array([a0[g] @ dm @ a0[g] for g in range(a0.shape[0])])
            ng = ao.shape[1]
            rho = np.zeros((5 if xctype == "MGGA" else 4, ng))
            for g in range(ng):
                rho[0, g] = ao[0, g] @ dm @ ao[0, g]
                for k in range(1, 4):
                    rho[k, g] = ao[k, g] @ dm @ ao[0, g] + ao[0, g] @ dm @ ao[k, g]
                if xctype == "MGGA":          # tau = 1/2 sum_k (d_k phi) D (d_k phi)   (pyscf eval_rho, no Laplacian)
                    rho[4, g] = 0.5 * sum(ao[k, g] @ dm @ ao[k, g] for k in range(1, 4))
            return rho
        return make_rho, ndms, self.p.nao

    def eval_rho2(self, mol, ao, mo_coeff, mo_occ, mask, xctype, with_lapl=False):
        dm = (mo_coeff * mo_occ) @ mo_coeff.T
        return self._gen_rho_evaluator(mol, dm)[0](0, ao, mask, xctype)

    def eval_xc_eff(self, xc, rho, deriv=1, omega=None, xctype=None, **kw):
        """Slater exchange (spin-polarised), density-only: e, v_s[2,nvar,g], f[2,nvar,2,nvar,g]."""
        ra, rb = np.asarray(rho[0]), np.asarray(rho[1])
        if ra.ndim == 1:
            ra, rb = ra[None], rb[None]
        nvar, ng = ra.shape
        vxc = np.zeros((2, nvar, ng))
        fxc = np.zeros((2, nvar, 2, nvar, ng))
        for s, r in enumerate((ra, rb)):
            r0 = np.maximum(r[0], 1e-300)
            vxc[s, 0] = -(4.0 / 3.0) * CX * 2 ** (1.0 / 3.0) * r0 ** (1.0 / 3.0)
            fxc[s, 0, s, 0] = -(4.0 / 9.0) * CX * 2 ** (1.0 / 3.0) * r0 ** (-2.0 / 3.0)
        return None, vxc, fxc, None

    def cache_xc_kernel(self, mol, grids, xc, mo_coeff, mo_occ, spin=0, max_memory=2000):
        return None, None, self.p.fxc_uks

    def nr_uks_fxc(self, mol, grids, xc, dm0, dms, relativity=0, hermi=0, rho0=None, vxc=None, fxc=None,
                   max_memory=2000, verbose=None):
        """pyscf.dft.numint.nr_uks_fxc, grid-point loops."""
        p = self.p
        dms = np.asarray(dms)
        nvar = 5 if p.xctype == "MGGA" else p.ao.shape[0]
        out = np.zeros_like(dms)
        make_a = self._gen_rho_evaluator(mol, dms[0])[0]
        make_b = self._gen_rho_evaluator(mol, dms[1])[0]
        for i in range(dms.shape[1]):
            ra = make_a(i, p.ao if nvar > 1 else p.ao[0], None, p.xctype).reshape(nvar, -1)
            rb = make_b(i, p.ao if nvar > 1 else p.ao[0], None, p.xctype).reshape(nvar, -1)
            rho1 = (ra, rb)
            for t in range(2):
                wv = np.zeros((nvar, p.ng))
                for s in range(2):
                    for c in range(nvar):
                        for d in range(nvar):
                            wv[d] += rho1[s][c] * fxc[s, c, t, d] * p.weights
                if nvar == 1:
                    for g in range(p.ng):
                        out[t, i] += wv[0, g] * np.outer(p.ao[0, g], p.ao[0, g])
                else:
                    wv[0] *= 0.5
                    m = np.zeros((p.nao, p.nao))
                    for g in range(p.ng):
                        aow = sum(wv[d, g] * p.ao[d, g] for d in range(4))
                        m += np.outer(p.ao[0, g], aow)
                    out[t, i] = m + m.T
                    if nvar == 5:             # meta-GGA: wv_tau halved, tau-dot added after the symmetrisation
                        for g in range(p.ng):
                            for k in range(1, 4):
                                out[t, i] += 0.5 * wv[4, g] * np.outer(p.ao[k, g], p.ao[k, g])
        return out


def _dot_ao_ao_sparse(bra, ket, wv, nbins, mask, pair_mask, ao_loc, hermi=0, out=None):
    k = ket if wv is None else ket * wv[:, None]
    r = bra.T @ k
    if out is None:
        return r
    out += r
    return out


def _scale_ao_sparse(ao, wv, mask, ao_loc, out=None):
    if ao.ndim == 2:
        return ao * wv[:, None] if wv.ndim == 1 else ao * wv[0][:, None]
    return sum(ao[c] * wv[c][:, None] for c in range(wv.shape[0]))


def _tau_dot_sparse(bra, ket, wv, nbins, mask, pair_mask, ao_loc, out=None):
    """pyscf.dft.numint._tau_dot_sparse: sum over x, y, z of (d_k bra)^T diag(wv) (d_k ket)."""
    r = sum(bra[k].T @ (ket[k] * wv[:, None]) for k in range(1, 4))
    if out is None:
        return r
    out += r
    return out


def full_eri(cderi):
    return np.einsum("Pij,Pkl->ijkl", cderi, cderi)


class FakeSCFBase:
    """Duck-typed mean-field object over a ProblemData."""
    with_x2c = None
    nlc = ""
    verbose = 0
    stdout = sys.stdout
    converged = True

    def __init__(self, p, form="ks"):
        self.p = p
        self.mol = FakeMol(p)
        self.form = form
        self.xc = "synthetic"
        self._numint = FakeNumInt(p)
        self.grids = FakeGrids(p)
        self.max_memory = 4000
        self.level_shift = p.level_shift
        self._eri = full_eri(p.cderi) if p.cderi is not None else None
        self._eri_lr = full_eri(p.cderi_lr) if p.cderi_lr is not None else None
        if p.restricted:
            self.mo_coeff = p.mo_coeff[0]
            self.mo_energy = p.mo_energy[0]
            occ = np.zeros(p.nmo)
            occ[:p.nc] = 2
            occ[p.nc:p.nc + p.no] = 1
            self.mo_occ = occ
        else:
            self.mo_coeff = p.mo_coeff
            self.mo_energy = p.mo_energy
            occ = np.zeros((2, p.nmo))
            occ[0, :p.nocc_a] = 1
            occ[1, :p.nocc_b] = 1
            self.mo_occ = occ

    def do_nlc(self):
        return False

    def make_rdm1(self, mo_coeff=None, mo_occ=None):
        p = self.p
        da = p.mo_coeff[0][:, :p.nocc_a] @ p.mo_coeff[0][:, :p.nocc_a].T
        db = p.mo_coeff[1][:, :p.nocc_b] @ p.mo_coeff[1][:, :p.nocc_b].T
        return tag(np.stack([da, db]))

    def get_hcore(self, mol=None):
        return np.zeros((self.p.nao, self.p.nao))

    def get_veff(self, mol=None, dm=None, *a, **k):
        p = self.p
        f = p.fock_ks if self.form == "ks" else p.fock_hf
        ca, cb = p.mo_coeff              # orthonormal: C^-T F C^-1 = C F C^T
        return tag(np.stack([ca @ f[0] @ ca.T, cb @ f[1] @ cb.T]))

    def spin_square(self):
        s = self.p.no / 2.0
        return s * (s + 1), 2 * s + 1

    def _eri_for(self, omega):
        if omega is None or omega == 0:
            return self._eri
        return self._eri_lr

    def get_j(self, mol=None, dm=None, hermi=0, omega=None):
        dm = np.asarray(dm)
        return np.einsum("ijkl,...ji->...kl", self._eri_for(omega), dm)

    def get_k(self, mol=None, dm=None, hermi=0, omega=None):
        dm = np.asarray(dm)
        return np.einsum("ijkl,...jk->...il", self._eri_for(omega), dm)

    def get_jk(self, mol=None, dm=None, hermi=0, with_j=True, with_k=True, omega=None):
        return (self.get_j(mol, dm, hermi, omega) if with_j else None,
                self.get_k(mol, dm, hermi, omega) if with_k else None)

    def x2c(self):
        return self


def install_stubs():
    """Install fake `pyscf`, `opt_einsum`, `cupy`, `gpu4pyscf`, `pandas`-free module tree."""
    def mod(name, **attrs):
        m = types.ModuleType(name)
        m.__dict__.update(attrs)
        sys.modules[name] = m
        parent, _, child = name.rpartition(".")
        if parent:
            setattr(sys.modules[parent], child, m)
        return m

    class KohnShamDFT:
        pass

    class SCF:
        pass

    class ROHF(SCF):
        """Marker base class; `ROHF(mol)` itself builds the pure-HF Fock provider (XTDA.py:608, XSF_TDA.py:1108)."""
        def __new__(cls, *args, **kw):
            if cls is ROHF:
                return object.__new__(FakeROHFofKS)
            return object.__new__(cls)

    class UHF(SCF):
        pass

    class FakeROKS(FakeSCFBase, ROHF, KohnShamDFT):
        pass

    class FakeUKS(FakeSCFBase, UHF, KohnShamDFT):
        pass

    class FakeROHFofKS(FakeSCFBase, ROHF):
        """`scf.ROHF(mol)`: pure-HF Fock of the KS density."""
        def __init__(self, mol):
            FakeSCFBase.__init__(self, mol.p, form="hf")
            self.mol = mol

    class TDBase:
        conv_tol = 1e-5
        lindep = 1e-12
        max_cycle = 100
        level_shift = 0
        deg_eia_thresh = 1e-3
        positive_eig_threshold = 1e-3

    class Logger:
        def __init__(self, *a, **k):
            self.verbose = 0

        def __getattr__(self, n):
            return lambda *a, **k: None

    logger = types.ModuleType("pyscf.lib.logger")
    logger.Logger = Logger
    logger.WARN = 2
    logger.DEBUG = 5
    for n in ("warn", "debug", "debug1", "info", "note"):
        setattr(logger, n, lambda *a, **k: None)

    mod("pyscf", __config__=types.SimpleNamespace())
    mod("pyscf.__config__")
    lib = mod("pyscf.lib", einsum=lambda *a, **k: np.einsum(*a, optimize=True),
              current_memory=lambda: (0, 0), num_threads=lambda: 1, logger=logger,
              hermi_sum=lambda a, axes=None: a + a.transpose(axes))
    sys.modules["pyscf.lib.logger"] = logger
    mod("pyscf.lib.misc", StreamObject=types.SimpleNamespace(stdout=sys.stdout))
    mod("pyscf.lib.exceptions", LinearDependencyError=RuntimeError)
    mod("pyscf.lib.linalg_helper", _fill_heff_hermitian=None, make_diag_precond=None, _Xlist=list, _qr=None,
        _sort_by_similarity=None, _sort_elast=None, _outprod_to_subspace=None, _normalize_xt_=None)
    scf = mod("pyscf.scf", ROHF=ROHF)
    hf = mod("pyscf.scf.hf", KohnShamDFT=KohnShamDFT, SCF=SCF)
    mod("pyscf.scf.rohf", ROHF=ROHF)
    mod("pyscf.scf.uhf", UHF=UHF)
    mod("pyscf.gto", mole=types.SimpleNamespace(chiral_mol=lambda m: False))
    mod("pyscf.ao2mo")
    mod("pyscf.tddft")
    mod("pyscf.symm", direct_prod=None)
    mod("pyscf.tdscf")
    mod("pyscf.tdscf.rhf", TDBase=TDBase)
    dft = mod("pyscf.dft")
    mod("pyscf.dft.numint", _dot_ao_ao_sparse=_dot_ao_ao_sparse, _scale_ao_sparse=_scale_ao_sparse,
        _tau_dot_sparse=_tau_dot_sparse, NumInt=lambda: None)
    mod("pyscf.dft.numint2c", NumInt2C=None)
    mod("pyscf.dft.xc_deriv")
    mod("pyscf.dft.gen_grid", NBINS=100)
    mod("opt_einsum", contract=lambda *a, **k: np.einsum(*a, optimize=True))
    mod("pandas")
    # CuPy stand-in: NumPy with the handful of cupy-only names the GPU class touches
    cp = types.ModuleType("cupy")
    for n in dir(np):
        if not n.startswith("__"):
            setattr(cp, n, getattr(np, n))
    cp.cuda = types.SimpleNamespace(Stream=types.SimpleNamespace(null=types.SimpleNamespace(synchronize=lambda: None)))
    sys.modules["cupy"] = cp
    mod("gpu4pyscf")
    mod("gpu4pyscf.dft")
    mod("gpu4pyscf.scf", ROHF=ROHF)
    mod("gpu4pyscf.scf.hf", KohnShamDFT=KohnShamDFT, SCF=SCF)
    mod("gpu4pyscf.scf.rohf", ROHF=ROHF)
    mod("gpu4pyscf.scf.uhf", UHF=UHF)
    mod("gpu4pyscf.tdscf")

    def nr_uks_fxc_sf(ni, mol, grids, xc, dm0, dms, relativity=0, hermi=0, rho0=None, vxc=None, fxc=None, **k):
        """gpu4pyscf.tdscf._uhf_resp_sf.nr_uks_fxc_sf: wv_a = sum_b rho1_b * 2 fxc_ba * w, GGA integration."""
        p = ni.p
        dms = np.asarray(dms)
        out = np.zeros_like(dms)
        make = ni._gen_rho_evaluator(mol, dms)[0]
        nvar = p.ao.shape[0]
        for i in range(dms.shape[0]):
            rho1 = make(i, p.ao if nvar > 1 else p.ao[0], None, p.xctype).reshape(nvar, -1)
            wv = np.zeros((nvar, p.ng))
            for a in range(nvar):
                for b in range(nvar):
                    wv[a] += rho1[b] * 2.0 * fxc[b, a] * p.weights
            if nvar == 1:
                out[i] = (p.ao[0] * wv[0][:, None]).T @ p.ao[0]
            else:
                wv[0] *= 0.5
                m = p.ao[0].T @ sum(p.ao[c] * wv[c][:, None] for c in range(4))
                out[i] = m + m.T
        return out

    mod("gpu4pyscf.tdscf._uhf_resp_sf", nr_uks_fxc_sf=nr_uks_fxc_sf, mcfun_eval_xc_adapter_sf=None)
    mod("gpu4pyscf.tdscf._lr_eig", eigh=None)
    mod("gpu4pyscf.lib")
    mod("gpu4pyscf.lib.cupy_helper", contract=lambda *a, **k: np.einsum(*a, optimize=True),
        tag_array=lambda a, **k: tag(a, **k))
    mod("gpu4pyscf.dft.numint", eval_rho2=None)
    return FakeROKS, FakeUKS


def load_reference_modules():
    """Import the reference package from $XTDDFT_REFERENCE with the Appendix-D source fixes applied in memory."""
    if not (REF and os.path.isdir(os.path.join(REF, "xtddft"))):
        raise SystemExit("set XTDDFT_REFERENCE to a checkout of the original XTDDFT source (the directory holding xtddft/)")
    sys.path.insert(0, REF)
    sys.path.insert(0, os.path.join(REF, "xtddft", "utils"))     # bare `import Davidson`
    sys.path.insert(0, os.path.join(REF, "xtddft"))              # bare `from utils import ...`
    mods = {}
    import xtddft  # noqa: F401  (namespace of the reference)
    from xtddft.utils import utils as ref_utils
    mods["utils"] = ref_utils
    mods["XTDA"] = importlib.import_module("xtddft.XTDA")
    mods["SF_TDA"] = importlib.import_module("xtddft.SF_TDA")
    # SF_TDA.py:142,1029 read a module-level MGGA_DENSITY_LAPL that the file never defines (it is a local of
    # cache_xc_kernel_sf, :42): the meta-GGA branches raise NameError as shipped.  Define it with the value the file uses.
    mods["SF_TDA"].MGGA_DENSITY_LAPL = False
    # XSF_TDA.py does not parse as shipped (full-width comma at line 1137): fix in memory
    path = os.path.join(REF, "xtddft", "XSF_TDA.py")
    src = open(path, encoding="utf-8").read().replace("，", ",")
    m = types.ModuleType("xtddft.XSF_TDA")
    m.__package__ = "xtddft"
    m.__file__ = path
    sys.modules["xtddft.XSF_TDA"] = m
    exec(compile(src, path, "exec"), m.__dict__)
    mods["XSF_TDA"] = m
    mods["XSF_TDA_GPU"] = importlib.import_module("xtddft.XSF_TDA_GPU")
    return mods


# =================================================================================================
# cases
# =================================================================================================
def rand_vectors(seed, x, dim):
    return np.random.default_rng(seed).standard_normal((x, dim))


def main():
    FakeROKS, FakeUKS = install_stubs()
    R = load_reference_modules()
    out = {}

    # ---- pure helpers ------------------------------------------------------------------------
    helpers = {}
    for (nc, no, nv) in [(2, 1, 3), (3, 2, 4), (1, 3, 2), (4, 1, 1)]:
        helpers[f"order_{nc}_{no}_{nv}"] = R["utils"].order_pyscf2my(nc, no, nv)
        dim = (nc + no) * nv + nc * (no + nv)
        v = rand_vectors(7, dim, 3)
        helpers[f"so2st_{nc}_{no}_{nv}"] = R["utils"].so2st(v, nc, no, nv)
        helpers[f"st2so_{nc}_{no}_{nv}"] = R["utils"].st2so(v, nc, no, nv)
    for no in (2, 3, 4):
        dummy = types.SimpleNamespace(no=no)
        helpers[f"vects_{no}"] = R["XSF_TDA"].XSF_TDA.get_vect(dummy)
    np.savez(os.path.join(OUT, "helpers.npz"), **helpers)

    # ---- X-TDA (XTDA.py) ---------------------------------------------------------------------
    xtda_cases = [
        dict(tag="roks_gga_no1", nc=3, no=1, nv=5, naux=11, ng=40, xctype="GGA", hyb=0.2, restricted=True, seed=11),
        dict(tag="roks_gga_no2", nc=2, no=2, nv=5, naux=10, ng=36, xctype="GGA", hyb=0.25, restricted=True, seed=12),
        dict(tag="roks_lda_no3", nc=2, no=3, nv=4, naux=9, ng=30, xctype="LDA", hyb=0.0, restricted=True, seed=13),
        dict(tag="roks_hf_no1", nc=3, no=1, nv=4, naux=9, ng=0, xctype="HF", hyb=1.0, restricted=True, seed=14),
        dict(tag="uks_gga_no1", nc=3, no=1, nv=5, naux=11, ng=40, xctype="GGA", hyb=0.2, restricted=False, seed=15),
        dict(tag="roks_mgga_no2", nc=3, no=2, nv=4, naux=10, ng=36, xctype="MGGA", hyb=0.1, restricted=True, seed=16),
    ]
    for c in xtda_cases:
        p = make_problem(c["nc"] + c["no"] + c["nv"], c["nc"], c["no"], c["nv"], c["naux"], c["ng"], xctype=c["xctype"],
                         hyb=c["hyb"], restricted=c["restricted"], seed=c["seed"])
        mf = (FakeROKS if c["restricted"] else FakeUKS)(p)
        if c["xctype"] == "HF":
            # a plain ROHF object: not a KohnShamDFT instance -> `elif with_j` branch (XTDA.py:546-550)
            mf.__class__ = type("FakeROHF", (FakeSCFBase, sys.modules["pyscf.scf.rohf"].ROHF), {})
        obj = R["XTDA"].XTDA(mf.mol, mf, nstates=3)
        vind, hdiag = obj.gen_vind(mf)
        dim = hdiag.size
        z = rand_vectors(c["seed"] + 100, 3, dim)
        hx = vind(z)
        x0 = obj.get_init_guess(mf, 3)
        np.savez(os.path.join(OUT, f"xtda_{c['tag']}.npz"), z=z, hx=hx, hdiag=hdiag, x0=x0,
                 params=np.array([c["nc"], c["no"], c["nv"], c["naux"], c["ng"], c["seed"], int(c["restricted"])]),
                 xctype=c["xctype"], hyb=c["hyb"])
        print("xtda", c["tag"], dim, float(np.abs(hx).max()))

    # ---- SF-TDA (SF_TDA.py) --------------------------------------------------------------------
    sf_cases = [
        dict(tag="down_gga", isf=-1, nc=3, no=2, nv=4, naux=10, ng=36, xctype="GGA", hyb=0.5, restricted=True, seed=21),
        dict(tag="up_gga", isf=1, nc=3, no=2, nv=4, naux=10, ng=36, xctype="GGA", hyb=0.5, restricted=True, seed=22),
        dict(tag="down_lda", isf=-1, nc=2, no=3, nv=4, naux=9, ng=33, xctype="LDA", hyb=0.3, restricted=True, seed=23),
        dict(tag="down_uks", isf=-1, nc=3, no=2, nv=4, naux=10, ng=36, xctype="GGA", hyb=0.5, restricted=False, seed=24),
        dict(tag="down_mgga", isf=-1, nc=3, no=2, nv=4, naux=10, ng=36, xctype="MGGA", hyb=0.4, restricted=True, seed=26),
    ]
    for c in sf_cases:
        p = make_problem(c["nc"] + c["no"] + c["nv"], c["nc"], c["no"], c["nv"], c["naux"], c["ng"], xctype=c["xctype"],
                         hyb=c["hyb"], restricted=c["restricted"], seed=c["seed"])
        mf = (FakeROKS if c["restricted"] else FakeUKS)(p)
        vind, hdiag = R["SF_TDA"].gen_tda_operation_sf(mf, c["isf"], 0)
        # the ALDA0 kernel the reference built from the stub's ground-state density (an INPUT of the path)
        fxc_alda0 = R["SF_TDA"].cache_xc_kernel_sf(mf, None, None, 1, 2000, isf=-1)
        z = rand_vectors(c["seed"] + 100, 3, hdiag.size)
        hx = vind(z)
        x0 = R["SF_TDA"].init_guess(mf, 3, c["isf"])
        extra = {}
        if c["isf"] == -1:
            v = rand_vectors(5, hdiag.size, 2)
            extra["deal_in"] = v
            extra["deal_out"] = R["SF_TDA"].deal_v_davidson(mf, 2, v)
        np.savez(os.path.join(OUT, f"sf_{c['tag']}.npz"), z=z, hx=hx, hdiag=hdiag, x0=x0, fxc_alda0=fxc_alda0,
                 params=np.array([c["nc"], c["no"], c["nv"], c["naux"], c["ng"], c["seed"], int(c["restricted"]), c["isf"]]),
                 xctype=c["xctype"], hyb=c["hyb"], **extra)
        print("sf", c["tag"], hdiag.size, float(np.abs(hx).max()))

    # multicollinear contraction (SF_TDA.py:976-1047) with a given kernel
    p = make_problem(9, 3, 2, 4, 10, 36, xctype="GGA", hyb=0.5, seed=25)
    mf = FakeROKS(p)
    co, cv = p.mo_coeff[0][:, :p.nocc_a], p.mo_coeff[1][:, p.nocc_b:]
    z = rand_vectors(125, 2, p.nocc_a * p.nvir_b).reshape(2, p.nocc_a, p.nvir_b)
    dms = np.einsum("xov,qv,po->xpq", z, cv, co)
    v_mc = R["SF_TDA"].nr_uks_fxc_sf_tda_mc(mf._numint, mf.mol, mf.grids, mf.xc, None, dms, 0, 0, None, None, p.fxc_mcol)
    np.savez(os.path.join(OUT, "sf_mcol_contraction.npz"), dms=dms, v=v_mc, params=np.array([3, 2, 4, 10, 36, 25]))
    # ... and its meta-GGA branch (tau component of the kernel, SF_TDA.py:1028-1040)
    p = make_problem(9, 3, 2, 4, 10, 36, xctype="MGGA", hyb=0.5, seed=27)
    mf = FakeROKS(p)
    co, cv = p.mo_coeff[0][:, :p.nocc_a], p.mo_coeff[1][:, p.nocc_b:]
    z = rand_vectors(127, 2, p.nocc_a * p.nvir_b).reshape(2, p.nocc_a, p.nvir_b)
    dms = np.einsum("xov,qv,po->xpq", z, cv, co)
    v_mc = R["SF_TDA"].nr_uks_fxc_sf_tda_mc(mf._numint, mf.mol, mf.grids, mf.xc, None, dms, 0, 0, None, None, p.fxc_mcol)
    np.savez(os.path.join(OUT, "sf_mcol_contraction_mgga.npz"), dms=dms, v=v_mc, params=np.array([3, 2, 4, 10, 36, 27]))

    # ---- XSF-TDA (XSF_TDA.py, block layout) ----------------------------------------------------------
    for (tagname, nc, no, nv, xct, seed) in [("gga_no2", 3, 2, 4, "GGA", 31), ("lda_no3", 2, 3, 3, "LDA", 32)]:
        p = make_problem(nc + no + nv, nc, no, nv, 10, 36, xctype=xct, hyb=0.5, seed=seed)
        mf = FakeROKS(p)
        fxc_alda0 = R["SF_TDA"].cache_xc_kernel_sf(mf, None, None, 1, 2000, isf=-1)
        res = dict(fxc_alda0=fxc_alda0, params=np.array([nc, no, nv, 10, 36, seed]), xctype=xct, hyb=0.5)
        for sa in (0, 1, 2, 3):
            for re in (False, True):
                obj = R["XSF_TDA"].XSF_TDA(mf, SA=sa, davidson=True, method=0)
                obj.re = re
                obj.nstates = 3
                obj.vects = obj.get_vect()
                vind, hdiag = obj.gen_tda_operation_sf(0.8, 0.7)
                z = rand_vectors(seed + 100 + sa, 2, hdiag.size)
                res[f"z_sa{sa}_re{int(re)}"] = z
                res[f"hx_sa{sa}_re{int(re)}"] = vind(z)
                res[f"hdiag_sa{sa}_re{int(re)}"] = hdiag
        # default fglobal rule (XSF_TDA.py:1511-1518) and init guess
        obj = R["XSF_TDA"].XSF_TDA(mf, SA=3)
        res["x0"] = obj._build_initial_guess_from_gaps(res["hdiag_sa3_re1"], 3)
        np.savez(os.path.join(OUT, f"xsf_{tagname}.npz"), **res)
        print("xsf", tagname, float(np.abs(res["hx_sa3_re1"]).max()))

    # ---- XSF-TDA GPU class (PySCF order; NumPy stands in for CuPy) -----------------------------
    cp = sys.modules["cupy"]
    for (tagname, nc, no, nv, xct, seed) in [("gga_no2", 3, 2, 4, "GGA", 41), ("gga_no3", 2, 3, 3, "GGA", 42)]:
        p = make_problem(nc + no + nv, nc, no, nv, 10, 36, xctype=xct, hyb=0.5, seed=seed)
        mf = FakeROKS(p)
        G = R["XSF_TDA_GPU"]
        # the class computes its own kernel through gpu4pyscf+mcfun; feed the synthetic mcol-form kernel instead
        G.cache_xc_kernel_sf = lambda *a, **k: (None, None, p.fxc_mcol)
        res = dict(params=np.array([nc, no, nv, 10, 36, seed]), xctype=xct, hyb=0.5)
        for X in (0, 1, 2, 3):
            for re in (False, True):
                obj = G.XSF_TDA_GPU(mf, X=X, collinear="mcol", nstates=3, extype=1, remove=re, foo=0.8, d_lda=0.3)
                obj.fglobal = 0.7
                vind, hdiag = obj.gen_vind()
                z = rand_vectors(seed + 100 + X, 2, hdiag.size)
                res[f"z_X{X}_re{int(re)}"] = z
                res[f"hx_X{X}_re{int(re)}"] = np.asarray(vind(z))
                res[f"hdiag_X{X}_re{int(re)}"] = np.asarray(hdiag)
        obj = G.XSF_TDA_GPU(mf, X=0, collinear="mcol", nstates=3, extype=0, remove=False)
        obj.fglobal = 0.7
        vind, hdiag = obj.gen_vind()
        z = rand_vectors(seed + 200, 2, hdiag.size)
        res["z_up"], res["hx_up"], res["hdiag_up"] = z, np.asarray(vind(z)), np.asarray(hdiag)
        np.savez(os.path.join(OUT, f"xsfgpu_{tagname}.npz"), **res)
        print("xsfgpu", tagname, float(np.abs(res["hx_X3_re1"]).max()))


if __name__ == "__main__":
    main()
