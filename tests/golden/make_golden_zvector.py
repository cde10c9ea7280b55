#!/usr/bin/env python
"""Golden vectors for the Z-vector equation of the spin-flip-up TDA gradients (SURVEY 8f row f3), produced by executing the
REFERENCE's own `grad_elec` functions from $XTDDFT_REFERENCE (see make_golden.py) on seeded synthetic inputs:

  xtddft/grad_hb/tdroks_sfu.py   grad_elec: internal variables, `_contract_xc_kernel` (collinear kernel), the Q matrix / right-hand
                                 side `w` (:207-274), the ROHF orbital-Hessian closure `matvec` (:284-321)
  xtddft/grad_hb/tduks_sfu.py    grad_elec: right-hand side (wvoa, wvob) (:205-244), the closure `fvind` (:249-258)

Both functions are run verbatim.  Their solver call (`lib.solve` / `ucphf.solve`) is a stub that records the closure and the right-hand side
it was handed and returns the unique solution of the equation (dense LAPACK solve of that closure); grad_elec then builds its W matrix
`im0` from it with its own code (tdroks_sfu.py:335-356, tduks_sfu.py:266-299) and is stopped at `nuc_grad_method()` -- the integral
derivatives that follow need libcint and are out of scope.  The fixture holds: seeded vectors and the closure's images (x, ax), the
right-hand side (rhs), the solution (z) and the W matrix (im0).

What is NOT in the reference tree and is supplied by stubs coded from the published definitions (as in make_golden.py):
`mf.gen_response(hermi=1)` (pyscf `_gen_uhf_response`: nr_uks_fxc + J - hyb K), `ni.eval_rho`, `ni.eval_xc_eff` (returns the
synthetic f_xc table of the problem: an input of the path), `pyscf.grad.tdrks._lda_eval_mat_ / _gga_eval_mat_` (value part only).

Usage:  python tests/golden/make_golden_zvector.py      -> tests/golden/zvector_*.npz
"""
import importlib.util
import os
import sys
import types

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.environ.get("XTD_GOLDEN_OUT", HERE)
sys.path.insert(0, HERE)
import make_golden as mg  # noqa: E402

from xtddft_b200.synth import make_problem  # noqa: E402


class Captured(Exception):
    pass


class Capture:
    """Stands in for `lib.solve` / `ucphf.solve`: keeps the operator closure and the right-hand side and returns the (unique) solution
    of the equation the real solver iterates on, from a dense LAPACK solve of the closure it was handed.  grad_elec then continues
    with its own code (W matrix) until `nuc_grad_method()`, where the stub stops it; the locals of its frame are read from the traceback."""
    def __init__(self):
        self.op = self.rhs = None

    def lib_solve(self, aop, b, *a, **k):
        self.op, self.rhs = aop, np.array(b)
        dense = np.stack([aop(e) for e in np.eye(b.size)], axis=1)
        return np.linalg.solve(dense, b)

    def ucphf_solve(self, fvind, mo_energy, mo_occ, h1, *a, **k):
        """pyscf.scf.ucphf.solve (solve_nos1): (e_a - e_i) z + fvind(z) = -h1; returns ((z_a [nvir_a, nocc_a], z_b), None)."""
        self.op, self.rhs = fvind, [np.array(h1[0]), np.array(h1[1])]
        h = np.hstack([h1[0].ravel(), h1[1].ravel()])
        gaps = np.hstack([(mo_energy[s][mo_occ[s] == 0][:, None] - mo_energy[s][mo_occ[s] > 0][None, :]).ravel() for s in (0, 1)])
        dense = np.stack([fvind(e[None]) for e in np.eye(h.size)], axis=1) + np.diag(gaps)
        z = np.linalg.solve(dense, -h)
        n0 = h1[0].size
        return (z[:n0].reshape(h1[0].shape), z[n0:].reshape(h1[1].shape)), None


CAP = Capture()


def _lda_eval_mat_(mol, vmat, ao, wv, mask, shls_slice, ao_loc):
    """pyscf.grad.tdrks._lda_eval_mat_, value part: vmat[0] += ao_0^T diag(wv_0) ao_0 (vmat[1:] are nuclear-derivative pieces)."""
    a0 = ao[0]
    vmat[0] += a0.T @ (a0 * wv[0][:, None])
    return vmat


def _gga_eval_mat_(mol, vmat, ao, wv, mask, shls_slice, ao_loc):
    """pyscf.grad.tdrks._gga_eval_mat_, value part: wv_0 halved, aow = sum_c ao_c wv_c, vmat[0] += ao_0^T aow + transpose."""
    w = np.array(wv[:4])
    w[0] *= 0.5
    aow = sum(ao[c] * w[c][:, None] for c in range(4))
    tmp = ao[0].T @ aow
    vmat[0] += tmp + tmp.T
    return vmat


def install_grad_stubs():
    FakeROKS, FakeUKS = mg.install_stubs()

    def mod(name, **attrs):
        m = types.ModuleType(name)
        m.__dict__.update(attrs)
        sys.modules[name] = m
        parent, _, child = name.rpartition(".")
        if parent:
            setattr(sys.modules[parent], child, m)
        return m

    class Gradients:
        pass

    log = types.SimpleNamespace(timer=lambda *a, **k: (0.0, 0.0), warn=lambda *a, **k: None)
    logger = sys.modules["pyscf.lib.logger"]
    logger.INFO = 4
    logger.new_logger = lambda *a, **k: log
    logger.process_clock = lambda: 0.0
    logger.perf_counter = lambda: 0.0
    sys.modules["pyscf.lib"].solve = CAP.lib_solve
    mod("pyscf.scf.ucphf", solve=CAP.ucphf_solve)
    mod("pyscf.grad")
    mod("pyscf.grad.rohf", Gradients=Gradients)
    mod("pyscf.grad.uhf", Gradients=Gradients)
    mod("pyscf.grad.tdrks", _lda_eval_mat_=_lda_eval_mat_, _gga_eval_mat_=_gga_eval_mat_, _mgga_eval_mat_=None)
    mod("pyscf.grad.tduks")
    mod("pyscf.sftda")
    mod("pyscf.sftda.numint2c_sftd", mcfun_eval_xc_adapter_sf=None)
    return FakeROKS, FakeUKS


class GradNumInt(mg.FakeNumInt):
    """FakeNumInt + the calls `_contract_xc_kernel` makes; `eval_xc_eff` hands back the problem's cached f_xc table for the block
    `block_loop` is on (the kernel is an input of the path, SURVEY row a3)."""
    def block_loop(self, mol, grids, nao=None, deriv=0, max_memory=2000, **kw):
        p = self.p
        edges = np.linspace(0, p.ng, self.blocks + 1).astype(int)
        for b0, b1 in zip(edges[:-1], edges[1:]):
            self._blk = (b0, b1)
            yield p.ao[:, b0:b1], None, p.weights[b0:b1], None

    def eval_rho(self, mol, ao, dm, mask=None, xctype="LDA", hermi=0, with_lapl=False, verbose=None):
        return self._gen_rho_evaluator(mol, dm)[0](0, ao, mask, xctype)

    def eval_xc_eff(self, xc, rho, deriv=1, omega=None, xctype=None, spin=0, **kw):
        b0, b1 = self._blk
        nvar = self.p.ao.shape[0]
        return None, np.zeros((2, nvar, b1 - b0)), self.p.fxc_uks[..., b0:b1], None


def gen_response(self, mo_coeff=None, mo_occ=None, hermi=0, **kw):
    """pyscf.scf._response_functions._gen_uhf_response (hybrid / pure / HF): v1 = f_xc[dm1] + J[dm1_a + dm1_b] - hyb K[dm1_s]."""
    p = self.p

    def vind(dm1):
        dm1 = np.asarray(dm1)
        if p.xctype != "HF":
            v1 = self._numint.nr_uks_fxc(self.mol, self.grids, self.xc, None, dm1[:, None], 0, hermi, None, None, p.fxc_uks)[:, 0]
        else:
            v1 = np.zeros_like(dm1)
        vj = self.get_j(self.mol, dm1, hermi=hermi)
        v1 = v1 + (vj[0] + vj[1])[None]
        if p.hyb != 0.0:
            v1 = v1 - p.hyb * self.get_k(self.mol, dm1, hermi=hermi)
        return v1
    return vind


def load_grad_module(name):
    """grad_hb is not a package: load the file by path (its bare `from SF_TDA import ...`, `from utils import ...` resolve through
    the sys.path entries make_golden.load_reference_modules adds)."""
    omp = os.environ.get("OMP_NUM_THREADS")
    path = os.path.join(mg.REF, "xtddft", "grad_hb", name + ".py")
    spec = importlib.util.spec_from_file_location("ref_" + name, path)
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    if omp is None:                      # the module sets OMP_NUM_THREADS=4 at import
        os.environ.pop("OMP_NUM_THREADS", None)
    else:
        os.environ["OMP_NUM_THREADS"] = omp
    return m


CASES = [
    dict(tag="roks_gga_no2", nc=3, no=2, nv=4, naux=10, ng=36, xctype="GGA", hyb=0.25, restricted=True, seed=71),
    dict(tag="roks_lda_no3", nc=2, no=3, nv=4, naux=9, ng=30, xctype="LDA", hyb=0.3, restricted=True, seed=72),
    dict(tag="roks_hf_no2", nc=3, no=2, nv=3, naux=9, ng=0, xctype="HF", hyb=1.0, restricted=True, seed=73),
    dict(tag="uks_gga_no2", nc=3, no=2, nv=4, naux=10, ng=36, xctype="GGA", hyb=0.2, restricted=False, seed=74),
    dict(tag="uks_lda_pure_no2", nc=2, no=2, nv=4, naux=9, ng=30, xctype="LDA", hyb=0.0, restricted=False, seed=75),
]


def main():
    FakeROKS, FakeUKS = install_grad_stubs()
    mg.load_reference_modules()
    roks = load_grad_module("tdroks_sfu")
    uks = load_grad_module("tduks_sfu")
    for c in CASES:
        p = make_problem(c["nc"] + c["no"] + c["nv"], c["nc"], c["no"], c["nv"], c["naux"], c["ng"], xctype=c["xctype"],
                         hyb=c["hyb"], restricted=c["restricted"], seed=c["seed"])
        mf = (FakeROKS if c["restricted"] else FakeUKS)(p)
        mf._numint = GradNumInt(p)
        mf.mol.nbas = p.nao
        mf.gen_response = types.MethodType(gen_response, mf)

        def stop(*a, **k):
            raise Captured()
        mf.nuc_grad_method = stop
        nc, no, nv = p.nc, p.no, p.nv
        occ = np.zeros((2, p.nmo))
        occ[0, :nc + no] = 1
        occ[1, :nc] = 1
        # the solved SF-TDA object (`td.base`): pseudo-UKS arrays the SF_TDA_up solver stores (tdroks_sfu.py:190-194)
        base = types.SimpleNamespace(_scf=mf, mo_coeff=p.mo_coeff, mo_occ=occ, mo_energy=p.mo_energy, collinear_samples=-1)
        amp = np.random.default_rng(c["seed"] + 200).standard_normal((nc * nv, 2))
        amp /= np.linalg.norm(amp, axis=0)
        td = types.SimpleNamespace(base=base, mol=mf.mol, v=amp, state=1, cphf_max_cycle=40, cphf_conv_tol=1e-8, dsolve_lindep=1e-13,
                                   verbose=0, stdout=sys.stdout)
        try:
            (roks if c["restricted"] else uks).grad_elec(td)
            raise RuntimeError("the stop stub was not reached")
        except Captured as e:
            tb = e.__traceback__
            frame = None
            while tb is not None:                      # the frame of grad_elec holds the solution and the W matrix it built from it
                if tb.tb_frame.f_code.co_name == "grad_elec":
                    frame = tb.tb_frame
                tb = tb.tb_next
            loc = frame.f_locals
        dim = nv * nc + nv * no + no * nc if c["restricted"] else nv * (nc + no) + (no + nv) * nc
        x = np.random.default_rng(c["seed"] + 100).standard_normal((3, dim))
        if c["restricted"]:
            ax = np.stack([CAP.op(xi) for xi in x])
            rhs = CAP.rhs
        else:
            ax = np.stack([CAP.op(xi[None]) for xi in x])
            rhs = np.hstack([CAP.rhs[0].ravel(), CAP.rhs[1].ravel()])
        if c["restricted"]:
            zsol = np.array(loc["z"])
        else:
            zsol = np.hstack([np.array(loc["z1a"]).ravel(), np.array(loc["z1b"]).ravel()])
        np.savez(os.path.join(OUT, f"zvector_{c['tag']}.npz"), x=x, ax=ax, rhs=rhs, amp=amp[:, 0], z=zsol, im0=np.array(loc["im0"]),
                 params=np.array([nc, no, nv, c["naux"], c["ng"], c["seed"], int(c["restricted"])]), xctype=c["xctype"], hyb=c["hyb"])
        print("zvector", c["tag"], dim, float(np.abs(ax).max()), float(np.abs(rhs).max()))


if __name__ == "__main__":
    main()
