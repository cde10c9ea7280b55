#!/usr/bin/env python
"""Golden vectors for the post-Davidson property pass (SURVEY 8f row f1), produced by executing the REFERENCE's own
methods from $XTDDFT_REFERENCE (see make_golden.py) on seeded synthetic states and one-electron integrals:

  xtddft/XTDA.py          XTDA.osc_str, XTDA.rot_str, XTDA.deltaS2                (ground -> excited moments)
  xtddft/XSF_TDA_GPU.py   XSF_TDA_GPU.calculate_TDM_R / calculate_TDM_U           (state-to-state oscillator matrix;
                          NumPy stands in for CuPy)
  xtddft/XSF_TDA.py       XSF_TDA.deltaS2_U, XSF_TDA.analyse (D<S^2> labels)

The third-party pieces (`mol.intor*`, `mf.get_ovlp`) are replaced by seeded arrays: they are inputs of this pass.
Usage:  python tests/golden/make_golden_properties.py      -> tests/golden/properties.npz
"""
import contextlib
import io
import os
import sys
import types

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.environ.get("XTD_GOLDEN_OUT", HERE)      # tests regenerate into a temporary directory and diff
sys.path.insert(0, HERE)
import make_golden as mg  # noqa: E402

from xtddft_b200.synth import make_problem  # noqa: E402


def one_electron(n, seed):
    r = np.random.default_rng(seed)
    dip = r.standard_normal((3, n, n))
    dip = dip + dip.transpose(0, 2, 1)                      # int1e_r: symmetric
    ipo = r.standard_normal((3, n, n))
    ipo = ipo - ipo.transpose(0, 2, 1)                      # int1e_ipovlp, hermi=2: anti-symmetric
    rxp = r.standard_normal((3, n, n))
    rxp = rxp - rxp.transpose(0, 2, 1)                      # int1e_cg_irxp, hermi=2
    a = r.standard_normal((n, n))
    ovlp = a @ a.T / n + np.eye(n)                          # a symmetric positive "overlap"
    return dip, ipo, rxp, ovlp


class Mol:
    groupname = "C1"

    def __init__(self, p, dip, ipo, rxp):
        self.p, self.spin = p, p.no
        self._ints = {"int1e_r": dip, "int1e_ipovlp": ipo, "int1e_cg_irxp": rxp}

    def intor_symmetric(self, name, comp=3):
        return self._ints[name]

    def intor(self, name, comp=3, hermi=0):
        return self._ints[name]


def orthonormal_states(dim, ns, seed):
    q, _ = np.linalg.qr(np.random.default_rng(seed).standard_normal((dim, ns)))
    return q


def main():
    FakeROKS, FakeUKS = mg.install_stubs()
    R = mg.load_reference_modules()
    out = {}

    # ---- X-TDA: osc_str / rot_str / deltaS2 --------------------------------------------------------------
    for tag, (nc, no, nv, seed) in {"xtda_a": (3, 1, 5, 51), "xtda_b": (2, 2, 4, 52)}.items():
        p = make_problem(nc + no + nv, nc, no, nv, 6, 0, xctype="HF", hyb=1.0, restricted=True, seed=seed)
        dip, ipo, rxp, _ = one_electron(p.nao, seed + 1)
        na, nb, nva = nc + no, nc, nv
        dim = na * nva + nb * (no + nv)
        ns = 4
        x1 = orthonormal_states(dim, ns, seed + 2).T                  # [ns, dim] PySCF order, as davidson returns
        e = np.sort(np.random.default_rng(seed + 3).uniform(0.1, 0.6, ns))
        util = R["utils"]
        s = types.SimpleNamespace()
        s.mf = types.SimpleNamespace(mo_coeff=p.mo_coeff[0])
        s.mol = Mol(p, dip, ipo, rxp)
        s.e, s.nstates = e, ns
        s.nc, s.no, s.nv = nc, no, nv
        s.order = util.order_pyscf2my(nc, no, nv)
        s.v = x1.T[s.order, :]                                        # XTDA.py:799-805
        s.xy_a, s.xy_b = s.v.T[:, :na * nva], s.v.T[:, na * nva:]
        s.xycv_a = s.v.T[:, :nb * nva]
        s.xycv_b = s.v.T[:, na * nva + nb * no:]
        occ = np.array([2] * nc + [1] * no + [0] * nv)
        s.occidx_a, s.viridx_a = np.where(occ >= 1)[0], np.where(occ == 0)[0]
        s.occidx_b, s.viridx_b = np.where(occ >= 2)[0], np.where(occ != 2)[0]
        X = R["XTDA"].XTDA
        out[f"{tag}_params"] = np.array([nc, no, nv, seed])
        out[f"{tag}_x1"], out[f"{tag}_e"] = x1, e
        out[f"{tag}_os"] = X.osc_str(s)
        out[f"{tag}_rs"] = X.rot_str(s)
        out[f"{tag}_dS2"] = X.deltaS2(s)
        print(tag, out[f"{tag}_os"], out[f"{tag}_rs"])

    # ---- spin-flip states: oscillator matrix on ROKS (all SA levels, with/without the removed OO vector) ------
    G = R["XSF_TDA_GPU"].XSF_TDA_GPU
    XS = R["XSF_TDA"].XSF_TDA
    for tag, (nc, no, nv, seed) in {"sf_a": (3, 2, 4, 61), "sf_b": (2, 3, 3, 62)}.items():
        p = make_problem(nc + no + nv, nc, no, nv, 6, 0, xctype="HF", hyb=1.0, restricted=True, seed=seed)
        dip, _, _, _ = one_electron(p.nao, seed + 1)
        ns = 4
        dimf = (nc + no) * (no + nv)
        e = np.sort(np.random.default_rng(seed + 3).uniform(0.05, 0.5, ns))
        out[f"{tag}_params"] = np.array([nc, no, nv, seed])
        out[f"{tag}_e"] = e
        vects = XS.get_vect(types.SimpleNamespace(no=no))
        for re in (0, 1):
            v = orthonormal_states(dimf - re, ns, seed + 4 + re)
            out[f"{tag}_v_re{re}"] = v
            for X in (0, 1, 3):
                s = types.SimpleNamespace(nstates=ns, nc=nc, no=no, nv=nv, e=e, v=v, re=bool(re), vects=vects, X=X,
                                          mol=Mol(p, dip, None, None), mf=types.SimpleNamespace(mo_coeff=p.mo_coeff[0]))
                out[f"{tag}_osc_X{X}_re{re}"] = np.asarray(G.calculate_TDM_R(s))
            # D<S^2> labels printed by analyse() for SA=0 on ROKS (XSF_TDA.py:771-779)
            s = types.SimpleNamespace(nstates=ns, nc=nc, no=no, nv=nv, e=e, v=v, re=bool(re), vects=vects, SA=0, type_u=False,
                                      ground_s=no / 2.0, mol=Mol(p, dip, None, None),
                                      mf=types.SimpleNamespace(e_tot=-1.0, get_wfnsym=lambda: (_ for _ in ()).throw(RuntimeError())))
            with contextlib.redirect_stdout(io.StringIO()):
                ds, _ = XS.analyse(s)
            out[f"{tag}_ds2_re{re}"] = np.asarray(ds)
        print(tag, out[f"{tag}_osc_X3_re1"][0], out[f"{tag}_ds2_re0"])

    # ---- spin-flip states on a UKS reference: oscillator matrix and D<S^2> ---------------------------------
    for tag, (nc, no, nv, seed) in {"usf_a": (3, 2, 4, 71)}.items():
        p = make_problem(nc + no + nv, nc, no, nv, 6, 0, xctype="HF", hyb=1.0, restricted=False, seed=seed)
        dip, _, _, ovlp = one_electron(p.nao, seed + 1)
        ns = 4
        v = orthonormal_states((nc + no) * (no + nv), ns, seed + 4)
        e = np.sort(np.random.default_rng(seed + 3).uniform(0.05, 0.5, ns))
        mo = np.asarray(p.mo_coeff)
        occ = np.zeros((2, p.nmo))
        occ[0, :nc + no] = 1
        occ[1, :nc] = 1
        mf = types.SimpleNamespace(mo_coeff=mo, mo_occ=occ, get_ovlp=lambda: ovlp)
        s = types.SimpleNamespace(nstates=ns, nc=nc, no=no, nv=nv, e=e, v=v, mol=Mol(p, dip, None, None), mf=mf)
        out[f"{tag}_params"] = np.array([nc, no, nv, seed])
        out[f"{tag}_e"], out[f"{tag}_v"] = e, v
        out[f"{tag}_osc"] = np.asarray(G.calculate_TDM_U(s))
        out[f"{tag}_pab"] = np.array([float(XS.deltaS2_U(s, k)) for k in range(ns)])
        print(tag, out[f"{tag}_osc"][0], out[f"{tag}_pab"])

    np.savez(os.path.join(OUT, "properties.npz"), **out)

    # ---- state-interaction wire format (SURVEY 8f row f4): the reference's own statements, x2c_hamiltonian/test_SOCSI.py:47-58,
    #      read from the reference tree and executed verbatim on a stand-in `xsf_tda` object --------------------------------
    src = open(os.path.join(mg.REF, "x2c_hamiltonian", "test_SOCSI.py")).read().splitlines()
    i0 = next(i for i, l in enumerate(src) if "trans the formulation of X vector" in l)
    i1 = next(i for i, l in enumerate(src) if l.strip().startswith("xm[dim+xsf_tda.no**2:,:]"))
    block = "\n".join(l[4:] for l in src[i0:i1 + 1])                      # de-indent the body of soc_mf()
    sd = {}
    for (nc, no, nv, seed) in [(3, 2, 4, 81), (2, 3, 3, 82)]:
        ns = 5
        vects = R["XSF_TDA"].XSF_TDA.get_vect(types.SimpleNamespace(no=no))
        dim_re = (nc + no) * (no + nv) - 1
        xm_ = np.random.default_rng(seed).standard_normal((dim_re, ns))
        ns_ = dict(numpy=np, xm_=xm_, xsf_tda=types.SimpleNamespace(nc=nc, no=no, nv=nv, nstates=ns, vects=vects))
        exec(block, ns_)
        sd[f"in_{nc}_{no}_{nv}"] = xm_
        sd[f"out_{nc}_{no}_{nv}"] = ns_["xm"]
    np.savez(os.path.join(OUT, "state_dict.npz"), **sd)
    print("state_dict", {k: v.shape for k, v in sd.items()})


if __name__ == "__main__":
    main()
