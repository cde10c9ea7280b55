"""Z-vector (coupled-perturbed) equation of the spin-flip-up TDA nuclear gradients on the B200 sigma engine (SURVEY 8f row f3).

The reference solves, for every state whose gradient is wanted,

  * ROKS reference:  matvec(z) = w            xtddft/grad_hb/tdroks_sfu.py:284-327  (`lib.solve(matvec, w, tol=1e-12, ...)`)
  * UKS reference:   (e_a - e_i) z + fvind(z) = -(wvoa, wvob)     xtddft/grad_hb/tduks_sfu.py:249-263  (`ucphf.solve(fvind, ...)`)

where `matvec` / `fvind` apply the hermi = 1 response `vresp` (grid f_xc + J - hyb K of the symmetrised rotation density) -- one AO
J/K build and one grid pass per iteration.  Here the operator is an engine plan (`plan.build_zvector_plan`): the MO-resident exchange
and Coulomb blocks, the MO-on-grid kernel contraction and the ROHF Fock couplings of the sigma path, plus the exchange of the
transposed density (`xtd_add_kterm_t`); the Krylov vectors live in HBM and the subspace algebra runs in the `xtd_vec_*` kernels.

The collinear right-hand side (the Q matrix: J/K and f_xc images of occupied-occupied and virtual-virtual densities) and the W matrix
come from `xtd_block_response` on the same engine (`ZVector.rhs`, `ZVector.w_matrix`).  The third-derivative kernel of multicollinear
functionals and the integral derivatives that follow the solve need pieces outside the sigma path (libxc third derivatives, libcint
derivative integrals).
"""
from __future__ import annotations

from typing import Optional

import numpy as np

from . import plan as planmod
from .adapters import problem_from_mf


def solve_linear(aop, b, hdiag, *, tol: float = 1e-12, max_cycle: int = 40, lindep: float = 1e-13, backend=None, verbose: int = 0):
    """Solve A x = b for a general (not necessarily symmetric) operator by Galerkin projection on a preconditioned Krylov space --
    the scheme of `pyscf.lib.linalg_helper.dsolve` that `lib.solve` names (tdroks_sfu.py:324): new direction = diagonally
    preconditioned residual, projected system solved on the host (<= max_cycle unknowns).  Differences: the directions are kept
    orthonormal (two Gram-Schmidt passes on the device), and vectors never leave the device.

    aop(X[k, dim]) -> [k, dim] on the backend's vectors; b, hdiag: host arrays.  Returns (x_host, converged, cycles, residual norm).
    """
    b = np.asarray(b, dtype=np.float64).ravel()
    dim = b.size
    vb = backend
    if vb is None:
        from .davidson import CudaVectors
        vb = CudaVectors(dim)
    m = min(max_cycle, dim)
    V, AV = vb.alloc(m), vb.alloc(m)
    bd = vb.from_host(b[None])
    hd = vb.from_host(np.asarray(hdiag, dtype=np.float64).ravel())
    t, r = vb.alloc(1), vb.alloc(1)
    zero = np.zeros(1)
    vb.copy(t, bd)
    H = np.zeros((m, m))
    g = np.zeros(m)
    c = np.zeros(0)
    res = float(np.linalg.norm(b))
    conv = res < tol
    k = 0
    while not conv and k < m:
        n0 = float(vb.precond(t, hd, zero)[0])                      # t <- t / hdiag   (|hdiag| clamped at 1e-8)
        if n0 <= 0.0:
            break
        vb.scale(t, np.array([1.0 / np.sqrt(n0)]))                  # unit length, so `lindep` is a relative threshold
        for _ in range(2):                                          # CGS2 against the kept directions
            if k:
                vb.lincomb(t, V[:k], -vb.dots(t, V[:k]), 1.0)
        nrm2 = float(vb.dots(t, t)[0, 0])
        if nrm2 <= lindep:
            break
        vb.scale(t, np.array([1.0 / np.sqrt(nrm2)]))
        vb.copy(V[k:k + 1], t)
        vb.copy(AV[k:k + 1], aop(V[k:k + 1]))
        k += 1
        H[:k, k - 1] = vb.dots(V[:k], AV[k - 1:k])[:, 0]
        H[k - 1, :k] = vb.dots(V[k - 1:k], AV[:k])[0]
        g[k - 1] = vb.dots(V[k - 1:k], bd)[0, 0]
        c = np.linalg.solve(H[:k, :k], g[:k])
        vb.lincomb(r, AV[:k], c[None], 0.0)
        vb.lincomb(r, bd, -np.ones((1, 1)), 1.0)                    # r = A x - b
        res = float(np.sqrt(vb.dots(r, r)[0, 0]))
        if verbose:
            print(f"zvector solve: cycle {k}  |r| = {res:.3e}")
        conv = res < tol
        vb.copy(t, r)
    x = vb.alloc(1)
    if k:
        vb.lincomb(x, V[:k], c[None], 0.0)
    return vb.to_host(x)[0], bool(conv), k, res


def rhs_intermediates(p, v, apply_response, apply_sf_exchange) -> dict:
    """The contractions behind the right-hand side and the W matrix of one state (collinear kernel: f1vo = k1ao = 0), as two engine
    plans on MO-basis matrices:

      apply_response(t[2, nmo, nmo]) -> C_s^T (f_xc[T] + J[T_a + T_b] - hyb K[T_s]) C_s      (plan.build_mo_response_plan)
      apply_sf_exchange(x[nmo, nmo]) -> C_b^T K[C_b x C_a^T] C_a                              (plan.build_mo_sf_exchange_plan)

    applied to the relaxed difference densities T_vv = v^T v (alpha), T_oo = -v v^T (beta) and to the transition density X = v
    (grad_hb/tdroks_sfu.py:207-214,241-254; tduks_sfu.py:205-212,219-232)."""
    nc, no, nv, nmo = p.nc, p.no, p.nv, p.nmo
    na, nb = nc + no, nc
    v = np.asarray(v, dtype=np.float64).reshape(nc, nv)
    dvva = v.T @ v                                   # T_ab
    doob = -(v @ v.T)                                # T_ij
    t = np.zeros((2, nmo, nmo))
    t[0, na:, na:] = dvva
    t[1, :nb, :nb] = doob
    g = np.asarray(apply_response(t)).reshape(2, nmo, nmo).copy()   # veff0doo in the MO basis
    veff0mo = np.zeros((nmo, nmo))
    if p.hyb != 0.0:
        x = np.zeros((nmo, nmo))
        x[:nb, na:] = v                              # X: beta occupied -> alpha virtual
        veff0mo = -p.hyb * np.asarray(apply_sf_exchange(x)).reshape(nmo, nmo)
    return dict(v=v, dvva=dvva, doob=doob, g=g, veff0mo=veff0mo)


def assemble_rhs(p, v, apply_response, apply_sf_exchange, inter: Optional[dict] = None):
    """Right-hand side of the Z-vector equation for the spin-flip-up TDA state with amplitudes v[nc, nv] -- grad_hb/tdroks_sfu.py:246-274
    (ROKS: `w`), grad_hb/tduks_sfu.py:223-234 (UKS: `(wvoa, wvob)`, returned stacked): the block bookkeeping of the reference (a few small
    einsums on nmo x nmo matrices) on top of `rhs_intermediates`."""
    nc, no = p.nc, p.no
    na, nb = nc + no, nc
    it = inter if inter is not None else rhs_intermediates(p, v, apply_response, apply_sf_exchange)
    v, dvva, doob, g, veff0mo = it["v"], it["dvva"], it["doob"], it["g"], it["veff0mo"]
    wvoa = g[0][na:, :na].copy()
    wvob = g[1][nb:, :nb].copy()
    wvoa -= np.einsum("jk,jc->ck", veff0mo[:nc, :na], v)
    wvob += np.einsum("ac,ka->ck", veff0mo.T[na:, nc:], v)
    if not p.restricted:
        return np.hstack([wvoa.ravel(), wvob.ravel()])
    fa, fb = p.fock_ks
    wvoa -= np.einsum("ac,ka->ck", dvva, fa[:na, na:])              # (:256)
    wvob += np.einsum("jk,jc->ck", doob, fb[:nc, nc:])              # (:258; the pure branch's :269 is a shape error, DESIGN section 9)
    wvc = wvoa[:, :nc] + wvob[no:, :]
    return np.hstack([wvc.ravel(), wvoa[:, nc:].ravel(), wvob[:no, :].ravel()]) * 2


def assemble_w(p, z, inter: dict, apply_response_z):
    """The W matrix `im0` (AO basis) that multiplies the overlap derivatives: grad_hb/tdroks_sfu.py:328-356 (ROKS, z = [zvc | zvo | zoc])
    / tduks_sfu.py:266-299 (UKS, z = the stacked halves `ucphf.solve` returns).  `apply_response_z(t[2, nmo, nmo])` is the full
    `vresp` on MO-basis matrices (plan.build_mo_response_plan with the range-separated part): one application to the symmetrised
    Z-vector density; the rest is the reference's block bookkeeping."""
    nc, no, nv, nmo = p.nc, p.no, p.nv, p.nmo
    na, nb = nc + no, nc
    v, dvva, doob, g, veff0mo = inter["v"], inter["dvva"], inter["doob"], inter["g"], inter["veff0mo"]
    z = np.asarray(z, dtype=np.float64).ravel()
    zs = np.zeros((2, nmo, nmo))
    if p.restricted:
        zvc = z[:nv * nc].reshape(nv, nc)
        zvo = z[nv * nc:nv * nc + nv * no].reshape(nv, no)
        zoc = z[nv * nc + nv * no:].reshape(no, nc)
        z1a, z1b = np.hstack((zvc, zvo)), np.vstack((zoc, zvc))
    else:
        z1a, z1b = z[:nv * na].reshape(nv, na), z[nv * na:].reshape(no + nv, nb)
    zs[0, na:, :na] = z1a
    zs[1, nb:, :nb] = z1b
    zs = zs + zs.transpose(0, 2, 1)
    if p.restricted:
        zs *= 0.5                                                    # (:339) Z^S = (z + z^T) / 2; UKS (:270): z + z^T
    veff = np.asarray(apply_response_z(zs)).reshape(2, nmo, nmo)
    ca, cb = p.mo_coeff
    im0a, im0b = np.zeros((nmo, nmo)), np.zeros((nmo, nmo))
    if p.restricted:
        fa, fb = p.fock_ks
        favc = 0.5 * (fa[na:, :nc] + fa[:nc, na:].T)                # symmetrised block (:227)
        im0a[:na, :na] = fa[:na, :na] + (g[0] + veff[0])[:na, :na]
        im0b[:nc, :nc] = fb[:nc, :nc] + (g[1] + veff[1])[:nc, :nc]
        im0a[na:, na:] = np.einsum("ac,bc->ab", dvva, fa[na:, na:]) + np.einsum("ia,ib->ab", v, veff0mo[:nc, na:])
        im0a[na:, :na] = (np.einsum("aj,ij->ai", z1a, fa[:na, :na]) + 2 * np.einsum("ac,ic->ai", dvva, fa[:na, na:])
                          + 2 * np.einsum("ia,ij->aj", v, veff0mo[:nc, :na]))
        im0b[:nc, :nc] += np.einsum("ik,kj->ij", doob, fb[:nc, :nc]) + np.einsum("ia,ja->ij", v, veff0mo[:nc, na:])
        im0b[nc:, :nc] = np.einsum("aj,ij->ai", z1b, fb[:nc, :nc])
        im0b[nc:na, :nc] += np.einsum("bt,bi->ti", zvo, favc)
        return ca @ (im0a + im0b) @ ca.T
    ea, eb = p.mo_energy
    im0a[:na, :na] = (g[0] + veff[0])[:na, :na]
    im0a[na:, na:] = np.einsum("jd,jc->dc", veff0mo[:nc, na:], v)
    im0a[:na, na:] = np.einsum("jk,jc->kc", veff0mo[:nc, :na], v) * 2
    im0b[:nc, :nc] = (g[1] + veff[1])[:nc, :nc] + np.einsum("al,ka->lk", veff0mo.T[na:, :nc], v)
    zeta_a = (ea[:, None] + ea) * 0.5
    zeta_a[:na, na:] = ea[na:]
    zeta_a[na:, :na] = ea[:na]
    dm1a = np.zeros((nmo, nmo))
    dm1a[na:, na:] = dvva
    dm1a[na:, :na] = z1a * 2
    dm1a[:na, :na] += np.eye(na)
    zeta_b = (eb[:, None] + eb) * 0.5
    zeta_b[nc:, :nc] = eb[:nc]
    zeta_b[:nc, nc:] = eb[nc:]
    dm1b = np.zeros((nmo, nmo))
    dm1b[:nc, :nc] = doob
    dm1b[nc:, :nc] = z1b * 2
    dm1b[:nc, :nc] += np.eye(nc)
    return ca @ (im0a + zeta_a * dm1a) @ ca.T + cb @ (im0b + zeta_b * dm1b) @ cb.T


def _pos_idx(idx):
    """(internal positions, MO indices) of the real orbitals of an index list (-1 = zero pad)."""
    idx = np.asarray(idx)
    pos = np.nonzero(idx >= 0)[0]
    return pos, idx[pos]


def mo_to_blocks(plan, t) -> np.ndarray:
    """Symmetric MO-basis densities t[2, nmo, nmo] (one per spin) -> the `xtd_block_response` input: per channel of the two-channel plan
    [Doo | Dvv | Dov] on the channel's internal positions.  Every channel's occupied and virtual sets together cover all orbitals of its
    spin, so nothing of t is lost; t must be symmetric (the virtual-occupied block is the transpose of Dov)."""
    t = np.asarray(t, dtype=np.float64)
    if not np.allclose(t, t.transpose(0, 2, 1), rtol=0.0, atol=1e-13 * max(1.0, float(np.abs(t).max()))):
        raise ValueError("mo_to_blocks: the densities must be symmetric")
    parts = []
    for ch in plan.channels:
        assert ch.spin_o == ch.spin_v
        m = t[ch.spin_o]
        (op, oi), (vp, vi) = _pos_idx(ch.occ_idx), _pos_idx(ch.vir_idx)
        for (rp, ri, nr), (cp, ci, ncol) in (((op, oi, ch.no), (op, oi, ch.no)), ((vp, vi, ch.nv), (vp, vi, ch.nv)),
                                             ((op, oi, ch.no), (vp, vi, ch.nv))):
            b = np.zeros((nr, ncol))
            b[np.ix_(rp, cp)] = m[np.ix_(ri, ci)]
            parts.append(b.ravel())
    return np.concatenate(parts)


def blocks_to_mo(plan, out, nmo: int) -> np.ndarray:
    """`xtd_block_response` output (per channel [Voo | Vov]) -> [2, nmo, nmo] MO-basis response matrices with the occupied-occupied,
    occupied-virtual and virtual-occupied blocks filled; the virtual-virtual block is not computed and is NaN."""
    res = np.full((2, nmo, nmo), np.nan)
    off = 0
    for ch in plan.channels:
        (op, oi), (vp, vi) = _pos_idx(ch.occ_idx), _pos_idx(ch.vir_idx)
        voo = out[off:off + ch.no * ch.no].reshape(ch.no, ch.no)
        off += ch.no * ch.no
        vov = out[off:off + ch.no * ch.nv].reshape(ch.no, ch.nv)
        off += ch.no * ch.nv
        r = res[ch.spin_o]
        r[np.ix_(oi, oi)] = voo[np.ix_(op, op)]
        r[np.ix_(oi, vi)] = vov[np.ix_(op, vp)]
        r[np.ix_(vi, oi)] = vov[np.ix_(op, vp)].T
    return res


def x_to_block(plan, x) -> np.ndarray:
    """Mixed-spin density x[nmo_b, nmo_a] (rows: spin of channel 1, columns: spin of channel 0), nonzero only on (channel-1 occupied) x
    (channel-0 virtual) -> the X block of `xtd_block_response`."""
    c0, c1 = plan.channels
    (op, oi), (vp, vi) = _pos_idx(c1.occ_idx), _pos_idx(c0.vir_idx)
    blk = np.zeros((c1.no, c0.nv))
    blk[np.ix_(op, vp)] = x[np.ix_(oi, vi)]
    rest = np.array(x, dtype=np.float64, copy=True)
    rest[np.ix_(oi, vi)] = 0.0
    if np.any(rest != 0.0):
        raise ValueError("x_to_block: the density has elements outside (channel-1 occupied) x (channel-0 virtual)")
    return blk


def xblock_to_mo(plan, xo, nmo: int) -> np.ndarray:
    """K[X] on (channel-1 occupied + virtual) x (channel-0 occupied + virtual) -> [nmo_b, nmo_a]."""
    c0, c1 = plan.channels
    xo = np.asarray(xo).reshape(c1.no + c1.nv, c0.no + c0.nv)
    rp, ri = _pos_idx(np.concatenate([c1.occ_idx, c1.vir_idx]))
    cp, ci = _pos_idx(np.concatenate([c0.occ_idx, c0.vir_idx]))
    res = np.zeros((nmo, nmo))
    res[np.ix_(ri, ci)] = xo[np.ix_(rp, cp)]
    return res


def block_callables(p, plan, apply_blocks):
    """The `apply_response` / `apply_sf_exchange` / `apply_response_z` callables of rhs_intermediates and assemble_w, computed by
    `apply_blocks(dens, coef, x) -> (out, xout)` -- the `xtd_block_response` contract on the Z-vector operator plan's index sets
    (alpha: [c|o] x v, beta: c x [o|v]) -- instead of whole-MO-space plans.  Coefficients (J, K full range, K long range, f_xc, K[X]):
    the operator engine's kernel table carries the plan's `xc_scale`, which the f_xc coefficient takes back out."""
    nmo = p.nmo
    cxc = 1.0 / plan.xc_scale if plan.xc_kind != "none" else 0.0
    ck0 = -p.hyb if p.hybrid else 0.0
    ck1 = -(p.alpha - p.hyb) if (p.hybrid and p.omega != 0.0 and p.has_df_lr) else 0.0

    def response(coef):
        return lambda t: blocks_to_mo(plan, apply_blocks(mo_to_blocks(plan, t), coef, None)[0], nmo)

    def sf_exchange(x):
        return xblock_to_mo(plan, apply_blocks(mo_to_blocks(plan, np.zeros((2, nmo, nmo))), (0.0, 0.0, 0.0, 0.0, 1.0),
                                               x_to_block(plan, x))[1], nmo)
    return response((1.0, ck0, 0.0, cxc, 0.0)), (sf_exchange if p.hyb != 0.0 else None), response((1.0, ck0, ck1, cxc, 0.0))


class ZVector:
    """Operator and solver of the Z-vector equation for one mean-field reference.

        zv = ZVector(mf_or_problem)          # ROKS or UKS reference, density-fitted
        az = zv.matvec(z)                    # the reference's `matvec` (ROKS) / `(e_a - e_i) z + fvind(z)` (UKS)
        z  = zv.solve(rhs)                   # ROKS: rhs = w;  UKS: rhs = hstack(wvoa.ravel(), wvob.ravel()), solves A z = -rhs

    Vector layout (virtual-major blocks, as the reference's closures take them): ROKS [vc (nv,nc) | vo (nv,no) | oc (no,nc)],
    UKS [alpha (nv, nocc_a) | beta (nvir_b, nocc_b)].  `with_diag=False` (UKS) gives the bare `fvind`.
    """
    cphf_max_cycle = 40          # grad_tdrhf_Gradients_cphf_max_cycle (20) + 20, tdroks_sfu.py:434
    cphf_conv_tol = 1e-8         # tduks_sfu.py:374

    def __init__(self, mf, *, with_diag: bool = True, max_nvec: int = 4, workspace_bytes: Optional[int] = None, distributed: bool = True):
        from .drivers_common import make_engine
        # the Z-vector plan uses the KS Fock blocks only: the ROHF-form Fock build of the spin-adaptation terms is skipped
        self.problem = p = problem_from_mf(mf, kernel="uks", rohf_fock="device")
        self.restricted = bool(p.restricted)
        self.nc, self.no, self.nv = p.nc, p.no, p.nv
        self.plan = planmod.build_zvector_plan(p, with_diag=with_diag)
        self.plan.block_response = True         # rhs / w_matrix read the operator engine's resident blocks
        self.engine = make_engine(self.plan, p, max_nvec=max_nvec, workspace_bytes=workspace_bytes, distributed=distributed)
        self.hdiag = np.asarray(self.plan.hdiag)
        self.dim = int(self.plan.ext_dim)

    def matvec(self, x) -> np.ndarray:
        x = np.asarray(x, dtype=np.float64)
        out = self.engine.sigma_host(x.reshape(-1, self.dim))
        return out[0] if x.ndim == 1 else out

    def solve(self, rhs, tol: Optional[float] = None, max_cycle: Optional[int] = None, lindep: float = 1e-13, verbose: int = 0):
        """Returns the stacked solution vector; `self.converged`, `self.cycles`, `self.residual` describe the run."""
        rhs = np.asarray(rhs, dtype=np.float64).ravel()
        if tol is None:
            tol = 1e-12 if self.restricted else self.cphf_conv_tol        # tdroks_sfu.py:325 / tduks_sfu.py:263
        b = rhs if self.restricted else -rhs
        z, self.converged, self.cycles, self.residual = solve_linear(self.engine.sigma, b, self.hdiag, tol=tol,
                                                                    max_cycle=max_cycle or self.cphf_max_cycle, lindep=lindep,
                                                                    verbose=verbose)
        return z

    def _mo_engines(self, workspace_bytes: Optional[int] = None):
        from .drivers_common import make_engine
        if getattr(self, "_rhs_engines", None) is None:
            p = self.problem
            resp = make_engine(planmod.build_mo_response_plan(p, range_separated=False), p, max_nvec=1, workspace_bytes=workspace_bytes)
            rsh = p.omega != 0.0 and p.has_df_lr
            full = make_engine(planmod.build_mo_response_plan(p), p, max_nvec=1, workspace_bytes=workspace_bytes) if rsh else resp
            sfx = (make_engine(planmod.build_mo_sf_exchange_plan(p), p, max_nvec=1, workspace_bytes=workspace_bytes)
                   if p.hyb != 0.0 else None)
            self._rhs_engines = (resp, sfx, full)
        return self._rhs_engines

    def rhs(self, v, workspace_bytes: Optional[int] = None, route: str = "blocks"):
        """Right-hand side for the state with spin-flip-up amplitudes v[nc, nv] (collinear kernel); the intermediates are kept for
        `w_matrix`.  route="blocks": the J / K / f_xc responses come from `xtd_block_response` on the operator engine's resident blocks
        (no further engine, no whole-MO-space tensor).  route="mo_space": two or three more engines on whole-MO-space plans
        (`_mo_engines`, built on the first call) -- a cross-check that needs naux x nmo^2 per spin."""
        p = self.problem
        if route == "blocks":
            resp, sfx, _ = block_callables(p, self.plan, self.engine.block_response)
        elif route == "mo_space":
            r, x, _ = self._mo_engines(workspace_bytes)
            resp = lambda t: r.sigma_host(t.reshape(1, -1))[0]
            sfx = (lambda t: x.sigma_host(t.reshape(1, -1))[0]) if x is not None else None
        else:
            raise ValueError(f"route {route!r}: 'blocks' or 'mo_space'")
        self._route = route
        self._inter = rhs_intermediates(p, v, resp, sfx)
        return assemble_rhs(p, v, None, None, inter=self._inter)

    def w_matrix(self, z):
        """W matrix `im0` (AO basis) from the solution of the Z-vector equation of the state `rhs` was last called for, on the same
        route."""
        if self._route == "blocks":
            full = block_callables(self.problem, self.plan, self.engine.block_response)[2]
        else:
            f = self._mo_engines()[2]
            full = lambda t: f.sigma_host(t.reshape(1, -1))[0]
        return assemble_w(self.problem, z, self._inter, full)

    def split(self, z):
        """The rotation blocks the reference continues with: ROKS (zvc, zvo, zoc) (tdroks_sfu.py:328-330), UKS (z1a, z1b)."""
        nc, no, nv = self.nc, self.no, self.nv
        z = np.asarray(z).ravel()
        if self.restricted:
            return z[:nv * nc].reshape(nv, nc), z[nv * nc:nv * nc + nv * no].reshape(nv, no), z[nv * nc + nv * no:].reshape(no, nc)
        return z[:nv * (nc + no)].reshape(nv, nc + no), z[nv * (nc + no):].reshape(no + nv, nc)
