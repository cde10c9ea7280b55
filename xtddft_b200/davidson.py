"""Block Davidson eigensolver with device-resident subspace.

Control flow, thresholds and return values follow the reference's solver (xtddft/utils/Davidson.py:21-298, a fork
of pyscf.lib.linalg_helper.davidson1 -- restart at max_space = 12 + 4(nroots-1), at most 40 new vectors per
cycle, `pick`, convergence |de| < tol and |r| < tol_residual, preconditioning with e[0], projection against the
subspace, linear-dependency drops).  What changes is where the vectors live: trial vectors, sigma vectors and the
subspace stay in HBM; Gram matrices, Ritz vectors, residuals, the diagonal preconditioner and the projections are
hand-written kernels behind the C-ABI (`xtd_vec_*`).  Only the tiny projected matrix (<= ~100 x 100) is
diagonalised on the host, as in the reference.

Deviations from the shipped file (SURVEY Appendix D): no CuPy `.get()` hops; the 4th return value `Davidcyc`
that every caller unpacks is returned as [cycles, sigma_vectors].
"""
from __future__ import annotations

import ctypes as C
import time
from typing import Callable, Optional

import numpy as np
import scipy.linalg

from . import _lib


class LinearDependencyError(RuntimeError):
    pass


# --------------------------------------------------------------------------------------------------------
# vector backend: rows of a [n_rows, dim] device matrix
# --------------------------------------------------------------------------------------------------------
class CudaVectors:
    """Vector algebra through libxtdsigma's `xtd_vec_*` kernels on torch-owned device buffers."""

    def __init__(self, dim: int, device=None):
        import torch
        if not torch.cuda.is_available():
            raise _lib.XtdError("the Davidson subspace algebra needs a CUDA device; there is no CPU fallback")
        self.torch = torch
        self.lib = _lib.load()
        self.dim = int(dim)
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else device

    def _stream(self):
        return C.c_void_p(self.torch.cuda.current_stream(self.device).cuda_stream)

    def sync(self):
        self.torch.cuda.synchronize(self.device)

    def alloc(self, rows: int):
        return self.torch.zeros((rows, self.dim), dtype=self.torch.float64, device=self.device)

    def from_host(self, a: np.ndarray):
        return self.torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).to(self.device)

    def to_host(self, m) -> np.ndarray:
        return m.cpu().numpy()

    def _small(self, a: np.ndarray):
        return self.torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).to(self.device)

    def copy(self, dst, src):
        dst.copy_(src)

    def dots(self, a, b) -> np.ndarray:
        m, k = a.shape[0], b.shape[0]
        if m == 0 or k == 0:
            return np.zeros((m, k))
        g = self.torch.empty((m, k), dtype=self.torch.float64, device=self.device)
        _lib.check(self.lib.xtd_vec_dots(self._stream(), C.c_void_p(g.data_ptr()), k, C.c_void_p(a.data_ptr()), a.stride(0), m,
                                         C.c_void_p(b.data_ptr()), b.stride(0), k, self.dim), "xtd_vec_dots")
        return g.cpu().numpy()

    def lincomb(self, y, x, c: np.ndarray, beta: float = 0.0):
        m, k = c.shape
        if m == 0:
            return
        cd = self._small(c)
        _lib.check(self.lib.xtd_vec_lincomb(self._stream(), C.c_void_p(y.data_ptr()), y.stride(0), C.c_void_p(x.data_ptr()),
                                            x.stride(0) if k else self.dim, C.c_void_p(cd.data_ptr()), max(k, 1), m, k, self.dim,
                                            float(beta)), "xtd_vec_lincomb")

    def residual(self, r, ax, x, e: np.ndarray) -> np.ndarray:
        k = len(e)
        ed = self._small(e)
        nrm = self.torch.empty(k, dtype=self.torch.float64, device=self.device)
        assert r.stride(0) == ax.stride(0) == x.stride(0)
        _lib.check(self.lib.xtd_vec_residual(self._stream(), C.c_void_p(r.data_ptr()), C.c_void_p(ax.data_ptr()), C.c_void_p(x.data_ptr()),
                                             r.stride(0), C.c_void_p(ed.data_ptr()), C.c_void_p(nrm.data_ptr()), k, self.dim),
                   "xtd_vec_residual")
        return nrm.cpu().numpy()

    def precond(self, x, hdiag, shift: np.ndarray) -> np.ndarray:
        k = len(shift)
        sd = self._small(shift)
        nrm = self.torch.empty(k, dtype=self.torch.float64, device=self.device)
        _lib.check(self.lib.xtd_vec_precond(self._stream(), C.c_void_p(x.data_ptr()), x.stride(0), C.c_void_p(hdiag.data_ptr()),
                                            C.c_void_p(sd.data_ptr()), C.c_void_p(nrm.data_ptr()), k, self.dim), "xtd_vec_precond")
        return nrm.cpu().numpy()

    def scale(self, x, s: np.ndarray):
        k = len(s)
        if k == 0:
            return
        sd = self._small(s)
        _lib.check(self.lib.xtd_vec_scale(self._stream(), C.c_void_p(x.data_ptr()), x.stride(0), C.c_void_p(sd.data_ptr()), k, self.dim),
                   "xtd_vec_scale")

    # ---- the same operations with the small coefficient arrays left on the device (no host round trip) -------------------
    def precond_normalise(self, x, hdiag, shift: np.ndarray):
        """x <- normalised (x / (hdiag - shift)): the squared norms never leave the device."""
        k = len(shift)
        sd = self._small(shift)
        nrm = self.torch.empty(k, dtype=self.torch.float64, device=self.device)
        _lib.check(self.lib.xtd_vec_precond(self._stream(), C.c_void_p(x.data_ptr()), x.stride(0), C.c_void_p(hdiag.data_ptr()),
                                            C.c_void_p(sd.data_ptr()), C.c_void_p(nrm.data_ptr()), k, self.dim), "xtd_vec_precond")
        inv = self.torch.rsqrt(self.torch.clamp_min(nrm, 1e-300))
        _lib.check(self.lib.xtd_vec_scale(self._stream(), C.c_void_p(x.data_ptr()), x.stride(0), C.c_void_p(inv.data_ptr()), k, self.dim),
                   "xtd_vec_scale")

    def project_out(self, y, x):
        """y <- y - (y x^T) x for orthonormal rows x: Gram block and update both on the device."""
        m, k = y.shape[0], x.shape[0]
        if m == 0 or k == 0:
            return
        g = self.torch.empty((m, k), dtype=self.torch.float64, device=self.device)
        _lib.check(self.lib.xtd_vec_dots(self._stream(), C.c_void_p(g.data_ptr()), k, C.c_void_p(y.data_ptr()), y.stride(0), m,
                                         C.c_void_p(x.data_ptr()), x.stride(0), k, self.dim), "xtd_vec_dots")
        g.neg_()
        _lib.check(self.lib.xtd_vec_lincomb(self._stream(), C.c_void_p(y.data_ptr()), y.stride(0), C.c_void_p(x.data_ptr()), x.stride(0),
                                            C.c_void_p(g.data_ptr()), k, m, k, self.dim, 1.0), "xtd_vec_lincomb")

    def transform(self, work, n_in: int, t: np.ndarray):
        """work[:n_out] <- t[n_out, n_in] work[:n_in]  (through a scratch block: the kernel must not alias input and output)."""
        n_out = t.shape[0]
        if n_out == 0:
            return
        tmp = getattr(self, "_tmp", None)
        if tmp is None or tmp.shape[0] < n_out:
            tmp = self._tmp = self.alloc(max(n_out, 40))
        self.lincomb(tmp[:n_out], work[:n_in], np.ascontiguousarray(t), 0.0)
        work[:n_out].copy_(tmp[:n_out])


# --------------------------------------------------------------------------------------------------------
# helpers on the backend
# --------------------------------------------------------------------------------------------------------
def _gs_coefficients(g: np.ndarray, lindep: float) -> np.ndarray:
    """Gram-Schmidt carried out on the Gram matrix g = W W^T: rows t of the result give orthonormal vectors t W, taken in
    order; a vector whose squared norm after projecting out the kept ones is <= lindep is dropped -- the criterion of the
    reference's `_qr` (pyscf.lib.linalg_helper), evaluated on the host from ONE device Gram product."""
    n = g.shape[0]
    rows = []
    for i in range(n):
        c = np.zeros(n)
        c[i] = 1.0
        for t in rows:
            c -= (c @ g @ t) * t
        nrm2 = float(c @ g @ c)
        if nrm2 > lindep:
            rows.append(c / np.sqrt(nrm2))
    return np.array(rows).reshape(len(rows), n)


def _orthonormalise(vb, work, n_in: int, lindep: float, gram: Optional[np.ndarray] = None) -> int:
    """Orthonormalise work[:n_in] in place, dropping dependent vectors; returns the number kept (compacted to the front).
    Block form: Gram matrix on the device, Gram-Schmidt coefficients on the host, one linear combination -- applied twice
    (the second pass restores orthogonality to rounding level, as CholQR2 / CGS2 do), i.e. two host round trips per call
    instead of five per vector.  `gram`: the Gram matrix of work[:n_in] if the caller already has it."""
    nv = n_in
    for it in range(2):
        if nv == 0:
            return 0
        g = gram if (it == 0 and gram is not None) else vb.dots(work[:nv], work[:nv])
        t = _gs_coefficients(g, lindep)
        vb.transform(work, nv, t)
        nv = t.shape[0]
    return nv


def _sort_elast(elast, conv_last, vlast, v):
    head, nroots = vlast.shape
    ovlp = abs(np.dot(v[:head].conj().T, vlast))
    mapping = np.argmax(ovlp, axis=1)
    found = np.any(ovlp > .5, axis=1)
    conv = conv_last[mapping]
    e = elast[mapping]
    conv[~found] = False
    e[~found] = 0.
    return e, conv


def davidson1(aop: Callable, x0, precond, tol: float = 1e-12, max_cycle: int = 50, max_space: int = 12, lindep: float = 1e-14,
              nroots: int = 1, pick: Optional[Callable] = None, tol_residual: Optional[float] = None, callback: Optional[Callable] = None,
              level_shift: float = 1e-3, backend=None, verbose: int = 0, timing: Optional[dict] = None):
    """Solve A c = e c for the lowest `nroots` roots.

    aop(X[k, dim] device matrix) -> [k, dim] device matrix;  x0: [n0, dim] host or device;  precond: diagonal (host or
    device vector; `make_diag_precond(diag, level_shift)` semantics) or a callable precond(r_host, e0, x_host) (compat).
    Returns (conv[nroots] bool, e[nroots], x (list of host vectors), [cycles, sigma_vectors])."""
    toloose = np.sqrt(tol) if tol_residual is None else tol_residual
    x0 = np.atleast_2d(x0) if isinstance(x0, np.ndarray) else x0
    dim = x0.shape[1]
    vb = backend if backend is not None else CudaVectors(dim)
    max_space = max_space + (nroots - 1) * 4
    # nroots close to dim (core-valence-separated spaces): the subspace may grow to the whole space, so it never restarts and
    # never takes more new vectors than there are dimensions left
    whole = max_space >= dim
    max_space = min(max_space, dim)
    cap = max_space + nroots + 40
    xs = vb.alloc(cap)
    ax = vb.alloc(cap)
    n0 = x0.shape[0]
    xt = vb.alloc(max(n0, nroots, 1))
    vb.copy(xt[:n0], vb.from_host(x0) if isinstance(x0, np.ndarray) else x0)
    nt = n0
    ritz = vb.alloc(nroots)
    aritz = vb.alloc(nroots)
    hdiag_dev = None
    if not callable(precond):
        hdiag_dev = vb.from_host(np.asarray(precond, dtype=np.float64).reshape(1, -1)) if isinstance(precond, np.ndarray) else precond

    heff = np.zeros((cap, cap))
    fresh_start = True
    xt_orthonormal = False
    e = v = None
    conv = np.zeros(nroots, dtype=bool)
    space = 0
    nsigma = 0
    icyc = -1
    nritz = 0
    for icyc in range(max_cycle):
        if fresh_start:
            space = 0
            nt_in = nt
            nt = _orthonormalise(vb, xt, nt, lindep)
            if nt == 0:
                raise LinearDependencyError("Initial guess is empty or zero" if icyc == 0 else
                                            "No more linearly independent basis were found.")
        elif nt > 1 and not xt_orthonormal:
            nt = _orthonormalise(vb, xt, nt, lindep)
            nt = min(nt, 40)
        xt_orthonormal = False
        if nt == 0:
            raise LinearDependencyError("No linearly independent basis found by the diagonalization solver.")
        if timing is not None:
            vb.sync(); _t0 = time.perf_counter()
        axt = aop(xt[:nt])
        if timing is not None:
            vb.sync(); timing["sigma_s"] = timing.get("sigma_s", 0.0) + time.perf_counter() - _t0
        nsigma += nt
        head, space = space, space + nt
        vb.copy(xs[head:space], xt[:nt])
        vb.copy(ax[head:space], axt)
        elast, vlast, conv_last = e, v, conv
        # projected matrix: new rows/columns only (reference `_fill_heff_hermitian`)
        d_all = vb.dots(xs[head:space], ax[:space])              # [nt, space]: one Gram product, one host round trip
        d_new = d_all[:, head:]
        for ip in range(nt):
            for jp in range(ip):
                heff[head + ip, head + jp] = heff[head + jp, head + ip] = d_new[ip, jp]
            heff[head + ip, head + ip] = d_new[ip, ip]
        if head:
            d_old = d_all[:, :head]                               # [nt, head]
            heff[head:space, :head] = d_old
            heff[:head, head:space] = d_old.T
        w, v = scipy.linalg.eigh(heff[:space, :space])
        if callable(pick):
            w, v, idx = pick(w, v, nroots, locals())
            if len(w) == 0:
                raise RuntimeError(f"Not enough eigenvalues found by {pick}")
        e = w[:nroots]
        v = v[:, :nroots]
        nritz = e.size
        conv = np.zeros(nritz, dtype=bool)
        if not fresh_start:
            elast, conv_last = _sort_elast(elast, conv_last, vlast, v)
        if elast is None or elast.size != e.size:
            de = e
        else:
            de = e - elast
        # Ritz vectors and their images, residuals
        vb.lincomb(ritz[:nritz], xs[:space], np.ascontiguousarray(v.T), 0.0)
        vb.lincomb(aritz[:nritz], ax[:space], np.ascontiguousarray(v.T), 0.0)
        if xt.shape[0] < nritz:
            xt = vb.alloc(nritz)
        nrm2 = vb.residual(xt[:nritz], aritz[:nritz], ritz[:nritz], e)
        dx_norm = np.sqrt(nrm2)
        conv = (abs(de) < tol) & (dx_norm < toloose)
        if verbose:
            print(f"davidson {icyc} space {space} max|r| {dx_norm.max():.3e} e0 {e[0]:.10f} conv {int(conv.sum())}/{nritz}", flush=True)
        if all(conv):
            break
        # precondition the unconverged residuals, normalise, project against the subspace, drop dependent ones
        keep = [k for k in range(nritz) if (not conv[k]) and dx_norm[k] ** 2 > lindep]
        for dst, k in enumerate(keep):
            if dst != k:
                vb.copy(xt[dst:dst + 1], xt[k:k + 1])
        nt = len(keep)
        if nt:
            fused = hdiag_dev is not None and hasattr(vb, "project_out")
            if fused:
                # precondition + normalise, project against the subspace: coefficients stay on the device
                vb.precond_normalise(xt[:nt], hdiag_dev, np.full(nt, e[0] - level_shift))
                vb.project_out(xt[:nt], xs[:space])
            else:
                if hdiag_dev is not None:
                    n2 = vb.precond(xt[:nt], hdiag_dev, np.full(nt, e[0] - level_shift))
                else:
                    host = vb.to_host(xt[:nt])
                    x_host = vb.to_host(ritz[:nritz])
                    for dst, k in enumerate(keep):
                        host[dst] = precond(host[dst], e[0], x_host[k])
                    vb.copy(xt[:nt], vb.from_host(host))
                    n2 = np.einsum("ij,ij->i", host, host)
                vb.scale(xt[:nt], 1.0 / np.sqrt(n2))
                # reference `_normalize_xt_`: subtract projections on all xs, keep if norm^2 > lindep, normalise
                d = vb.dots(xt[:nt], xs[:space])
                vb.lincomb(xt[:nt], xs[:space], -d, beta=1.0)
            # ONE Gram matrix serves the `_normalize_xt_` filter (its diagonal), the normalisation and the first
            # Gram-Schmidt pass of the next cycle's `_qr` (rows / columns rescaled on the host)
            gm = vb.dots(xt[:nt], xt[:nt])
            n2 = np.diag(gm).copy()
            good = [k for k in range(nt) if n2[k] > lindep]
            if good:
                inv = 1.0 / np.sqrt(n2[good])
                sel = np.zeros((len(good), nt))
                sel[np.arange(len(good)), good] = inv
                if len(good) > 1 and not (space + nroots > max_space and not whole):
                    gs = gm[np.ix_(good, good)] * inv[:, None] * inv[None, :]
                    t1 = _gs_coefficients(gs, lindep)
                    vb.transform(xt, nt, t1 @ sel)
                    nt = t1.shape[0]
                    if nt > 1:                                   # second pass (rounding-level orthogonality)
                        g2 = vb.dots(xt[:nt], xt[:nt])
                        t2 = _gs_coefficients(g2, lindep)
                        vb.transform(xt, nt, t2)
                        nt = t2.shape[0]
                    nt = min(nt, 40)
                    xt_orthonormal = True
                else:
                    vb.transform(xt, nt, sel)
                    nt = len(good)
            else:
                nt = 0
        if whole:
            nt = min(nt, dim - space)
        if nt == 0:
            conv = dx_norm < toloose
            break
        fresh_start = space + nroots > max_space and not whole
        if fresh_start:
            # restart from the current Ritz vectors (reference: x0 = _gen_x0(v, xs) then re-orthogonalised)
            if xt.shape[0] < nritz:
                xt = vb.alloc(nritz)
            vb.copy(xt[:nritz], ritz[:nritz])
            nt = nritz
        if callable(callback):
            callback(locals())
    x = [row for row in vb.to_host(ritz[:nritz])]
    return np.asarray(conv), e, x, [icyc + 1, nsigma]


# --------------------------------------------------------------------------------------------------------
# solver settings of each reference driver (SURVEY Appendix A.4) and the initial guess
# --------------------------------------------------------------------------------------------------------
SOLVER = {
    # XTDA.py:775-777 with TDBase defaults; pick keeps w > 1e-3; preconditioner level shift = mf.level_shift (0)
    "xtda": dict(tol=1e-12, tol_residual=1e-5, lindep=1e-12, max_cycle=100, level_shift=0.0, window=1e-3, pick_positive=True),
    # SF_TDA.py:392-395 (lib.davidson1 defaults: tol_residual = sqrt(tol), precond level shift 1e-3)
    "sf_down": dict(tol=1e-7, tol_residual=None, lindep=1e-14, max_cycle=3000, level_shift=1e-3, window=1e-5, pick_positive=False),
    "sf_up": dict(tol=1e-7, tol_residual=None, lindep=1e-14, max_cycle=3000, level_shift=1e-3, window=1e-5, pick_positive=False),
    # XSF_TDA.py:1467-1470
    "xsf": dict(tol=1e-8, tol_residual=None, lindep=1e-9, max_cycle=1000, level_shift=1e-3, window=1e-5, pick_positive=False),
    # XSF_TDA_GPU.py:915-918 / XTDA_GPU.py:393-395 (host Davidson branch)
    "gpu_class": dict(tol=1e-12, tol_residual=1e-5, lindep=1e-12, max_cycle=100, level_shift=1e-3, window=1e-5, pick_positive=False),
}


def init_guess(gaps: np.ndarray, nstates: int, window: float) -> np.ndarray:
    """Unit vectors on the nstates lowest gaps plus everything within `window` above the nstates-th
    (XTDA.py:700-734 window 1e-3; SF_TDA.py:348-380 and XSF_TDA.py:964-982 window 1e-5)."""
    gaps = np.asarray(gaps)
    nstates = min(nstates, gaps.size)
    thr = np.sort(gaps)[nstates - 1] + window
    idx = np.where(gaps <= thr)[0]
    x0 = np.zeros((idx.size, gaps.size))
    x0[np.arange(idx.size), idx] = 1.0
    return x0


def pick_positive(w, v, nroots, envs):
    idx = np.where(w > 1e-3)[0]
    return w[idx], v[:, idx], idx


def davidson_native(eng, x0: np.ndarray, hdiag: np.ndarray, nroots: int, *, tol: float, tol_residual: Optional[float], lindep: float,
                    max_cycle: int, level_shift: float, pick_positive: bool, max_space: int = 12):
    """The same solver with its host control flow inside libxtdsigma (`xtd_davidson`): no interpreter / ctypes round trip per vector
    operation -- what a launch-bound small molecule spends most of its time on.  Same return values as `davidson1`."""
    torch = eng.torch
    lib = eng.lib
    x0 = np.atleast_2d(np.ascontiguousarray(x0, dtype=np.float64))
    dim = x0.shape[1]
    x0d = torch.from_numpy(x0).to(eng.device)
    hd = torch.from_numpy(np.ascontiguousarray(hdiag, dtype=np.float64)).to(eng.device)
    xout = torch.zeros((nroots, dim), dtype=torch.float64, device=eng.device)
    e = np.zeros(nroots)
    conv = np.zeros(nroots, dtype=np.int32)
    ncyc, nsig = C.c_int(), C.c_int()
    opts = _lib.XtdSolverOpts()
    opts.tol, opts.tol_residual, opts.lindep, opts.level_shift = tol, (tol_residual or 0.0), lindep, level_shift
    opts.max_cycle, opts.max_space, opts.pick_positive = max_cycle, max_space, int(bool(pick_positive))
    cb = None
    red = eng.reducer
    if red is not None and red.enabled:
        from .engine import _as_tensor

        def _allreduce(ctx, ptr, n):
            try:
                red.allreduce_(_as_tensor(torch, ptr, n, eng.device))
                return 0
            except Exception:                      # never let an exception cross the C boundary
                return 1
        cb = _lib.ALLREDUCE_FN(_allreduce)
        opts.allreduce = cb
    eng._set_stream()
    nfound = _lib.check(lib.xtd_davidson(eng._h, nroots, C.byref(opts), C.c_void_p(hd.data_ptr()), C.c_void_p(x0d.data_ptr()), x0.shape[0],
                                         C.c_void_p(e.ctypes.data), C.c_void_p(xout.data_ptr()), C.c_void_p(conv.ctypes.data),
                                         C.byref(ncyc), C.byref(nsig)), "xtd_davidson")
    x = [row for row in xout[:nfound].cpu().numpy()]
    return conv[:nfound].astype(bool), e[:nfound].copy(), x, [ncyc.value, nsig.value]


NATIVE_MAX_DIM = 50000      # below this a sigma call is launch-bound and the interpreter overhead of the Python solver dominates


def davidson_for_engine(eng, nroots: int, method: str, guess_gaps: Optional[np.ndarray] = None, verbose: int = 0,
                        timing: Optional[dict] = None, native: Optional[bool] = None, **over):
    """Run the reference's Davidson settings for `method` on a SigmaEngine (vectors stay on the device).  `native`: run the
    solver loop inside libxtdsigma (default for problems below NATIVE_MAX_DIM unknowns when no timing breakdown is asked for)."""
    cfg = dict(SOLVER[method])
    cfg.update(over)
    hdiag = eng.hdiag()
    gaps = hdiag if guess_gaps is None else guess_gaps
    x0 = init_guess(gaps, nroots, cfg["window"])
    if native is None:
        native = hdiag.size < NATIVE_MAX_DIM and timing is None and not verbose
    if native:
        return davidson_native(eng, x0, hdiag, min(nroots, hdiag.size), tol=cfg["tol"], tol_residual=cfg["tol_residual"], lindep=cfg["lindep"],
                               max_cycle=cfg["max_cycle"], level_shift=cfg["level_shift"], pick_positive=cfg["pick_positive"])
    return davidson1(eng.sigma, x0, hdiag, tol=cfg["tol"], tol_residual=cfg["tol_residual"], lindep=cfg["lindep"],
                     max_cycle=cfg["max_cycle"], nroots=min(nroots, hdiag.size), level_shift=cfg["level_shift"],
                     pick=pick_positive if cfg["pick_positive"] else None, verbose=verbose, timing=timing)
