"""Post-Davidson property pass on the device (SURVEY 8f row f1).

What the reference computes after its Davidson with O(nstates^2) Python loops over `np.trace` chains
(xtddft/XTDA.py:838-890 osc_str / rot_str; xtddft/XSF_TDA.py:435-592 and xtddft/XSF_TDA_GPU.py:943-1116 state-to-state
transition dipoles; xtddft/XSF_TDA.py:613-649 D<S^2> on a UKS reference) is evaluated here with the kernels of
libxtdsigma.so:

* one-electron integrals are transformed to the MO basis with the FP64 tensor-core GEMM (`xtd_dgemm_tn`);
* ground -> excited moments are Gram products between amplitude rows and property rows (`xtd_vec_dots`);
* every state-to-state quantity is a bilinear form  q[i,j] = <v_i | T | v_j>  whose operator T consists of block
  left / right products and rank-1 trace terms -- exactly the "local term" vocabulary of the sigma engine
  (plan.LocalGemm / plan.Rank1).  T is compiled to an operator plan that shares the layout maps of the sigma plan
  (block or PySCF order, removed OO vector included), applied to all states at once by the engine, and contracted with
  the states by one Gram kernel: no per-pair loop, no host arithmetic beyond the final 2/3 |de| |tdm|^2 scaling.

No CPU fallback: constructing PropertyPass without a CUDA device or the built library raises XtdError.
"""
from __future__ import annotations

import ctypes as C
import math
from typing import List, Optional, Sequence

import numpy as np

from . import _lib
from . import plan as planmod
from .engine import SigmaEngine, _pad16
from .problem import ProblemData

CGS2AU = 1.0 / (235.7220 * 2)          # xtddft/utils/unit.py:10


def sa_factors(no: int, sa: int):
    """factor1, factor2, factor3 of calculate_TDM_R (XSF_TDA.py:498-505)."""
    s = no / 2.0
    if sa == 0:
        return 1.0, 1.0, 0.0
    return math.sqrt((2 * s + 1) / (2 * s)), math.sqrt((2 * s) / (2 * s - 1)), 1.0 / math.sqrt(2 * s * (2 * s - 1))


def operator_plan(p: ProblemData, layout: str, remove: bool, r_c: np.ndarray, r_o: np.ndarray, l_o: np.ndarray, l_v: np.ndarray,
                  rank1: Sequence = ()) -> planmod.Plan:
    """Plan of a block operator on spin-flip-down vectors c[(c,o) x (o,v)]:

        T(c)[rows C] += c[rows C] r_c      T(c)[rows O] += c[rows O] r_o         (r_*: [(o,v), (o,v)] true indices)
        T(c)[:, cols o] += l_o c[:, cols o]   T(c)[:, cols v] += l_v c[:, cols v]   (l_*: [(c,o), (c,o)])
        T(c) += u <w, c>  for (u, w) in rank1                                     (u, w: [(c,o), (o,v)])

    The layout maps (block / PySCF order, removed OO vector) are those of the sigma plan (plan.build_sf_plan)."""
    base = planmod.build_sf_plan(p, isf=-1, method=2, sa=0, layout=layout, remove=remove, hdiag_kind="sf")
    ch = base.channels[0]
    nc, no, nv = p.nc, p.no, p.nv
    o_pos, v_pos = planmod._pos(ch.o_blocks), planmod._pos(ch.v_blocks)
    o2off, v2off = base.meta["o2off"], base.meta["v2off"]
    emb_v = lambda m: planmod._embed(m, v_pos, v_pos, ch.nv, ch.nv)
    emb_o = lambda m: planmod._embed(m, o_pos, o_pos, ch.no, ch.no)
    emb_ov = lambda m: planmod._embed(m, o_pos, v_pos, ch.no, ch.nv)
    out = planmod.Plan("operator", [ch], xc_kind="none")
    out.ext_dim, out.layout_entries, out.layout_coefs = base.ext_dim, base.layout_entries, base.layout_coefs
    out.meta = dict(base.meta)
    out.hdiag = np.zeros(base.ext_dim)
    LG = planmod.LocalGemm
    if nc > 0:
        out.local_gemms.append(LG("R", (0, 0, nc, 0, ch.nv), (0, 0, 0), emb_v(r_c), 1.0))
    out.local_gemms.append(LG("R", (0, o2off, no, 0, ch.nv), (0, o2off, 0), emb_v(r_o), 1.0))
    out.local_gemms.append(LG("L", (0, 0, ch.no, 0, no), (0, 0, 0), emb_o(l_o), 1.0))
    out.local_gemms.append(LG("L", (0, 0, ch.no, v2off, nv), (0, 0, v2off), emb_o(l_v), 1.0))
    out.rank1s = [planmod.Rank1(0, emb_ov(u), 0, emb_ov(w)) for (u, w) in rank1]
    return out


def _scaled_blocks(m: np.ndarray, n1: int, f: float) -> np.ndarray:
    """copy of m with the two off-diagonal blocks (split at n1) multiplied by f"""
    out = np.array(m, dtype=np.float64, copy=True)
    out[:n1, n1:] *= f
    out[n1:, :n1] *= f
    return out


def tdm_r_operator(p: ProblemData, d_mo: np.ndarray, sa: int, layout: str, remove: bool) -> planmod.Plan:
    """State-to-state transition-moment operator of one MO-basis integral matrix d_mo[nmo, nmo] on a ROKS reference:
    the 16 block couplings of XSF_TDA.py:526-590 / XSF_TDA_GPU.py:1038-1113 as two right products (rows C scaled by
    factor1 off the block diagonal, rows O by factor2), two left products (columns o: factor2, columns v: factor1) and
    the factor3 trace terms."""
    nc, no = p.nc, p.no
    f1, f2, f3 = sa_factors(no, sa)
    na = nc + no
    d_vir = d_mo[nc:, nc:].T                         # sum_a c[i,a] D[a',a]
    d_occ = d_mo[:na, :na]
    rank1 = []
    if f3 != 0.0:
        w = np.zeros((na, d_vir.shape[0]))
        w[:nc, :no] = f3 * d_mo[:nc, nc:na]          # CO block:  +factor3 D_co
        w[nc:, no:] = -f3 * d_mo[nc:na, na:]         # OV block:  -factor3 D_ov
        e = np.zeros_like(w)
        e[nc + np.arange(no), np.arange(no)] = 1.0   # identity on the OO block
        rank1 = [(w, e), (e, w)]
    return operator_plan(p, layout, remove, _scaled_blocks(d_vir, no, f1), _scaled_blocks(d_vir, no, f2),
                         -_scaled_blocks(d_occ, nc, f2), -_scaled_blocks(d_occ, nc, f1), rank1)


def tdm_u_operator(p: ProblemData, d_aa: np.ndarray, d_bb: np.ndarray, layout: str) -> planmod.Plan:
    """UKS reference (XSF_TDA.py:451-476): T(c) = c D^bb_vir^T - D^aa_occ c."""
    nc, na = p.nc, p.nc + p.no
    r = d_bb[nc:, nc:].T
    l = -d_aa[:na, :na]
    return operator_plan(p, layout, False, r, r, l, l)


def s2_u_operator(p: ProblemData, sba_oo: np.ndarray, sba_vo: np.ndarray, layout: str) -> planmod.Plan:
    """P_ab of XSF_TDA.py:643-646 as <c|T|c>: T(c) = (S_ab S_ba)_oo c - c (S_ba,vo S_ba,vo^T) + w <w, c>, w = S_ba,vo^T."""
    m = sba_oo.T @ sba_oo                            # [nocc_a, nocc_a]
    n = sba_vo @ sba_vo.T                            # [nvir_b, nvir_b]
    w = sba_vo.T.copy()
    return operator_plan(p, layout, False, -n, -n, m, m, [(w, w)])


class PropertyPass:
    """Device-side property evaluation for one SCF reference (`ProblemData`)."""

    def __init__(self, problem: ProblemData, device=None):
        import torch
        if not torch.cuda.is_available():
            raise _lib.XtdError("the property pass needs a CUDA device (sm_100a); there is no CPU fallback")
        self.torch, self.lib, self.p = torch, _lib.load(), problem
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)

    # ---- plumbing ---------------------------------------------------------------------------------------
    def _stream(self):
        return C.c_void_p(self.torch.cuda.current_stream(self.device).cuda_stream)

    def _padded(self, a: np.ndarray):
        """host [r, c] -> device [r, pad16(c)] (zero padded), as the TMA-fed GEMM wants its operands"""
        t = self.torch
        a = np.ascontiguousarray(a, dtype=np.float64)
        buf = t.zeros((a.shape[0], _pad16(a.shape[1])), dtype=t.float64, device=self.device)
        buf[:, :a.shape[1]] = t.from_numpy(a).to(self.device)
        return buf

    def _gemm_tn(self, a, m: int, b, n: int, k: int, c):
        """c[m, n] = sum_k a[m, k] b[n, k] on device buffers with padded leading dimensions"""
        _lib.check(self.lib.xtd_dgemm_tn(self._stream(), m, n, k, 1.0, C.c_void_p(a.data_ptr()), a.stride(0), C.c_void_p(b.data_ptr()),
                                         b.stride(0), C.c_void_p(c.data_ptr()), c.stride(0), 0), "xtd_dgemm_tn")

    def mo_transform(self, ints_ao: np.ndarray, cbra: np.ndarray, cket: np.ndarray) -> np.ndarray:
        """out[x, i, j] = sum_pq cbra[p, i] ints_ao[x, p, q] cket[q, j]  (two tensor-core GEMMs per component)."""
        t = self.torch
        ints_ao = np.asarray(ints_ao, dtype=np.float64)
        n, nb, nk = ints_ao.shape[1], cbra.shape[1], cket.shape[1]
        bra_t, ket_t = self._padded(cbra.T), self._padded(cket.T)                 # [nb, N], [nk, N]
        half = t.zeros((nb, _pad16(n)), dtype=t.float64, device=self.device)
        res = t.zeros((nb, _pad16(nk)), dtype=t.float64, device=self.device)
        out = np.empty((ints_ao.shape[0], nb, nk))
        for x, d in enumerate(ints_ao):
            dt = self._padded(d.T)                                                # rows q, contiguous p
            self._gemm_tn(bra_t, nb, dt, n, n, half)                              # half[i, q] = sum_p cbra[p,i] d[p,q]
            self._gemm_tn(half, nb, ket_t, nk, n, res)                            # res[i, j] = sum_q half[i,q] cket[q,j]
            out[x] = res[:, :nk].cpu().numpy()
        return out

    def _dots(self, a, b) -> np.ndarray:
        t = self.torch
        m, k, n = a.shape[0], b.shape[0], a.shape[1]
        g = t.empty((m, k), dtype=t.float64, device=self.device)
        _lib.check(self.lib.xtd_vec_dots(self._stream(), C.c_void_p(g.data_ptr()), k, C.c_void_p(a.data_ptr()), a.stride(0), m,
                                         C.c_void_p(b.data_ptr()), b.stride(0), k, n), "xtd_vec_dots")
        return g.cpu().numpy()

    def _rows(self, x) -> "object":
        """states as contiguous device rows [nstates, dim]"""
        t = self.torch
        if isinstance(x, np.ndarray):
            return t.from_numpy(np.ascontiguousarray(x, dtype=np.float64)).to(self.device)
        return x.contiguous()

    # ---- X-TDA: ground -> excited moments (PySCF order rows) ------------------------------------------------
    def xtda_moments(self, x_rows, ints_ao: np.ndarray, rows: Optional[np.ndarray] = None) -> np.ndarray:
        """trans[s, k] (XTDA.py:849-857): Gram product of the amplitude rows with the MO-basis integral rows.  `rows`: the amplitudes
        live on these rows of the PySCF-order layout only (core-valence separation, `utils.cvs_rows`)."""
        p = self.p
        ca, cb = p.mo_coeff
        na, nb = p.nocc_a, p.nocc_b
        ma = self.mo_transform(ints_ao, ca[:, :na], ca[:, na:]).reshape(len(ints_ao), -1)
        mb = self.mo_transform(ints_ao, cb[:, :nb], cb[:, nb:]).reshape(len(ints_ao), -1)
        m = np.hstack([ma, mb])
        if rows is not None:
            m = m[:, rows]
        return self._dots(self._rows(x_rows), self._rows(m))

    def xtda_osc_str(self, e: np.ndarray, x_rows, dip_ao: np.ndarray, rows: Optional[np.ndarray] = None) -> np.ndarray:
        td = self.xtda_moments(x_rows, dip_ao, rows)
        return 2.0 / 3.0 * np.asarray(e) * np.einsum("sx,sx->s", td, td)

    def xtda_rot_str(self, e: np.ndarray, x_rows, ipovlp_ao: np.ndarray, irxp_ao: np.ndarray, rows: Optional[np.ndarray] = None) -> np.ndarray:
        ele = -self.xtda_moments(x_rows, ipovlp_ao, rows)
        mag = 0.5 * self.xtda_moments(x_rows, irxp_ao, rows)
        return np.einsum("s,sx,sx->s", 1.0 / np.asarray(e), ele, mag) / CGS2AU

    # ---- spin-flip states: bilinear forms through operator plans ---------------------------------------------
    def bilinear(self, plans: List[planmod.Plan], v_rows) -> np.ndarray:
        """q[k, i, j] = <v_i | T_k | v_j> for operator plans T_k (all states at once per operator)."""
        v = self._rows(v_rows)
        ns, dim = v.shape
        out = np.empty((len(plans), ns, ns))
        ch = plans[0].channels[0]
        ws = int(max(64 << 20, 8 * (6 * ns * (ch.no + 16) * (ch.nv + 16)) + (48 << 20)))
        for k, pl in enumerate(plans):
            assert pl.ext_dim == dim, (pl.ext_dim, dim)
            eng = SigmaEngine.from_problem(pl, self.p, max_nvec=ns, workspace_bytes=ws, device=self.device)
            try:
                out[k] = self._dots(v, eng.sigma(v))
            finally:
                eng.close()
        return out

    def tdm_r(self, v_rows, ints_ao: np.ndarray, sa: int, layout: str = planmod.LAYOUT_BLOCK, remove: bool = False) -> np.ndarray:
        c = self.p.mo_coeff[0]
        d_mo = self.mo_transform(ints_ao, c, c)
        return self.bilinear([tdm_r_operator(self.p, d, sa, layout, remove) for d in d_mo], v_rows)

    def tdm_u(self, v_rows, ints_ao: np.ndarray, layout: str = planmod.LAYOUT_BLOCK) -> np.ndarray:
        ca, cb = self.p.mo_coeff
        aa, bb = self.mo_transform(ints_ao, ca, ca), self.mo_transform(ints_ao, cb, cb)
        return self.bilinear([tdm_u_operator(self.p, a, b, layout) for a, b in zip(aa, bb)], v_rows)

    @staticmethod
    def osc_matrix(e: np.ndarray, tdm: np.ndarray) -> np.ndarray:
        """osc[i, j] = 2/3 |e_i - e_j| |tdm_ij|^2 (XSF_TDA_GPU.py:989, 1114)."""
        e = np.asarray(e)
        return 2.0 / 3.0 * np.abs(e[:, None] - e[None, :]) * np.einsum("xij,xij->ij", tdm, tdm)

    def delta_s2_u(self, v_rows, ovlp: np.ndarray, layout: str = planmod.LAYOUT_BLOCK) -> np.ndarray:
        """D<S^2> of each state on a UKS reference: P_ab - no + 1 (XSF_TDA.py:613-649, 781-784)."""
        p = self.p
        ca, cb = p.mo_coeff
        na, nb = p.nocc_a, p.nocc_b
        s_ba = self.mo_transform(np.asarray(ovlp)[None], cb, ca[:, :na])[0]       # [nmo_b, nocc_a]
        q = self.bilinear([s2_u_operator(p, s_ba[:nb], s_ba[nb:], layout)], v_rows)[0]
        return np.diag(q) - p.no + 1
